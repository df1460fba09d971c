"""CPU checks of the drop-in boundary: the C-ABI library loads without a GPU, exports every symbol that
include/kgeb200.h declares, and the ctypes signatures in kge-1_b200/lib.py agree with the header."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CTYPE = {"c_void_p": "p", "c_int": "i", "c_long": "l", "c_float": "f"}


def _header_decls():
    text = open(os.path.join(ROOT, "include", "kgeb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    decls = {}
    for m in re.finditer(r"\b(int64_t|int|const char\*)\s+(kgeb_\w+)\s*\(([^;]*?)\)\s*;", text, flags=re.S):
        ret, name, args = m.group(1), m.group(2), m.group(3)
        kinds = []
        for a in [x.strip() for x in args.split(",") if x.strip() and x.strip() != "void"]:
            if "*" in a:
                kinds.append("p")
            elif a.startswith("int64_t"):
                kinds.append("l")
            elif a.startswith("uint64_t"):
                kinds.append("u")
            elif a.startswith("float"):
                kinds.append("f")
            elif a.startswith("int"):
                kinds.append("i")
            else:
                raise AssertionError(f"unparsed argument {a!r} of {name}")
        decls[name] = (ret, kinds)
    return decls


@pytest.fixture(scope="module")
def kb():
    import __graft_entry__ as ge
    import kgeb200
    if not os.path.exists(kgeb200.lib.LIB_PATH):
        ge.build()
    return kgeb200


def test_library_loads_and_exports_every_declared_symbol(kb):
    lib = kb.lib.load()
    decls = _header_decls()
    assert len(decls) >= 20
    for name in decls:
        assert hasattr(lib, name), f"{name} declared in include/kgeb200.h but not exported"
    assert "sm_100a" in kb.lib.version()


def test_ctypes_signatures_agree_with_header(kb):
    import ctypes
    decls = _header_decls()
    code = {ctypes.c_void_p: "p", ctypes.c_int: "i", ctypes.c_int64: "l", ctypes.c_float: "f", ctypes.c_char_p: "p",
            ctypes.c_uint64: "u"}
    for name, argtypes in {**kb.lib.SIGNATURES, **kb.lib._INT64_RESULT}.items():
        assert name in decls, f"{name} bound in lib.py but not declared in the header"
        assert [code[a] for a in argtypes] == decls[name][1], name
    bound = set(kb.lib.SIGNATURES) | set(kb.lib._INT64_RESULT) | {"kgeb_last_error", "kgeb_version"}
    assert bound == set(decls), sorted(set(decls) ^ bound)


def test_no_cpu_path(kb):
    """The product path fails loudly on CPU tensors instead of falling back."""
    import torch
    m = kb.KgeModel("distmult", 10, 3, 8)
    with pytest.raises(ValueError, match="CUDA"):
        m.score_spo(torch.tensor([1]), torch.tensor([1]), torch.tensor([2]))


@pytest.mark.parametrize("entry", ["kgeb_pairs_bwd", "kgeb_ns_bwd_q", "kgeb_ns_cand_grad"])
@pytest.mark.parametrize("kind", [3, 4])
def test_rotate_pair_kinds_refuse_odd_dim(kb, entry, kind):
    """The RotatE kinds pair column k with k + d/2: an odd d is refused before any launch (kgeb_pairs_score did so
    already; the backward entries used to drop the last column).  Dummy non-null pointers: nothing is dereferenced."""
    p, b, m, d = 256, 4, 3, 15
    args = {"kgeb_pairs_bwd": (kind, p, p, p, 1, b, m, d, p, p, p, p, None),
            "kgeb_ns_bwd_q": (kind, p, p, p, b, m, d, p, p, p, None),
            "kgeb_ns_cand_grad": (kind, p, p, p, b, m, d, p, p, 100, p, p, 1 << 20, None)}[entry]
    with pytest.raises(ValueError, match="even dimensionality"):
        kb.lib.call(entry, *args)
