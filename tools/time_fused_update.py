"""Times the table-gradient + Adagrad tile kernel (kgeb_fused_bwd_update) and the storing table-gradient kernel
(kgeb_fused_bwd with BWD_OVERWRITE_TABLE) alone, with CUDA events, at bench.py's shape: DistMult 1vsAll + KL, E = 4.6 M,
d = 128, 2,048 query rows, an empty label CSR (only the tile kernel and its small pre-kernels run), lr 0, no touched rows.
The operands (2.4 GB fp32 table, 2.4 GB state, 1.2 GB bf16 mirror) are far larger than L2.

Several builds of the library can be compared in one process: `--lib NAME=PATH` loads each with its own ctypes handle, and
the rounds alternate between them (and between the cases of --debug) so that clock drift under the power cap spreads over
all of them.  `--debug` lists KGEB_UPD_DEBUG values for builds that read that variable (1 = no W / state loads, 2 = no
stores, 16 = update warps skip the work but keep the hand-over); builds without it ignore it.

  python tools/time_fused_update.py --lib old=kge-1_b200/variants/libkgeb200_parent.so --lib new=kge-1_b200/libkgeb200.so
"""
import argparse
import ctypes
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench_fb237  # noqa: E402


def _signatures():
    """kge-1_b200/lib.py (argument types and constants) without loading its library: the package directory's name is not
    an identifier, and each build here gets its own ctypes handle."""
    spec = importlib.util.spec_from_file_location("kgeb_lib", os.path.join(ROOT, "kge-1_b200", "lib.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load(path, L):
    lib = ctypes.CDLL(os.path.abspath(path))
    for name in ("kgeb_fused_bwd_update", "kgeb_fused_bwd"):
        getattr(lib, name).argtypes = L.SIGNATURES[name]
        getattr(lib, name).restype = ctypes.c_int
    lib.kgeb_fused_workspace_bytes.argtypes = L._INT64_RESULT["kgeb_fused_workspace_bytes"]
    lib.kgeb_fused_workspace_bytes.restype = ctypes.c_int64
    lib.kgeb_last_error.restype = ctypes.c_char_p
    return lib


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", required=True, help="NAME=PATH of a libkgeb200.so build (repeatable)")
    ap.add_argument("--debug", default="0", help="comma-separated KGEB_UPD_DEBUG values timed per build")
    ap.add_argument("--store", action="store_true", help="also time the storing table-gradient kernel of each build")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--launches", type=int, default=10, help="timed launches per case and round")
    ap.add_argument("--entities", type=int, default=4_600_000)
    ap.add_argument("--out", default=None, help="append the JSON lines here")
    args = ap.parse_args()

    L = _signatures()
    libs = {}
    for spec in args.lib:
        name, path = spec.split("=", 1)
        libs[name] = load(path, L)
    E, d, rows = args.entities, 128, 2048
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev).manual_seed(0)
    w = torch.randn(E, d, device=dev, generator=gen) * 0.1
    state = torch.full((E, d), 0.1, device=dev)
    mirror = w.bfloat16()
    gtmp = torch.empty(E, d, device=dev)
    q = torch.randn(rows, d, device=dev, generator=gen) * 0.5
    lse = torch.full((rows,), 15.3, device=dev)
    off0 = torch.zeros(rows + 1, dtype=torch.int64, device=dev)
    slot_of = torch.full((E,), -1, dtype=torch.int32, device=dev)
    gbuf = torch.zeros(1, d, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    ws_bytes = max(lib.kgeb_fused_workspace_bytes(rows, d, E, 0) for lib in libs.values())
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)

    def upd(lib):
        return lib.kgeb_fused_bwd_update(L.LOSS_KL, q.data_ptr(), rows, d, w.data_ptr(), 0, E, E, off0.data_ptr(), 0.0, 0.0,
                                         lse.data_ptr(), 1.0 / 1024, None, mirror.data_ptr(), state.data_ptr(), 0.0, 1e-10,
                                         slot_of.data_ptr(), gbuf.data_ptr(), None, ws.data_ptr(), ws_bytes, stream)

    def store(lib):
        return lib.kgeb_fused_bwd(L.LOSS_KL, L.MATH_BF16, q.data_ptr(), rows, d, w.data_ptr(), 0, E, E, off0.data_ptr(),
                                  off0.data_ptr(), 0, None, 0.0, 0.0, lse.data_ptr(), 1.0 / 1024, None, mirror.data_ptr(),
                                  None, gtmp.data_ptr(), None, L.BWD_OVERWRITE_TABLE, ws.data_ptr(), ws_bytes, stream)

    cases = []
    for name, lib in libs.items():
        for dbg in [int(x) for x in args.debug.split(",")]:
            cases.append((f"{name} fused_bwd_update debug={dbg}", lib, upd, dbg))
        if args.store:
            cases.append((f"{name} fused_bwd store", lib, store, 0))
    times = {c[0]: [] for c in cases}
    info = gpu_info()
    with bench_fb237.ClockSampler(torch.cuda.current_device()) as clocks:
        for r in range(args.rounds):
            for label, lib, fn, dbg in (cases if r % 2 == 0 else cases[::-1]):
                os.environ["KGEB_UPD_DEBUG"] = str(dbg)
                for _ in range(2):
                    if fn(lib):
                        raise RuntimeError(f"{label}: {lib.kgeb_last_error().decode()}")
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.launches):
                    fn(lib)
                b.record()
                torch.cuda.synchronize()
                times[label].append(a.elapsed_time(b) / args.launches)
    os.environ.pop("KGEB_UPD_DEBUG", None)
    out = []
    for label, ts in times.items():
        out.append({"case": label, "ms_median": float(np.median(ts)), "ms_min": float(np.min(ts)), "ms_max": float(np.max(ts)),
                    "rounds_ms": [round(t, 4) for t in ts], "launches_per_round": args.launches,
                    "shape": f"KL, E={E}, d={d}, rows={rows}, lr 0, no touched rows", "gpu": info,
                    "clocks": clocks.summary()})
    for o in out:
        print(json.dumps(o))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for o in out:
                f.write(json.dumps(o) + "\n")


if __name__ == "__main__":
    main()
