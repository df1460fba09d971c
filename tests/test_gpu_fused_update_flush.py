"""The flush of the table-gradient + Adagrad tile kernel (kgeb_fused_bwd_update[_sched], B200): the update warps read the
accumulator from tensor memory and move W / state in TMA boxes of 32 rows x 32 columns.

Reference: the stored-gradient flow, kgeb_fused_bwd with BWD_OVERWRITE_TABLE on the same inputs (the same tile kernel
pipeline, so the same accumulator bits).  Touched rows (slot_of >= 0) must park exactly that gradient in gbuf[slot] and keep
W, state and mirror bit-unchanged; every other row gets state + g*g (one fma: equal to float64 to the last bit but for rare
double-rounding ties) and the Adagrad step with the MUFU square root and reciprocal (within a few ulp of the IEEE term);
the mirror is exactly bf16(W); rows past the shard are never written.  Covers ragged last blocks (n = 128 k + 1, + 97),
touched rows at the first / last row of a 32-row box, in the ragged block and filling a whole box, KL and BCE, d = 64 / 128
(accumulator columns parked in tensor memory) / 256 (no room to park), a shard with e_lo > 0, the skip word and a
learning-rate word changed between launches."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu
GUARD = 40            # rows behind the shard that must stay untouched
EPS = 1e-10


@pytest.fixture(scope="module")
def kb():
    import kgeb200
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return kgeb200


def _stream():
    return torch.cuda.current_stream().cuda_stream


class Problem:
    def __init__(self, kb, n, d, loss, e_lo=0, seed=0):
        self.kb, self.n, self.d, self.e_lo = kb, n, d, e_lo
        self.kind = kb.lib.LOSS_KL if loss == "kl" else kb.lib.LOSS_BCE
        self.b = 256
        self.num_entities = e_lo + n + 1000
        gen = torch.Generator(device="cuda").manual_seed(seed)
        self.w0 = torch.randn(n + GUARD, d, device="cuda", generator=gen) * 0.1
        self.s0 = torch.rand(n + GUARD, d, device="cuda", generator=gen) * 0.1 + 0.01
        self.q = torch.randn(self.b, d, device="cuda", generator=gen) * 0.5
        self.lse = torch.randn(self.b, device="cuda", generator=gen) + 3.0
        self.lab_off = torch.zeros(self.b + 1, dtype=torch.int64, device="cuda")
        self.ws = torch.empty(kb.lib.load().kgeb_fused_workspace_bytes(self.b, d, n, 0), dtype=torch.uint8, device="cuda")

    def dense_gradient(self):
        """G^T Q of the dense part through the storing kernel."""
        g = torch.empty(self.n, self.d, device="cuda")
        mirror = self.w0[:self.n].bfloat16()
        self.kb.lib.call("kgeb_fused_bwd", self.kind, self.kb.lib.MATH_BF16, self.q.data_ptr(), self.b, self.d,
                         self.w0.data_ptr(), self.e_lo, self.e_lo + self.n, self.num_entities, self.lab_off.data_ptr(),
                         self.lab_off.data_ptr(), 0, None, 0.0, 0.0, self.lse.data_ptr() if self.kind == 0 else None,
                         1.0 / self.b, None, mirror.data_ptr(), None, g.data_ptr(), None, self.kb.lib.BWD_OVERWRITE_TABLE,
                         self.ws.data_ptr(), self.ws.numel(), _stream())
        return g

    def fused(self, touched_rows, rate, sched=False, skip=0):
        """One launch of the fused kernel on fresh copies; returns (W, state, mirror, gbuf, slot_of) with guard rows."""
        w, s = self.w0.clone(), self.s0.clone()
        mirror = self.w0.bfloat16()
        slot_of = torch.full((self.n,), -1, dtype=torch.int32, device="cuda")
        rows = torch.tensor(sorted(touched_rows), dtype=torch.int64, device="cuda")
        slot_of[rows] = torch.arange(rows.numel(), dtype=torch.int32, device="cuda")
        gbuf = torch.full((max(rows.numel(), 1), self.d), 7.0, device="cuda")
        flag = torch.tensor([skip], dtype=torch.int32, device="cuda")
        if sched:
            word = torch.tensor([rate], dtype=torch.float32, device="cuda")
            name, r = "kgeb_fused_bwd_update_sched", word.data_ptr()
        else:
            name, r = "kgeb_fused_bwd_update", rate
        self.kb.lib.call(name, self.kind, self.q.data_ptr(), self.b, self.d, w.data_ptr(), self.e_lo, self.e_lo + self.n,
                         self.num_entities, self.lab_off.data_ptr(), 0.0, 0.0, self.lse.data_ptr() if self.kind == 0 else None,
                         1.0 / self.b, None, mirror.data_ptr(), s.data_ptr(), r, EPS, slot_of.data_ptr(), gbuf.data_ptr(),
                         flag.data_ptr(), self.ws.data_ptr(), self.ws.numel(), _stream())
        torch.cuda.synchronize()
        return w, s, mirror, gbuf, rows

    def check(self, out, g, rate):
        w, s, mirror, gbuf, rows = out
        n = self.n
        # behind the shard: untouched (the TMA clips the ragged block's boxes)
        assert torch.equal(w[n:], self.w0[n:]) and torch.equal(s[n:], self.s0[n:])
        assert torch.equal(mirror[n:], self.w0[n:].bfloat16())
        # touched rows: the dense gradient parked bit for bit, W / state / mirror bit-unchanged
        if rows.numel():
            assert torch.equal(gbuf[:rows.numel()], g[rows])
            assert torch.equal(w[rows], self.w0[rows]) and torch.equal(s[rows], self.s0[rows])
            assert torch.equal(mirror[rows], self.w0[rows].bfloat16())
        keep = torch.ones(n, dtype=torch.bool, device="cuda")
        keep[rows] = False
        g64, s64, w64 = g[keep].double(), self.s0[:n][keep].double(), self.w0[:n][keep].double()
        s_ref = (s64 + g64 * g64).float()
        ds = (s[:n][keep] - s_ref).abs()
        assert (ds <= s_ref.abs() * 2.0 ** -23).all(), float(ds.max())
        assert float((s[:n][keep] != s_ref).float().mean()) < 1e-3
        dw_ref = -rate * g64 / (s[:n][keep].double().sqrt() + EPS)
        err = (w[:n][keep].double() - (w64 + dw_ref)).abs()
        assert (err <= 1e-5 * dw_ref.abs() + (w64 + dw_ref).abs() * 2.0 ** -23 + 1e-12).all(), float(err.max())
        assert torch.equal(mirror[:n], w[:n].bfloat16())


@pytest.mark.parametrize("loss", ["kl", "bce"])
@pytest.mark.parametrize("n", [128 * 40, 128 * 40 + 1, 128 * 40 + 97])
def test_flush_against_the_stored_gradient(kb, loss, n):
    p = Problem(kb, n, 128, loss, seed=n)
    k = (n // 128) * 128
    # first and last row of a 32-row box, a whole touched box (rows 224..255 = quadrant 3 of block 1), the ragged block
    touched = {32, 95, *range(224, 256), n - 1}
    if n > k:
        touched.add(k)
    g = p.dense_gradient()
    assert float(g.abs().max()) > 0
    p.check(p.fused(touched, 0.2), g, 0.2)
    p.check(p.fused(set(), 0.2), g, 0.2)           # every box through the TMA store


@pytest.mark.parametrize("d", [64, 256])
def test_flush_dims(kb, d):
    """d = 64: two boxes per warp, both in the ring at the start; d = 256: eight boxes, no tensor-memory room to park."""
    n = 128 * 12 + 97
    p = Problem(kb, n, d, "kl", seed=d)
    g = p.dense_gradient()
    p.check(p.fused({0, 31, 64, 130, n - 1}, 0.1), g, 0.1)


def test_flush_shard_with_offset(kb):
    n = 128 * 9 + 33
    p = Problem(kb, n, 128, "bce", e_lo=5000, seed=3)
    g = p.dense_gradient()
    p.check(p.fused({3, 63, n - 2}, 0.3), g, 0.3)


def test_flush_skip_word_changes_nothing(kb):
    n = 128 * 7 + 5
    p = Problem(kb, n, 128, "kl", seed=4)
    for sched in (False, True):
        w, s, mirror, gbuf, _ = p.fused({10, 200}, 0.2, sched=sched, skip=1)
        assert torch.equal(w, p.w0) and torch.equal(s, p.s0) and torch.equal(mirror, p.w0.bfloat16())
        assert bool((gbuf == 7.0).all())


def test_flush_rate_word_between_launches(kb):
    """The _sched entry with its word rewritten between two launches equals the by-value entry at each rate, bit for bit,
    on a table of >= 64 MB (140,001 x 128 fp32: the size from which the steppers take this kernel)."""
    n = 140_001
    p = Problem(kb, n, 128, "kl", seed=5)
    touched = {0, 777, 140_000}
    word = torch.tensor([0.2], dtype=torch.float32, device="cuda")
    for rate in (0.2, 0.05):
        word.fill_(rate)
        ref = p.fused(touched, rate)
        w, s = p.w0.clone(), p.s0.clone()
        mirror = p.w0.bfloat16()
        slot_of = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        rows = ref[4]
        slot_of[rows] = torch.arange(rows.numel(), dtype=torch.int32, device="cuda")
        gbuf = torch.full((rows.numel(), 128), 7.0, device="cuda")
        kb.lib.call("kgeb_fused_bwd_update_sched", p.kind, p.q.data_ptr(), p.b, 128, w.data_ptr(), 0, n, p.num_entities,
                    p.lab_off.data_ptr(), 0.0, 0.0, p.lse.data_ptr(), 1.0 / p.b, None, mirror.data_ptr(), s.data_ptr(),
                    word.data_ptr(), EPS, slot_of.data_ptr(), gbuf.data_ptr(), None, p.ws.data_ptr(), p.ws.numel(), _stream())
        torch.cuda.synchronize()
        for a, b in zip((w, s, mirror, gbuf), ref[:4]):
            assert torch.equal(a, b), rate
    p.check(ref, p.dense_gradient(), 0.05)
