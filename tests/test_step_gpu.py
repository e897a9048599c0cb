"""Op-level parity of the decode step's kernels, each driven alone through the host code the decode frame uses
(fsb_op_step_gemm / fsb_op_step_finalize / fsb_op_attn_decode, include/fishb200.h):

  step_gemm_kernel<0/1>      (csrc/lm_gemm.cu) stream-K weight-streaming GEMM, <1> normalising operand X on load
  step_finalize_kernel       (csrc/lm_gemm.cu) slot-ordered partial sums + bias / residual / sums of squares, or SwiGLU
  attn_decode_kernel<DH, G>  (csrc/lm_kernels.cu) qkv partial sums, bias, per-head RMSNorm, RoPE, KV append, attention

GEMM results are held to a float64 reference. Everything whose operation order is fixed -- slot-ordered fp32 sums,
bias and residual adds, bf16 round-to-nearest-even, separately rounded RoPE products -- is compared bit for bit with
a float32 replica fed with the GPU's own raw partials. The library is built without fast math: adds, multiplies and
divisions are IEEE, and only expf / rsqrtf are approximate. Where one of those decides a bf16 rounding, the element is
"ambiguous": the replica is evaluated with the approximated value scaled by (1 +- 2^-21), and the GPU may give any of
the results; the share of such elements is bounded so that the allowance cannot hide an error.

The tiny model and S2-Pro only reach these kernels end to end; the shapes here add what they never run: every
finalize row block, G in {1, 2, 8}, more than 16 partials per tile, a CTA walking several tiles, K % 64 != 0 and a
partial last 128-feature tile."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROWS = 32  # batch rows of a step GEMM (kStepRows)
SSQ = 32   # floats per row of a sum-of-squares array (kSsqStride)
CTAS = 296  # two CTAs per SM on a B200
EPS = 1e-5
AMB = 2.0 ** -21  # relative window around expf / rsqrtf results


def _st():
    return torch.cuda.current_stream().cuda_stream


def _lib():
    from fish_speech_b200 import _lib

    return _lib, _lib.lib()


def cdiv(a, b):
    return (a + b - 1) // b


def rbf(x):
    """fp32 -> nearest bf16 (ties to even) -> fp32."""
    return x.float().to(torch.bfloat16).float()


def bits(t):
    """Bit pattern of a tensor (NaNs compare equal when their bits do)."""
    return t.view({torch.float32: torch.int32, torch.bfloat16: torch.int16}[t.dtype])


def f32(x):
    return torch.tensor(x, dtype=torch.float32)


def slot_sums(ws, nparts, n_out):
    """[32, n_out] fp32 value of a partial set: slots q < nparts[tile] added in slot order, as the kernels do."""
    tiles = ws.shape[1]
    acc = torch.zeros(tiles, ROWS, 128)
    npt = torch.as_tensor(np.asarray(nparts)).view(tiles, 1, 1)
    for q in range(int(npt.max())):
        acc = torch.where(npt > q, acc + ws[q], acc)
    return acc.permute(1, 0, 2).reshape(ROWS, tiles * 128)[:, :n_out]


def gemm_bound(w64, x64, K, max_parts):
    """Per-element bound of fp32 tensor-core accumulation: (ceil(K/16) + max_parts) * 2^-22 * sum_k |w x|."""
    return (cdiv(K, 16) + max_parts) * 2.0 ** -22 * (x64.abs() @ w64.abs().T)


def step_gemm(w, x, rows, num_ctas, stages=4, norm=None):
    """Run one step GEMM into a NaN-poisoned workspace. w [n_out, K], x [32, K] bf16 on the device;
    norm = (x_ssq [32, 32] fp32, x_nt, norm_w [K] bf16, eps) for normalise-on-load.
    Returns (ws [slots, tiles, 32, 128] fp32 on the host, nparts, max_parts, grid, stages used)."""
    _l, L = _lib()
    import ctypes as C

    n_out, K = w.shape
    tiles = cdiv(n_out, 128)
    slots = min(num_ctas, cdiv(K, 64))  # a tile is never split into more ranges than it has k-blocks
    ws = torch.full((slots, tiles, ROWS, 128), float("nan"), device="cuda")
    nparts = (C.c_int32 * tiles)()
    maxp, grid, st_used = C.c_int(), C.c_int(), C.c_int()
    ssq, x_nt, nw, eps = norm if norm is not None else (None, 0, None, 0.0)
    _l.check(L.fsb_op_step_gemm(w.data_ptr(), n_out, K, x.data_ptr(), rows, int(norm is not None),
                                ssq.data_ptr() if ssq is not None else None, x_nt,
                                nw.data_ptr() if nw is not None else None, eps, num_ctas, stages, ws.data_ptr(),
                                ws.numel(), nparts, C.byref(maxp), C.byref(grid), C.byref(st_used), _st()))
    return ws.cpu(), np.array(nparts[:], dtype=np.int32), maxp.value, grid.value, st_used.value


def dead_rows(x, rows):
    """Operand rows past the live batch hold NaN / Inf: nothing of them may reach a live row."""
    x = x.clone()
    if rows < ROWS:
        x[rows:] = float("nan")
        x[rows::2] = float("inf")
    return x


def check_partials_layout(ws, nparts, maxp, rows, what):
    """Slots past a tile's count and rows past the batch are never written; every live value is finite."""
    tiles = ws.shape[1]
    assert maxp == nparts.max() and (nparts >= 1).all(), what
    for t in range(tiles):
        live = ws[: nparts[t], t, :rows]
        assert torch.isfinite(live).all(), (what, t)
        assert torch.isnan(ws[nparts[t]:, t]).all() and torch.isnan(ws[:, t, rows:]).all(), (what, t)


def check_gemm_value(ws, nparts, maxp, w, x, rows, widen=None):
    """Slot-ordered sum of the partials against float64 W.X^T; returns the worst err / bound."""
    n_out, K = w.shape
    got = slot_sums(ws, nparts, n_out)[:rows].double()
    w64, x64 = w.double(), x[:rows].double()
    ref = x64 @ w64.T
    bound = gemm_bound(w64, x64, K, maxp)
    if widen is not None:
        bound = bound + widen
    ratio = ((got - ref).abs() / bound.clamp_min(1e-300)).max().item()
    assert ratio <= 1.0, f"partial sums off the fp64 product: err/bound {ratio:.3f}"
    return ratio


GEMM_CASES = [
    # n_out, K, rows, num_ctas
    (128, 64, 32, 1),       # one unit
    (97, 256, 5, 296),      # tiny head: ragged n_out, CTAs capped at the unit count
    (4097, 2560, 32, 296),  # restricted head: the last tile has one row
    (6144, 2560, 32, 296),  # qkv
    (2560, 9728, 8, 296),   # w2: about 16 partials per tile
    (256, 9728, 32, 296),   # about 148 partials per tile: many rounds of the finalize's partial loads
    (640, 200, 3, 3),       # K % 64 != 0 (TMA zero fill), ragged ranges
    (640, 2560, 32, 1),     # one CTA walks five tiles (TMEM accumulator ping-pong)
]


@pytest.mark.parametrize("n_out,K,rows,ctas", GEMM_CASES)
def test_step_gemm(n_out, K, rows, ctas):
    g = torch.Generator().manual_seed(n_out * 7 + K)
    w = (torch.randn(n_out, K, generator=g) * 0.05).bfloat16()
    x = torch.randn(ROWS, K, generator=g).bfloat16()
    dw, dx = w.cuda(), dead_rows(x, rows).cuda()
    ws, nparts, maxp, grid, stages = step_gemm(dw, dx, rows, ctas)
    check_partials_layout(ws, nparts, maxp, rows, "stages 4")
    ratio = check_gemm_value(ws, nparts, maxp, w.float(), x.float(), rows)
    # the same bits from a second run, and with a two-deep ring (wraps every other k-block)
    again = step_gemm(dw, dx, rows, ctas)[0]
    assert torch.equal(bits(again), bits(ws)), "two runs differ"
    ws2, np2, _, _, st2 = step_gemm(dw, dx, rows, ctas, stages=2)
    assert st2 == 2 and (np2 == nparts).all()
    assert torch.equal(bits(ws2), bits(ws)), "ring depth changed the partials"
    # a row computed alone (row 0 of a one-row batch) gives the bits it gets inside the batch
    for j in sorted({0, rows // 2, rows - 1}):
        xj = torch.full_like(x, float("nan"))
        xj[0] = x[j]
        wsj = step_gemm(dw, xj.cuda(), 1, ctas)[0]
        for t in range(ws.shape[1]):
            assert torch.equal(bits(wsj[: nparts[t], t, 0]), bits(ws[: nparts[t], t, j])), (j, t)
    print(f"\nstep GEMM n_out={n_out} K={K} rows={rows} ctas={ctas}: grid {grid}, stages {stages}, "
          f"max_parts {maxp}, worst err/bound {ratio:.3f}, ambiguous 0")


# ---- normalise-on-load ----

def norm_replica(x, x_ssq, x_nt, norm_w, K, eps):
    """llama.py:990-1001 as the normalisers compute it: r = rsqrt(sum of the tile sums (in tile order) / K + eps),
    xn = rbf(rbf(x * r) * w). Returns xn, xn at r * (1 - 2^-21), xn at r * (1 + 2^-21)."""
    tot = torch.zeros(ROWS)
    for t in range(x_nt):
        tot = tot + x_ssq[:, t]
    a = tot / f32(K) + f32(eps)
    r = (1.0 / torch.sqrt(a.double()))

    def xn(rr):
        return rbf(rbf(x * rr.float()[:, None]) * norm_w[None, :])

    return xn(r), xn(r * (1 - AMB)), xn(r * (1 + AMB))


def check_norm_on_load(dw, dx, d_ssq, x_nt, d_norm_w, rows, ctas, eps=EPS):
    """NORM=1 partials: bit-identical to NORM=0 partials of the host-normalised operand on every row without an
    ambiguous element; within the fp64 bound (widened by the ambiguous elements' possible flips) everywhere.
    Returns (worst err/bound, ambiguous elements, max_parts)."""
    n_out, K = dw.shape
    w, x, x_ssq, norm_w = dw.float().cpu(), dx.float().cpu(), d_ssq.cpu(), d_norm_w.float().cpu()
    mid, lo, hi = norm_replica(x, x_ssq, x_nt, norm_w, K, eps)
    amb = ((lo != mid) | (hi != mid))[:rows]
    assert torch.isfinite(mid[:rows]).all()
    n_amb = int(amb.sum())
    assert n_amb < 0.01 * amb.numel(), f"{n_amb} ambiguous elements of {amb.numel()}"
    ws1, nparts, maxp, _, _ = step_gemm(dw, dx, rows, ctas, norm=(d_ssq, x_nt, d_norm_w, eps))
    check_partials_layout(ws1, nparts, maxp, rows, "norm on load")
    xn = dead_rows(mid, rows).bfloat16()
    ws0, np0, _, _, _ = step_gemm(dw, xn.cuda(), rows, ctas)
    assert (np0 == nparts).all()
    for j in range(rows):
        if not amb[j].any():
            assert torch.equal(bits(ws1[:, :, j]), bits(ws0[:, :, j])), f"row {j}: NORM=1 != NORM=0 on the normalised row"
    spread = torch.where(amb, (hi[:rows] - lo[:rows]).abs(), torch.zeros(()))
    widen = spread.double() @ w.double().abs().T
    ratio = check_gemm_value(ws1, nparts, maxp, w, mid, rows, widen=widen)
    return ratio, n_amb, maxp


def tile_ssq(x, K):
    """Per-128-feature sums of squares of the bf16 rows (fp64, stored fp32); entries past the last tile are NaN."""
    ssq = torch.full((ROWS, SSQ), float("nan"))
    x64 = x.double()
    for t in range(cdiv(K, 128)):
        ssq[:, t] = (x64[:, t * 128:(t + 1) * 128] ** 2).sum(1).float()
    return ssq


@pytest.mark.parametrize("K", [256, 2560, 4096, 200])
def test_step_gemm_normalise_on_load(K):
    n_out = 640
    g = torch.Generator().manual_seed(K + 1)
    w = (torch.randn(n_out, K, generator=g) * 0.05).bfloat16()
    x = torch.randn(ROWS, K, generator=g)
    x[3] *= 1e3   # large row
    x[5] *= 1e-3  # mean(x^2) ~ 1e-6 < eps: eps matters
    x = x.bfloat16()
    norm_w = (1 + 0.2 * torch.randn(K, generator=g)).bfloat16()
    ssq = tile_ssq(x.float(), K)
    ratio, n_amb, maxp = check_norm_on_load(w.cuda(), x.cuda(), ssq.cuda(), cdiv(K, 128), norm_w.cuda(), ROWS, CTAS)
    print(f"\nnormalise-on-load K={K}: max_parts {maxp}, worst err/bound {ratio:.3f}, ambiguous {n_amb}")


def test_step_gemm_rejects_norm_wider_than_the_ssq_row():
    _l, _ = _lib()
    K = SSQ * 128 + 128
    w = torch.zeros(128, K, dtype=torch.bfloat16, device="cuda")
    x = torch.zeros(ROWS, K, dtype=torch.bfloat16, device="cuda")
    ssq = torch.zeros(ROWS, SSQ, device="cuda")
    with pytest.raises(_l.FsbError, match="normalise-on-load"):
        step_gemm(w, x, ROWS, CTAS, norm=(ssq, SSQ, torch.ones(K, dtype=torch.bfloat16, device="cuda"), EPS))


# ---- PRO_RESID finalize ----

_PARTIALS = {}


def gemm_partials(n_out, K, seed):
    """One NaN-poisoned step GEMM partial set (cached per shape): (ws on the device, nparts on the device, host copies)."""
    key = (n_out, K, seed)
    if key not in _PARTIALS:
        g = torch.Generator().manual_seed(seed)
        w = (torch.randn(n_out, K, generator=g) * 0.05).bfloat16()
        x = torch.randn(ROWS, K, generator=g).bfloat16()
        ws, nparts, maxp, _, _ = step_gemm(w.cuda(), x.cuda(), ROWS, CTAS)
        _PARTIALS[key] = (ws.cuda(), torch.from_numpy(nparts).cuda(), ws, nparts, maxp, w, x)
    return _PARTIALS[key]


def finalize(pro, parts, n_out, rows, rb, bias=None, resid=None, x_out=None, ssq_out=None, h=None, I=0):
    _l, L = _lib()
    dws, dnp, ws, _, maxp = parts[:5]
    p = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
    _l.check(L.fsb_op_step_finalize(pro, dws.data_ptr(), dnp.data_ptr(), ws.shape[1], n_out, maxp, rows, rb, p(bias),
                                    p(resid), p(x_out), p(ssq_out), p(h), I, _st()))


RBS = [1, 2, 4, 8, 16, 32]


@pytest.mark.parametrize("rb", RBS)
@pytest.mark.parametrize("n_out", [2560, 200])
def test_finalize_resid(n_out, rb):
    """x_out = rbf(resid + rbf(sum + bias)) bit for bit (llama.py:842-845), per-tile sums of squares of x_out within
    4 fp32 ulps of fp64; nothing outside [rows, n_out] / the live ssq tiles is written."""
    parts = gemm_partials(n_out, 9728, n_out)
    ws, nparts, maxp = parts[2], parts[3], parts[4]
    S = slot_sums(ws, nparts, n_out)
    tiles = ws.shape[1]
    g = torch.Generator().manual_seed(rb)
    worst_ulp = 0.0
    for rows in (1, 3, 17, 32):
        for with_bias in (False, True):
            for mode in ("none", "separate", "alias"):
                bias = (torch.randn(n_out, generator=g) * 0.3).bfloat16() if with_bias else None
                resid = torch.randn(ROWS, n_out, generator=g).bfloat16()
                canary = torch.randn(ROWS * n_out + 64, generator=g).bfloat16()
                if mode == "alias":  # the engine's call: the residual stream is updated in place
                    canary[: ROWS * n_out] = resid.reshape(-1)
                x_out = canary.cuda()
                ssq_canary = torch.randn(ROWS * SSQ + 8, generator=g)
                ssq_out = ssq_canary.cuda()
                dres = {"none": None, "separate": resid.cuda(), "alias": x_out}[mode]
                finalize(1, parts, n_out, rows, rb, bias=bias.cuda() if with_bias else None, resid=dres,
                         x_out=x_out, ssq_out=ssq_out)
                y = rbf(S[:rows] + bias.float()) if with_bias else rbf(S[:rows])
                ref = y if mode == "none" else rbf(resid[:rows].float() + y)
                got = x_out.cpu()
                what = (rows, with_bias, mode)
                assert torch.equal(bits(got[: rows * n_out].view(rows, n_out)), bits(ref.bfloat16())), what
                assert torch.equal(bits(got[rows * n_out:]), bits(canary[rows * n_out:])), ("rows past the batch", what)
                gs = ssq_out.cpu()
                live = gs[: ROWS * SSQ].view(ROWS, SSQ)[:rows, :tiles]
                x64 = torch.zeros(rows, tiles * 128, dtype=torch.float64)
                x64[:, :n_out] = ref.double()
                want = (x64.view(rows, tiles, 128) ** 2).sum(-1)
                ulp = torch.from_numpy(np.spacing(want.float().numpy())).double()
                worst_ulp = max(worst_ulp, ((live.double() - want).abs() / ulp).max().item())
                keep = torch.ones(ROWS * SSQ + 8, dtype=torch.bool)
                keep[: ROWS * SSQ].view(ROWS, SSQ)[:rows, :tiles] = False
                assert torch.equal(bits(gs[keep]), bits(ssq_canary[keep])), ("ssq written outside", what)
    assert worst_ulp <= 4.0, f"sum of squares {worst_ulp:.2f} ulps off fp64"
    print(f"\nPRO_RESID n_out={n_out} rb={rb}: max_parts {maxp}, nparts {nparts.min()}..{nparts.max()}, "
          f"worst ssq {worst_ulp:.2f} ulp, ambiguous 0")


@pytest.mark.parametrize("n_out", [2560, 200])
def test_finalize_resid_feeds_normalise_on_load(n_out):
    """The engine's wo -> w1|w3 and w2 -> next qkv pair: a NORM=1 GEMM consuming this x_out and ssq_out."""
    parts = gemm_partials(n_out, 9728, n_out)
    g = torch.Generator().manual_seed(n_out + 3)
    bias = (torch.randn(n_out, generator=g) * 0.3).bfloat16().cuda()
    x_out = torch.randn(ROWS, n_out, generator=g).bfloat16().cuda()
    ssq_out = torch.full((ROWS, SSQ), float("nan"), device="cuda")
    finalize(1, parts, n_out, ROWS, 0, bias=bias, resid=x_out, x_out=x_out, ssq_out=ssq_out)
    w2 = (torch.randn(640, n_out, generator=g) * 0.05).bfloat16().cuda()
    norm_w = (1 + 0.2 * torch.randn(n_out, generator=g)).bfloat16().cuda()
    ratio, n_amb, maxp = check_norm_on_load(w2, x_out, ssq_out, cdiv(n_out, 128), norm_w, ROWS, CTAS)
    print(f"\nPRO_RESID -> NORM=1 K={n_out}: max_parts {maxp}, worst err/bound {ratio:.3f}, ambiguous {n_amb}")


# ---- PRO_SWIGLU finalize ----

def gate_row(f):
    """Row of w1[f] in the interleaved w1|w3 weight (include/fishb200.h d_w13); w3[f] is 16 rows further."""
    return (f >> 6) * 128 + ((f >> 4) & 3) * 32 + (f & 15)


def silu_replica(g, e_scale=1.0):
    e = (torch.exp(-g.double()) * e_scale).float()
    return rbf(g / (f32(1.0) + e))


@pytest.mark.parametrize("rb", RBS)
@pytest.mark.parametrize("I", [512, 9728, 500])
def test_finalize_swiglu(I, rb):
    """h = rbf(rbf(silu(g)) * u), g / u = rbf(slot sums of the w1 / w3 rows) bit for bit (llama.py:979-987), except where
    expf decides the rounding of silu; the gate / up rows of each feature are those of w1[f] / w3[f] (fp64)."""
    from fish_speech_b200.engine import interleave_w13

    K = 1024 if I > 4096 else 2560
    key = ("w13", I)
    if key not in _PARTIALS:
        g = torch.Generator().manual_seed(I)
        w1 = (torch.randn(I, K, generator=g) / math.sqrt(K)).bfloat16()  # gate pre-activations ~ N(0, 1)
        w3 = (torch.randn(I, K, generator=g) / math.sqrt(K)).bfloat16()
        x = torch.randn(ROWS, K, generator=g).bfloat16()
        w13 = interleave_w13(w1, w3)
        ws, nparts, maxp, _, _ = step_gemm(w13.cuda(), x.cuda(), ROWS, CTAS)
        S = slot_sums(ws, nparts, w13.shape[0])
        f = torch.arange(I)
        gr = gate_row(f)
        gate, up = S[:, gr], S[:, gr + 16]
        # the replica's row mapping is the weight's: w1 rows and w3 rows against fp64
        x64 = x.double()
        for what, got, wi in (("gate", gate, w1), ("up", up, w3)):
            bound = gemm_bound(wi.double(), x64, K, maxp)
            assert ((got.double() - x64 @ wi.double().T).abs() <= bound).all(), what
        _PARTIALS[key] = (ws.cuda(), torch.from_numpy(nparts).cuda(), ws, nparts, maxp, gate, up, w13.shape[0])
    parts = _PARTIALS[key]
    ws, nparts, maxp, gate, up, n13 = parts[2], parts[3], parts[4], parts[5], parts[6], parts[7]
    gq, uq = rbf(gate), rbf(up)
    mid = rbf(silu_replica(gq) * uq)
    lo = rbf(silu_replica(gq, 1 - AMB) * uq)
    hi = rbf(silu_replica(gq, 1 + AMB) * uq)
    amb_all = (lo != mid) | (hi != mid)
    n_amb = int(amb_all.sum())
    assert n_amb < 1e-3 * amb_all.numel(), f"{n_amb} ambiguous silu roundings of {amb_all.numel()}"
    gen = torch.Generator().manual_seed(rb + I)
    for rows in (1, 5, 32):
        canary = torch.randn(ROWS * I + 64, generator=gen).bfloat16()
        h = canary.cuda()
        finalize(2, parts, n13, rows, rb, h=h, I=I)
        got = h.cpu()
        live = got[: rows * I].view(rows, I).float()
        amb = amb_all[:rows]
        exact = live == mid[:rows]
        ok = exact | (amb & ((live == lo[:rows]) | (live == hi[:rows])))
        assert ok.all(), f"rows={rows}: {int((~ok).sum())} elements differ from the replica"
        assert torch.equal(bits(got[rows * I:]), bits(canary[rows * I:])), ("h written past the live rows", rows)
    print(f"\nPRO_SWIGLU I={I} rb={rb}: max_parts {maxp}, nparts {nparts.min()}..{nparts.max()}, "
          f"ambiguous {n_amb}")


# ---- decode attention ----

def synth_partials(tiles, maxp, g, scale):
    """A qkv partial set with per-tile slot counts 1..maxp (both ends present); dead slots and rows are NaN."""
    nparts = torch.randint(1, maxp + 1, (tiles,), generator=g, dtype=torch.int32)
    nparts[0], nparts[-1] = maxp, max(1, maxp - 3)
    ws = torch.randn(maxp, tiles, ROWS, 128, generator=g) * scale
    for t in range(tiles):
        ws[nparts[t]:, t] = float("nan")
    return ws, nparts


def warp_butterfly_sum(v):
    """warp_sum (common.cuh) on [..., 32] lanes: xor butterfly 16, 8, 4, 2, 1."""
    for o in (16, 8, 4, 2, 1):
        v = v + v[..., torch.arange(32) ^ o]
    return v[..., 0]


def head_replica(v, norm_w, eps, rope, cs):
    """One head of one row (llama.py:891-911): v = rbf(sum + bias) [Dh]; nn.RMSNorm in fp32 (weight included, one
    rounding; the sum of squares per warp by butterfly, then across the head's warps in order); interleaved RoPE with
    separately rounded fp32 products, then rbf. Returns the results at rsqrt r, r (1 - 2^-21), r (1 + 2^-21)."""
    Dh = v.numel()
    outs = []
    if norm_w is not None:
        tot = torch.zeros(())
        for s in warp_butterfly_sum((v * v).view(Dh // 32, 32)):
            tot = tot + s
        r = 1.0 / math.sqrt(float(tot / f32(Dh) + f32(eps)))
        rs = [r, r * (1 - AMB), r * (1 + AMB)]
    else:
        rs = [None]
    for r in rs:
        x = v if r is None else rbf(v * f32(r) * norm_w)
        if rope:
            c, s = cs[:, 0], cs[:, 1]
            x0, x1 = x[0::2], x[1::2]
            o = torch.empty_like(x)
            o[0::2] = x0 * c - x1 * s
            o[1::2] = x1 * c + x0 * s
            x = rbf(o)
        outs.append(x)
    return outs if len(outs) == 3 else outs * 3  # without a norm there is no rsqrt to be ambiguous about


def match(got, outs):
    """got equals the replica, or -- on an element whose rounding the rsqrt window decides -- one of its neighbours."""
    mid, lo, hi = outs
    amb = (lo != mid) | (hi != mid)
    ok = (got == mid) | (amb & ((got == lo) | (got == hi)))
    return bool(ok.all()), int(amb.sum())


@pytest.mark.parametrize("bf16_math", [0, 1])
@pytest.mark.parametrize("qk_norm", [False, True])
@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("G", [1, 2, 4, 8])
@pytest.mark.parametrize("Dh", [64, 128])
def test_attn_decode(Dh, G, bias, qk_norm, bf16_math):
    from oracle import lm_oracle as O

    _l, L = _lib()
    Hkv, S, lcap, slots = 2, 512, 300, 6
    H = G * Hkv
    n_out = (H + 2 * Hkv) * Dh
    tiles, maxp = cdiv(n_out, 128), 11  # two rounds of eight partial loads
    g = torch.Generator().manual_seed(Dh * 100 + G * 10 + 2 * bias + qk_norm + 7 * bf16_math)
    ws, nparts = synth_partials(tiles, maxp, g, 0.4)
    rows = 6
    seq = torch.tensor([3, 0, 5, 1, 2, 4], dtype=torch.int32)
    pos = torch.tensor([0, 1, lcap - 1, 37, -1, 150], dtype=torch.int32)  # row 4 is parked
    ws[:, :, rows:] = float("nan")
    b = (torch.randn(n_out, generator=g) * 0.5).bfloat16() if bias else None
    qn = (1 + 0.2 * torch.randn(Dh, generator=g)).bfloat16() if qk_norm else None
    kn = (1 + 0.2 * torch.randn(Dh, generator=g)).bfloat16() if qk_norm else None
    freqs = O.precompute_freqs_cis(S, Dh, 10000.0)
    kc0 = torch.randn(slots, Hkv, S, Dh, generator=g).bfloat16()
    vc0 = torch.randn(slots, Hkv, S, Dh, generator=g).bfloat16()
    dws, dnp, dseq, dpos, dfr = ws.cuda(), nparts.cuda(), seq.cuda(), pos.cuda(), freqs.cuda()
    db, dqn, dkn = (t.cuda() if t is not None else None for t in (b, qn, kn))
    p = lambda t: t.data_ptr() if t is not None else None  # noqa: E731

    def run(kv_only=0, chunk=0):
        kc, vc = kc0.cuda(), vc0.cuda()
        out = torch.full((rows, H * Dh), float("nan"), dtype=torch.bfloat16, device="cuda")
        _l.check(L.fsb_op_attn_score_chunk(chunk))
        try:
            _l.check(L.fsb_op_attn_decode(dws.data_ptr(), dnp.data_ptr(), tiles, maxp, p(db), p(dqn), p(dkn),
                                          dfr.data_ptr(), kc.data_ptr(), vc.data_ptr(), dseq.data_ptr(),
                                          dpos.data_ptr(), out.data_ptr(), rows, H, Hkv, Dh, S, lcap, bf16_math,
                                          kv_only, EPS, _st()))
        finally:
            L.fsb_op_attn_score_chunk(0)
        return kc.cpu(), vc.cpu(), out.cpu()

    kc, vc, out = run()
    Ssum = slot_sums(ws, nparts, n_out)
    kc_want, vc_want = kc0.clone(), vc0.clone()
    n_amb, worst = 0, 0.0
    scale = 1.0 / math.sqrt(Dh)
    for j in range(rows):
        pj, sj = int(pos[j]), int(seq[j])
        if pj < 0:
            assert torch.isnan(out[j].float()).all(), "parked row's output written"
            continue
        v = Ssum[j] + b.float() if bias else Ssum[j]
        v = rbf(v)
        cs = freqs[pj].float()
        for gi in range(Hkv):
            qs = []
            for hh in range(G):
                hd = gi * G + hh
                outs = head_replica(v[hd * Dh:(hd + 1) * Dh], qn.float() if qk_norm else None, EPS, True, cs)
                n_amb += int(((outs[1] != outs[0]) | (outs[2] != outs[0])).sum())
                qs.append(outs[0])
            kh, vh = H + gi, H + Hkv + gi
            k_outs = head_replica(v[kh * Dh:(kh + 1) * Dh], kn.float() if qk_norm else None, EPS, True, cs)
            ok, na = match(kc[sj, gi, pj].float(), k_outs)
            assert ok, f"row {j} group {gi}: appended K differs from the replica"
            n_amb += na
            assert torch.equal(bits(vc[sj, gi, pj]), bits(v[vh * Dh:(vh + 1) * Dh].bfloat16())), f"row {j}: appended V"
            kc_want[sj, gi, pj] = kc[sj, gi, pj]
            vc_want[sj, gi, pj] = vc[sj, gi, pj]
            # attention over positions [0, pos] of the cache as the kernel left it
            K_ = kc[sj, gi, : pj + 1]
            V_ = vc[sj, gi, : pj + 1]
            q = torch.stack(qs)  # [G, Dh]
            if bf16_math:  # the fast stack's all-bf16 attention (llama.py:948-976)
                mask = torch.ones(1, 1, 1, pj + 1, dtype=torch.bool)
                ref = O._eq_sdpa(q.bfloat16()[None, :, None], K_[None, None].expand(1, G, -1, -1),
                                 V_[None, None].expand(1, G, -1, -1), mask)[0, :, 0].double()
                tol = 2 ** -7 * ref.abs().max().item() + 2e-3  # one bf16 ulp per rounded tensor, rounded twice
            else:
                s = (q.double() @ K_.double().T) * scale
                ref = torch.softmax(s, -1) @ V_.double()
                tol = 2 ** -8 * ref.abs().max().item() + 1e-3
            got = out[j, gi * G * Dh:(gi + 1) * G * Dh].double().view(G, Dh)
            err = (got - ref).abs().max().item()
            assert err <= tol, f"row {j} group {gi}: attention err {err:.3g} > {tol:.3g}"
            worst = max(worst, err / tol)
    assert torch.equal(bits(kc), bits(kc_want)) and torch.equal(bits(vc), bits(vc_want)), "cache written elsewhere"
    assert n_amb < 0.01 * rows * n_out, n_amb
    # kv_only: the same cache, the output untouched
    kc1, vc1, out1 = run(kv_only=1)
    assert torch.equal(bits(kc1), bits(kc)) and torch.equal(bits(vc1), bits(vc))
    assert torch.isnan(out1.float()).all(), "kv_only wrote the output"
    # contexts longer than the score buffer (forced to 64 positions) are walked in chunks, bit-identically
    kc2, vc2, out2 = run(chunk=64)
    assert torch.equal(bits(kc2), bits(kc)) and torch.equal(bits(out2), bits(out)), "chunked attention differs"
    print(f"\nattn_decode Dh={Dh} G={G} bias={bias} qk_norm={qk_norm} bf16_math={bf16_math}: max_parts {maxp}, "
          f"worst err/bound {worst:.3f}, ambiguous {n_amb}")


@pytest.mark.parametrize("H,Hkv,Dh", [(8, 2, 128), (4, 4, 64)])
def test_attention_past_the_score_buffer_is_chunked_bit_identically(H, Hkv, Dh):
    """Contexts longer than the shared-memory score buffer (11 648 positions at G=4, head_dim 128) are walked in chunks
    by attend(): same bits whatever the chunk (forced to 64 / 4096 positions here), and the fp32 SDPA answer
    (llama.py:916-934) at 20 000. Every row has its own KV slot holding the same history, since the kernel appends the
    row's K/V at its position. q, k and v come as a one-slot partial set of bf16 values, without bias or qk-norm and
    with a RoPE table of (cos, sin) = (1, 0): they reach the scores and the cache unchanged. A row's own key scores a
    little above the history's maximum for almost every head, so the maximum sits in the last chunk of every walk;
    the history still carries much of a long row's weight."""
    _l, L = _lib()
    S = 20000
    G = H // Hkv
    n_out = (H + 2 * Hkv) * Dh
    tiles = cdiv(n_out, 128)
    g = torch.Generator().manual_seed(S + H)
    k = torch.randn(Hkv, S, Dh, generator=g).bfloat16()
    v = torch.randn(Hkv, S, Dh, generator=g).bfloat16()
    pos = torch.tensor([0, 31, 32, 63, 64, 4095, 4096, 12543, 12544, 17001, S - 1], dtype=torch.int32)
    rows = pos.numel()
    q = (torch.randn(rows, Hkv, G, Dh, generator=g) * 1.5).bfloat16().float()
    k_new = q.sum(2)  # scaled so that q . k_new / sqrt(Dh) is 8 on average (the history's maximum is about 6)
    k_new = (k_new * (8 * math.sqrt(Dh) / torch.einsum("rhgd,rhd->rhg", q, k_new).mean())).bfloat16().float()
    v_new = torch.randn(rows, Hkv * Dh, generator=g).bfloat16().float()
    qkv = torch.full((ROWS, tiles * 128), float("nan"))
    qkv[:rows, :n_out] = torch.cat([q.reshape(rows, -1), k_new.reshape(rows, -1), v_new], 1)
    ws = qkv.view(ROWS, tiles, 128).transpose(0, 1).contiguous()[None]  # slot 0 of [slots, tiles, 32, 128]
    freqs = torch.zeros(S, Dh // 2, 2)
    freqs[..., 0] = 1.0
    dws, dnp = ws.cuda(), torch.ones(tiles, dtype=torch.int32, device="cuda")
    dfr, dseq, dpos = freqs.bfloat16().cuda(), torch.arange(rows, dtype=torch.int32).cuda(), pos.cuda()
    kc, vc = k.cuda()[None].repeat(rows, 1, 1, 1), v.cuda()[None].repeat(rows, 1, 1, 1)

    def run(chunk):  # every run appends the same K/V at the same positions: the cache is the same for all of them
        out = torch.full((rows, H * Dh), float("nan"), dtype=torch.bfloat16, device="cuda")
        _l.check(L.fsb_op_attn_score_chunk(chunk))
        try:
            _l.check(L.fsb_op_attn_decode(dws.data_ptr(), dnp.data_ptr(), tiles, 1, None, None, None, dfr.data_ptr(),
                                          kc.data_ptr(), vc.data_ptr(), dseq.data_ptr(), dpos.data_ptr(),
                                          out.data_ptr(), rows, H, Hkv, Dh, S, 0, 0, 0, EPS, _st()))
        finally:
            L.fsb_op_attn_score_chunk(0)
        return out.cpu()

    auto = run(0)
    assert torch.equal(bits(run(64)), bits(auto)) and torch.equal(bits(run(4096)), bits(auto))
    scale = 1.0 / math.sqrt(Dh)
    for i, p in enumerate(pos.tolist()):
        K_, V_ = kc[i, :, : p + 1].cpu(), vc[i, :, : p + 1].cpu()  # the cache as the kernel left it
        assert torch.equal(bits(K_[:, p]), bits(qkv[i, H * Dh : (H + Hkv) * Dh].bfloat16().view(Hkv, Dh)))
        assert torch.equal(bits(V_[:, p]), bits(qkv[i, (H + Hkv) * Dh : n_out].bfloat16().view(Hkv, Dh)))
        qi = qkv[i, : H * Dh].double().view(Hkv, G, Dh)
        s = torch.einsum("hgd,hsd->hgs", qi, K_.double()) * scale
        ref = torch.einsum("hgs,hsd->hgd", torch.softmax(s, -1), V_.double()).reshape(-1)
        err = (auto[i].double() - ref).abs().max().item()
        assert err <= 2 ** -7 * ref.abs().max().item() + 1e-3, (p, err)
