"""Per-op parity of the glue kernels through the C-ABI (fp32 GEMM results in, bf16 operands out) against
plain PyTorch fp32 references of the same op with the reference's rounding points."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


def _st():
    return torch.cuda.current_stream().cuda_stream


def _lib():
    from fish_speech_b200 import _lib

    return _lib, _lib.lib()


def rbf(x):
    return x.to(torch.bfloat16).float()


@pytest.mark.parametrize("rows,D", [(1, 256), (32, 2560), (7, 1024)])
def test_resid_scale_norm(rows, D):
    _l, L = _lib()
    g = torch.Generator().manual_seed(rows * D)
    y = torch.randn(rows, D, generator=g)
    x = torch.randn(rows, D, generator=g).bfloat16()
    scale = (0.3 + 0.1 * torch.randn(D, generator=g)).bfloat16()
    w = (1 + 0.1 * torch.randn(D, generator=g)).bfloat16()
    # reference: x' = rbf(x + rbf(y) * scale); n = rbf(rbf(x' * rsqrt(mean(x'^2) + eps)) * w)   (llama.py:990-1001)
    xr = rbf(x.float() + rbf(y) * scale.float())
    n = rbf(rbf(xr * torch.rsqrt((xr * xr).mean(-1, keepdim=True) + 1e-5)) * w.float())
    dy, dx, ds, dw = y.cuda(), x.cuda(), scale.cuda(), w.cuda()
    xo, no = torch.empty_like(dx), torch.empty_like(dx)
    _l.check(L.fsb_resid_scale_norm(dy.data_ptr(), D, ds.data_ptr(), dx.data_ptr(), xo.data_ptr(), dw.data_ptr(),
                                    no.data_ptr(), rows, D, 1e-5, 0, _st()))
    torch.cuda.synchronize()
    assert torch.equal(xo.cpu().float(), xr)
    # the row reduction order differs from torch's: allow one bf16 ulp on a handful of elements
    diff = (no.cpu().float() - n).abs()
    assert (diff > 0).float().mean() < 0.02 and diff.max() <= 2 ** -6 * n.abs().max()


@pytest.mark.parametrize("rows,I", [(3, 512), (32, 9728)])
def test_swiglu(rows, I):
    _l, L = _lib()
    g = torch.Generator().manual_seed(I)
    y = torch.randn(rows, 2 * I, generator=g) * 2
    a, c = rbf(y[:, :I]), rbf(y[:, I:])
    ref = rbf(rbf(a / (1 + torch.exp(-a))) * c)
    dy = y.cuda()
    h = torch.empty(rows, I, dtype=torch.bfloat16, device="cuda")
    _l.check(L.fsb_swiglu_f32(dy.data_ptr(), rows, I, h.data_ptr(), _st()))
    torch.cuda.synchronize()
    diff = (h.cpu().float() - ref).abs()
    assert (diff > 0).float().mean() < 0.01 and diff.max() <= 2 ** -6 * ref.abs().max()  # expf vs torch.exp: rare 1-ulp flips


@pytest.mark.parametrize("H,Hkv,Dh,T,window", [(4, 4, 64, 40, 16), (8, 2, 128, 33, 0), (16, 16, 64, 150, 128)])
def test_qkv_rope_and_window_attention(H, Hkv, Dh, T, window):
    """qkv post-processing (RoPE with a bf16 table, cache write) + banded causal attention vs torch SDPA."""
    _l, L = _lib()
    B = 2
    rows = B * T
    g = torch.Generator().manual_seed(H * T)
    qkv = torch.randn(rows, (H + 2 * Hkv) * Dh, generator=g)
    inv = 1.0 / (10000 ** (torch.arange(0, Dh, 2).float() / Dh))
    ang = torch.outer(torch.arange(T), inv)
    freqs = torch.stack([torch.cos(ang), torch.sin(ang)], -1).bfloat16()
    seq = torch.arange(B, dtype=torch.int32).repeat_interleave(T)
    pos = torch.arange(T, dtype=torch.int32).repeat(B)
    d = lambda t: t.cuda()
    dq = torch.empty(rows, H, Dh, dtype=torch.bfloat16, device="cuda")
    dk = torch.zeros(B, Hkv, T, Dh, dtype=torch.bfloat16, device="cuda")
    dv = torch.zeros_like(dk)
    dqkv, dfr, dseq, dpos = d(qkv), d(freqs), d(seq), d(pos)
    _l.check(L.fsb_qkv_rope(dqkv.data_ptr(), rows, H, Hkv, Dh, dfr.data_ptr(), dseq.data_ptr(), dpos.data_ptr(),
                            dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), T, _st()))
    out = torch.empty(rows, H * Dh, dtype=torch.bfloat16, device="cuda")
    _l.check(L.fsb_window_attn(dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), dseq.data_ptr(), dpos.data_ptr(), rows, H,
                               Hkv, Dh, T, window, out.data_ptr(), _st()))
    torch.cuda.synchronize()

    # reference (llama.py:1026-1038 rotary, modded_dac.py:380-398 window mask)
    def rope(x):  # [B,T,h,Dh]
        xs = x.float().reshape(*x.shape[:-1], -1, 2)
        fr = freqs.float().view(1, T, 1, Dh // 2, 2)
        o = torch.stack([xs[..., 0] * fr[..., 0] - xs[..., 1] * fr[..., 1],
                         xs[..., 1] * fr[..., 0] + xs[..., 0] * fr[..., 1]], -1)
        return rbf(o.flatten(3))

    q, k, v = rbf(qkv).view(B, T, -1).split([H * Dh, Hkv * Dh, Hkv * Dh], -1)
    q, k, v = rope(q.view(B, T, H, Dh)), rope(k.view(B, T, Hkv, Dh)), v.view(B, T, Hkv, Dh)
    assert torch.equal(dq.cpu().float().view(B, T, H, Dh), q)
    assert torch.equal(dk.cpu().float().transpose(1, 2), k)
    idx = torch.arange(T)
    mask = idx[None, :] <= idx[:, None]
    if window:
        mask &= idx[None, :] >= (idx[:, None] - window + 1)
    kk = k.transpose(1, 2).repeat_interleave(H // Hkv, dim=1)
    vv = v.transpose(1, 2).repeat_interleave(H // Hkv, dim=1)
    ref = torch.nn.functional.scaled_dot_product_attention(q.transpose(1, 2), kk, vv, attn_mask=mask)
    ref = ref.transpose(1, 2).reshape(rows, H * Dh)
    err = (out.cpu().float() - ref).abs().max().item()
    assert err <= 2 ** -7 * ref.abs().max().item() + 1e-3, err


@pytest.mark.parametrize("rows,K,N", [(5, 256, 384), (300, 1024, 3072), (32, 9728, 2560)])
def test_linear_f32(rows, K, N):
    _l, L = _lib()
    g = torch.Generator().manual_seed(K)
    x = (torch.randn(rows, K, generator=g) * 0.5).bfloat16()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16()
    ref = x.float() @ w.float().t()
    dx, dw = x.cuda(), w.cuda()
    ws = torch.empty(rows, N, device="cuda")
    _l.check(L.fsb_linear_f32(dx.data_ptr(), rows, K, dw.data_ptr(), N, ws.data_ptr(), _st()))
    torch.cuda.synchronize()
    assert (ws.cpu() - ref).abs().max() <= 2e-3 * max(1.0, ref.abs().max())


def test_conv_gemm_causal_dilated_and_transposed():
    """fsb_conv_gemm against F.conv1d / F.conv_transpose1d with the codec's causal padding rules."""
    from fish_speech_b200.models.dac.modded_dac import DAC, CodecConfig

    B, T, Cin, Cout = 2, 300, 96, 192
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, Cin, T, generator=g).bfloat16().float()
    dac = object.__new__(DAC)
    dac._device = torch.device("cuda")
    dac._keep, dac._bufs = [], {}
    from fish_speech_b200 import _lib as _l

    dac.lib = _l.lib()
    for dil in (1, 3, 9):
        w = (torch.randn(Cout, Cin, 7, generator=g) / math.sqrt(7 * Cin)).bfloat16().float()
        b = torch.randn(Cout, generator=g) * 0.1
        dac._sd = {"c.weight": w, "c.bias": b}
        cv = dac._conv("c", dilation=dil)
        xin = x.transpose(1, 2).contiguous().bfloat16().cuda()  # [B][T][C]
        out = torch.empty(B, T, Cout, dtype=torch.bfloat16, device="cuda")
        dac._gemm(cv, xin, B, T, Cin, T, out0=out)
        torch.cuda.synchronize()
        ref = torch.nn.functional.conv1d(torch.nn.functional.pad(x, (6 * dil, 0)), w, b, dilation=dil)
        err = (out.cpu().float().transpose(1, 2) - ref).abs().max().item()
        assert err <= 2e-2 * max(1.0, ref.abs().max().item()), (dil, err)
    # transposed conv k = 2 * stride, right trim k - stride (modded_dac.py:574-580)
    s = 4
    wt = (torch.randn(Cin, Cout, 2 * s, generator=g) / math.sqrt(2 * Cin)).bfloat16().float()
    bt = torch.randn(Cout, generator=g) * 0.1
    dac._sd = {"t.weight": wt, "t.bias": bt}
    cv = dac._convT("t", s)
    out = torch.empty(B, T * s, Cout, dtype=torch.bfloat16, device="cuda")
    dac._gemm(cv, xin, B, T, Cin, T, out0=out)
    torch.cuda.synchronize()
    ref = torch.nn.functional.conv_transpose1d(x, wt, bt, stride=s)[..., : T * s]
    err = (out.cpu().float().transpose(1, 2) - ref).abs().max().item()
    assert err <= 2e-2 * max(1.0, ref.abs().max().item()), err


@pytest.mark.parametrize("C,dil,B,T", [(96, 1, 2, 300), (192, 3, 1, 517), (192, 9, 2, 128), (384, 9, 2, 260), (96, 9, 1, 40)])
def test_fused_residual_unit_equals_two_conv_launches(C, dil, B, T):
    """csrc/codec_resunit.cu (Snake -> dilated conv7 -> Snake -> conv1 -> + x in one kernel, the intermediate in shared
    memory) against the same unit as two fsb_conv_gemm launches: identical bits (same MMA order, same rounding points),
    and both against fp32 torch (modded_dac.py:599-620 with the causal pad of :546-552)."""
    _l, L = _lib()
    import ctypes as Ct
    g = torch.Generator().manual_seed(C + dil + T)
    cp = (C + 63) // 64 * 64
    x = torch.randn(B, T, C, generator=g).bfloat16()
    a0 = torch.rand(C, generator=g) + 0.5
    a1 = torch.rand(C, generator=g) + 0.5
    an = torch.rand(C, generator=g) + 0.5
    snake = lambda v, al: v + (al + 1e-9).reciprocal() * torch.sin(al * v) ** 2
    a = snake(x.float(), a0).bfloat16()
    w7 = (torch.randn(C, C, 7, generator=g) * (7 * C) ** -0.5).bfloat16()
    w1 = (torch.randn(C, C, 1, generator=g) * C ** -0.5).bfloat16()
    b7 = torch.randn(C, generator=g) * 0.1
    b1 = torch.randn(C, generator=g) * 0.1
    pack = lambda w: torch.nn.functional.pad(w.permute(0, 2, 1).float(), (0, cp - C)).reshape(C, -1).bfloat16().cuda()
    dw7, dw1 = pack(w7), pack(w1)
    d = lambda t: t.cuda()
    da, dx = d(a), d(x)
    db7, db1 = d(b7), d(b1)
    al1, iv1, aln, ivn = d(a1), d((a1 + 1e-9).reciprocal()), d(an), d((an + 1e-9).reciprocal())
    # two launches (the existing path)
    h = torch.empty_like(da)
    y0, y1 = torch.empty_like(dx), torch.empty_like(dx)
    sh7 = (Ct.c_int * 7)(*[-(6 - j) * dil for j in range(7)])
    sh1 = (Ct.c_int * 1)(0)
    _l.check(L.fsb_conv_gemm(da.data_ptr(), B, T, C, C, T * C, dw7.data_ptr(), C, 7, cp, sh7, T, db7.data_ptr(), None, None,
                             0, None, h.data_ptr(), al1.data_ptr(), iv1.data_ptr(), 0, _st()))
    _l.check(L.fsb_conv_gemm(h.data_ptr(), B, T, C, C, T * C, dw1.data_ptr(), C, 1, cp, sh1, T, db1.data_ptr(), None,
                             dx.data_ptr(), 0, y0.data_ptr(), y1.data_ptr(), aln.data_ptr(), ivn.data_ptr(), 0, _st()))
    # one kernel
    f0, f1 = torch.empty_like(dx), torch.empty_like(dx)
    assert L.fsb_res_unit_supported(C) == 1
    _l.check(L.fsb_res_unit(da.data_ptr(), dx.data_ptr(), B, T, C, dil, dw7.data_ptr(), db7.data_ptr(), al1.data_ptr(),
                            iv1.data_ptr(), dw1.data_ptr(), db1.data_ptr(), f0.data_ptr(), f1.data_ptr(), aln.data_ptr(),
                            ivn.data_ptr(), _st()))
    torch.cuda.synchronize()
    assert torch.equal(f0, y0), (f0.float() - y0.float()).abs().max()
    assert torch.equal(f1, y1), (f1.float() - y1.float()).abs().max()
    # in place over x, raw output dropped
    x2 = dx.clone()
    f2 = torch.empty_like(dx)
    _l.check(L.fsb_res_unit(da.data_ptr(), x2.data_ptr(), B, T, C, dil, dw7.data_ptr(), db7.data_ptr(), al1.data_ptr(),
                            iv1.data_ptr(), dw1.data_ptr(), db1.data_ptr(), x2.data_ptr(), f2.data_ptr(), aln.data_ptr(),
                            ivn.data_ptr(), _st()))
    torch.cuda.synchronize()
    assert torch.equal(x2, y0) and torch.equal(f2, y1)
    # fp32 reference
    xin = torch.nn.functional.pad(a.float().transpose(1, 2), (6 * dil, 0))
    hh = torch.nn.functional.conv1d(xin, w7.float(), b7, dilation=dil)
    hh = snake(hh.transpose(1, 2), a1).bfloat16().float().transpose(1, 2)
    yy = torch.nn.functional.conv1d(hh, w1.float(), b1).transpose(1, 2) + x.float()
    err = (f0.cpu().float() - yy).abs().max().item()
    assert err <= 2 ** -6 * yy.abs().max().item() + 2e-2, err
    err1 = (f1.cpu().float() - snake(yy, an)).abs().max().item()
    assert err1 <= 2 ** -5 * snake(yy, an).abs().max().item() + 3e-2, err1


@pytest.mark.parametrize("H,Hkv,Dh,window", [(8, 2, 128, 0), (16, 16, 64, 128)])
def test_tiled_attention_matches_sdpa_and_is_grouping_independent(H, Hkv, Dh, window):
    """csrc/attn_tile.cu (64 rows per CTA, mma.sync, online softmax) on ragged multi-sequence row sets: against fp32
    SDPA, and bit-identical whichever rows share a tile (the rows of a prompt prefilled in one pass, in chunks, or next
    to other sequences) -- what prefix KV reuse relies on."""
    _l, L = _lib()
    S = 700
    lens = [333, 70, 1, 200]
    B = len(lens)
    g = torch.Generator().manual_seed(H + window)
    k = torch.randn(B, Hkv, S, Dh, generator=g).bfloat16()
    v = torch.randn(B, Hkv, S, Dh, generator=g).bfloat16()
    seq = torch.cat([torch.full((n,), b, dtype=torch.int32) for b, n in enumerate(lens)])
    pos = torch.cat([torch.arange(n, dtype=torch.int32) for n in lens])
    rows = seq.numel()
    q = (torch.randn(rows, H, Dh, generator=g) * 1.5).bfloat16()
    dk, dv = k.cuda(), v.cuda()

    def run(idx):
        idx = torch.as_tensor(idx, dtype=torch.long)
        dq, dseq, dpos = q[idx].cuda().contiguous(), seq[idx].cuda(), pos[idx].cuda()
        out = torch.empty(idx.numel(), H * Dh, dtype=torch.bfloat16, device="cuda")
        _l.check(L.fsb_window_attn(dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), dseq.data_ptr(), dpos.data_ptr(),
                                   idx.numel(), H, Hkv, Dh, S, window, out.data_ptr(), _st()))
        torch.cuda.synchronize()
        return out.cpu()

    full = run(range(rows))
    # sequence 0 alone from position 100 on (a later prefill chunk), and everything shifted by 7 rows (other tiling)
    part = run(range(100, 333))
    assert torch.equal(part, full[100:333])
    shifted = run(list(range(7, rows)))
    assert torch.equal(shifted, full[7:])
    kk = k.float().repeat_interleave(H // Hkv, dim=1)
    vv = v.float().repeat_interleave(H // Hkv, dim=1)
    for r in (0, 1, 63, 64, 150, 332, 333, 402, 403, 404, rows - 1):
        b, p = int(seq[r]), int(pos[r])
        lo = max(0, p - window + 1) if window else 0
        s = torch.einsum("hd,hsd->hs", q[r].float(), kk[b, :, lo:p + 1]) / Dh ** 0.5
        ref = torch.einsum("hs,hsd->hd", torch.softmax(s, -1), vv[b, :, lo:p + 1]).reshape(-1)
        err = (full[r].float() - ref).abs().max().item()
        assert err <= 2 ** -7 * ref.abs().max().item() + 2e-3, (r, err)
