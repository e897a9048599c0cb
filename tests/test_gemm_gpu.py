"""tcgen05/TMA GEMM of prefill and the codec (csrc/gemm_tc.cu) against an fp32 matmul of the same bf16 operands.

The stream-K cases run gemm_tc.cu's own stream-K schedule (gemm_plan_streamk), not the decode step GEMM of
csrc/lm_gemm.cu; that one and its finalize are tested op by op in test_step_gpu.py."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _run(m, n, k, bn, streamk, seed=0):
    from fish_speech_b200 import _lib

    L = _lib.lib()
    g = torch.Generator().manual_seed(seed)
    a = (torch.randn(m, k, generator=g) * 0.5).bfloat16()
    b = (torch.randn(n, k, generator=g) * 0.5).bfloat16()
    ref = b.float() @ a.float().T  # [n, m]
    da, db = a.cuda(), b.cuda()
    out = torch.full((n, m), float("nan"), device="cuda", dtype=torch.float32)
    _lib.check(L.fsb_op_gemm(da.data_ptr(), db.data_ptr(), out.data_ptr(), m, n, k, bn, streamk,
                             torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    got = out.cpu()
    assert torch.isfinite(got).all(), f"non-finite output m={m} n={n} k={k}"
    err = (got - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert err <= 2e-3 * max(scale, 1.0), f"m={m} n={n} k={k} bn={bn} sk={streamk}: err {err} scale {scale}"


@pytest.mark.parametrize("m,n,k,bn", [
    (128, 32, 64, 32),      # one tile, one k-block
    (128, 32, 256, 32),     # k pipeline
    (256, 32, 1024, 32),    # ring wrap (stages < k-blocks)
    (384, 17, 200, 32),     # ragged n, k not a multiple of 64 (TMA zero fill)
    (200, 64, 128, 64),     # ragged m
    (128, 128, 512, 128),
    (256, 300, 320, 128),   # several column tiles
    (128, 256, 256, 256),
    (96, 512, 672, 256),    # codec-like: 96 channels, 7x96 taps flattened
])
def test_gemm_direct(m, n, k, bn):
    _run(m, n, k, bn, 0)


@pytest.mark.parametrize("m,n,k,ctas", [
    (128, 32, 256, 1),
    (128, 32, 256, 3),      # split one tile over 3 CTAs
    (640, 32, 2560, 148),   # many segments, ragged ranges
    (6144, 32, 2560, 148),  # many tiles, about 3 segments per tile
    (2560, 8, 9728, 148),   # long K: about 8 segments per tile, 8 columns
    (4097, 5, 2560, 148),   # a last tile of one row, 5 columns
])
def test_gemm_streamk(m, n, k, ctas):
    _run(m, n, k, 32, ctas)


def test_tile_width_does_not_change_the_bits():
    """Prefill uses 256-row tiles of the token rows when there are enough of them and 128-row tiles otherwise
    (csrc/lm_engine.cu launch_rows_of): per output element the K loop is the same MMA sequence, so the two give the same
    bits -- what keeps chunked prefill, prefix reuse and batch invariance bit-exact."""
    from fish_speech_b200 import _lib

    L = _lib.lib()
    g = torch.Generator().manual_seed(5)
    m, n, k = 640, 700, 2560
    a = (torch.randn(m, k, generator=g) * 0.5).bfloat16().cuda()
    b = (torch.randn(n, k, generator=g) * 0.5).bfloat16().cuda()
    outs = []
    for bn in (64, 128, 256):
        out = torch.full((n, m), float("nan"), device="cuda", dtype=torch.float32)
        _lib.check(L.fsb_op_gemm(a.data_ptr(), b.data_ptr(), out.data_ptr(), m, n, k, bn, 0,
                                 torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        outs.append(out.cpu())
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[1], outs[2])
