"""K4 (tensor-core weight-gradient GEMM with in-SMEM sparse operand expansion) against a dense
fp32 torch reference of the same product: OUT = alpha * S^T @ R, S = scatter(values at idx)."""

import pytest
import torch

pytestmark = pytest.mark.gpu


def _case(B, d, F, k, seed, pitch=None):
    from whisper_sae_b200 import ops

    g = torch.Generator().manual_seed(seed)
    dev = "cuda"
    scores = torch.rand(B, F, generator=g)
    idx = scores.topk(k, dim=1).indices.to(torch.int32)            # unique per row
    val = torch.randn(B, k, generator=g)                            # ~half inactive (<= 0)
    dpre = torch.randn(B, k, generator=g) * (val > 0)
    pitch = pitch or d
    R = torch.zeros(B, pitch)
    R[:, :d] = torch.randn(B, d, generator=g)
    R_bf = R.to(torch.bfloat16)
    idx_d, val_d, dpre_d, R_d = idx.to(dev), val.to(dev), dpre.to(dev), R_bf.to(dev)
    buckets = ops.bucket_by_tile(idx_d, val_d, dpre_d, F)
    n_chunks, n_ft = ops.bucket_cells(B, F)
    offs = buckets.offsets.cpu().view(n_chunks, n_ft + 1)    # per 64-row chunk: cell starts + end
    active = int((val > 0).sum())
    assert torch.equal(offs[:, 0], torch.arange(n_chunks, dtype=torch.int32) * 64 * k)
    assert int((offs[:, -1] - offs[:, 0]).sum()) == active
    assert bool((offs[:, 1:] >= offs[:, :-1]).all())

    def dense(values):
        S = torch.zeros(B, F, dtype=torch.float64)
        S.scatter_(1, idx.long(), (values * (val > 0)).to(torch.bfloat16).double())
        return S.t() @ R_bf[:, :d].double()

    for values_d, values, alpha in ((buckets.dpre, dpre, 1.0), (buckets.act, val.clamp_min(0), 0.25)):
        out = torch.full((F, d), 0.5, dtype=torch.float32, device=dev)   # accumulates (+=)
        go = torch.tensor(2.0, device=dev)
        ops.wgrad_gemm_(out, R_d, B, d, buckets, values_d, go, alpha)
        ref = 0.5 + 2.0 * alpha * dense(values)
        err = (out.cpu().double() - ref).abs().max().item()
        scale = ref.abs().max().item()
        assert err <= 2e-5 * scale + 1e-5, (B, d, F, k, err, scale)


@pytest.mark.parametrize("B,d,F,k", [
    (64, 64, 128, 4),
    (100, 64, 200, 8),          # ragged rows / features
    (256, 384, 3072, 32),       # whisper-tiny
    (1000, 96, 1000, 16),       # d not a multiple of 64
    (512, 768, 6144, 32),       # whisper-small (N = 768: three MMAs per k-step? -> n tiles)
    (300, 1280, 2048, 32),      # large-v3 width (n tiles of 7*64 / 6*64 columns)
    (300, 512, 4096, 32),       # whisper-base: 8 x 64-column n tiles, 2 stages, second MMA at N = 256
    (200, 1024, 2176, 32),      # whisper-medium: the same n tiling, odd feature-tile count
])
def test_wgrad_gemm_matches_dense(B, d, F, k):
    _case(B, d, F, k, seed=B + d)


def test_wgrad_gemm_padded_pitch():
    _case(384, 384, 3072, 32, seed=5, pitch=448)      # the packed-activation layout (Kp = 448)


def test_wgrad_large_batch_linearity():
    """Full bench size: GEMM(S, R1 + R2) == GEMM(S, R1) + GEMM(S, R2) up to bf16 rounding of R."""
    from whisper_sae_b200 import ops

    B, d, F, k = 16384, 384, 3072, 32
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(7)
    idx = torch.rand(B, F, device=dev, generator=g).topk(k, dim=1).indices.to(torch.int32)
    val = torch.rand(B, k, device=dev, generator=g) + 0.1
    dpre = torch.randn(B, k, device=dev, generator=g)
    buckets = ops.bucket_by_tile(idx, val, dpre, F)
    R1 = (torch.randint(-8, 9, (B, d), device=dev, generator=g).float() / 8).to(torch.bfloat16)
    R2 = (torch.randint(-8, 9, (B, d), device=dev, generator=g).float() / 8).to(torch.bfloat16)
    outs = []
    for R in (R1, R2, (R1 + R2)):
        out = torch.zeros(F, d, device=dev)
        ops.wgrad_gemm_(out, R.contiguous(), B, d, buckets, buckets.dpre, None, 1.0)
        outs.append(out)
    err = (outs[0] + outs[1] - outs[2]).abs().max().item()
    assert err <= 1e-3 * outs[2].abs().max().item()
    # and against a dense product on a feature slice
    S = torch.zeros(B, F, device=dev)
    S.scatter_(1, idx.long(), dpre.to(torch.bfloat16).float())
    ref = S[:, :256].t() @ R1.float()
    assert (outs[0][:256] - ref).abs().max().item() <= 1e-3 * ref.abs().max().item()
