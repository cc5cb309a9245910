"""The train-step kernels at shapes of real Whisper SAEs that the BASELINE configs do not reach: the base
(d = 512) and medium (d = 1024) widths, and more than 65 536 features.

K1 is checked exactly: its values must be bit for bit the pre-activations of ``ops.encode_dense`` at
the returned indices, and its index set must be the first k of a stable descending sort of that fp32
matrix (ties to the lowest index, NaN never selected).  Every other comparison is against float64
evaluated on the same bf16-rounded operands the kernel reads, so what is left is fp32 accumulation.
That is bounded per element by the size of the element's own terms:

    |got - ref| <= C * 2^-24 * n * (|A|^T |B|)_ij      (n = number of terms summed into the element)

C = 2 allows for the tensor core's accumulation.  The worst measured ratio of error to bound of each
comparison on a B200 is written beside it.  References are computed with torch on the GPU: the CPU
oracle is too slow at these sizes."""

import pytest
import torch

pytestmark = pytest.mark.gpu

C = 2.0
U = 2.0 ** -24            # fp32 unit roundoff


def _ops():
    from whisper_sae_b200 import ops
    return ops


def _within(got, ref, bound, name):
    """max |got - ref| / bound over the elements; an element with bound 0 must be exact."""
    err = (got.double() - ref).abs()
    ratio = (err / bound.clamp_min(1e-300)).max().item()
    print(f"{name}: worst error / bound = {ratio:.3g}")
    assert ratio <= 1.0, f"{name}: error exceeds the per-element bound by {ratio:.3g}x"
    return ratio


# ------------------------------------------------------------------------------------------------
# 1. K1 at any F
# ------------------------------------------------------------------------------------------------
def _k1_operands(B, d, F, seed, nan_features=()):
    """Packed bf16 operands.  Row 1 is all zeros, so with the constant bias every pre-activation of it
    ties; row 2 is NaN, so it has no valid pre-activation.  ``nan_features``: NaN encoder rows, NaN in
    every row's pre-activations at those features."""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, d, device="cuda", generator=g)
    x[1] = 0.0
    x[2] = float("nan")
    w = torch.randn(F, d, device="cuda", generator=g) / d ** 0.5
    w[list(nan_features)] = float("nan")
    b = torch.full((F,), 0.25, device="cuda")
    return ops.pack_activations(x, None, 1), ops.pack_encoder(w, b, 1)


def _dense_pre(a, w, B, F, d):
    """encode_dense's fp32 [B, F] on the same packed operands (it stores 16-byte vectors, so F % 4 != 0
    is computed at the next multiple of 4 over the zero padding rows of the packed encoder)."""
    F4 = (F + 3) // 4 * 4
    return _ops().encode_dense(a, w, B, F4, d, 1)[:, :F]


def _check_topk_exact(idx, val, pre, k):
    B, F = pre.shape
    nan = torch.isnan(pre)
    key = pre.masked_fill(nan, float("-inf"))
    want = torch.sort(key, dim=1, descending=True, stable=True).indices[:, :k]
    n_valid = (~nan).sum(1, keepdim=True)
    want = torch.where(torch.arange(k, device=pre.device) < n_valid, want, -1)
    got = idx.long()
    assert torch.equal(torch.sort(got, 1).values, torch.sort(want, 1).values), \
        f"{int((torch.sort(got, 1).values != torch.sort(want, 1).values).any(1).sum())} rows differ"
    ok = got >= 0
    assert torch.equal(val[ok], pre.gather(1, got.clamp_min(0))[ok]), "values are not the fp32 pre-activations"
    assert bool((val[~ok] == float("-inf")).all())


@pytest.mark.parametrize("F", [51200, 81920, 131072, 3002])
@pytest.mark.parametrize("k", [65, 128, 256])
@pytest.mark.parametrize("B", [100, 1300])
def test_k1_chunked_any_f_exact(B, F, k):
    """k > 64 (the chunked route): column slices above 49 152 features and their merge, and a row pitch
    for F % 4 != 0; one chunk (100 rows) and several (1300 rows)."""
    ops = _ops()
    d = 1024 if k == 128 else 512
    assert ops.encode_route(B, F, k) == "chunked"
    a, w = _k1_operands(B, d, F, seed=B + F + k, nan_features=(0, 7, F - 1))
    idx, val = ops.encode_topk(a, w, B, F, d, 1, k)
    pre = _dense_pre(a, w, B, F, d)
    torch.cuda.synchronize()
    _check_topk_exact(idx, val, pre, k)
    lowest = [f for f in range(k + 2) if f not in (0, 7)][:k]           # all-equal row: the lowest non-NaN
    assert idx[1].tolist() == lowest and bool((idx[2] == -1).all())
    full = idx[(idx >= 0).all(1)]
    assert bool((full[:, 1:] > full[:, :-1]).all()), "ascending feature order"


@pytest.mark.parametrize("F", [81920, 131072])
@pytest.mark.parametrize("k", [32, 64])
@pytest.mark.parametrize("B,nsplit", [(300, 8), (1300, 16), (1300, None)])
def test_k1_fused_wide_f_exact(B, F, k, nsplit):
    """k <= 64 (the fused route) above 65 536 features, with an F-split whose lists the merge reduces;
    1300 rows run the CTA-pair kernel."""
    ops = _ops()
    d = 512 if k == 32 else 1024
    assert ops.encode_route(B, F, k, nsplit) == "fused"
    if nsplit is not None:
        assert ops._lib.load().wsae_encode_effective_splits(F, nsplit) > 1
    a, w = _k1_operands(B, d, F, seed=B + F + k)
    idx, val = ops.encode_topk(a, w, B, F, d, 1, k, nsplit=nsplit)
    pre = _dense_pre(a, w, B, F, d)
    torch.cuda.synchronize()
    _check_topk_exact(idx, val, pre, k)


def test_k1_chunked_slice_limit():
    """The merge keeps at most 64 candidates per lane: F up to 8 x 49 152 at k = 256, and above that
    WSAE_E_UNSUPPORTED, not a wrong answer."""
    ops = _ops()
    B, d, k = 130, 64, 256
    F = 8 * 49152
    a, w = _k1_operands(B, d, F, seed=1)
    idx, val = ops.encode_topk(a, w, B, F, d, 1, k)
    _check_topk_exact(idx, val, _dense_pre(a, w, B, F, d), k)
    a, w = _k1_operands(8, d, F + 1, seed=2)
    with pytest.raises(RuntimeError, match="wsae_encode_topk_chunked"):
        ops.encode_topk(a, w, 8, F + 1, d, 1, k)
        torch.cuda.synchronize()


@pytest.mark.parametrize("B,d,F", [(1300, 512, 81920), (300, 1024, 131072), (1000, 1024, 3004)])
def test_encode_dense_matches_float64(B, d, F):
    """The GEMM of K1 against float64 of the packed operands (d bf16 products and three bias pieces per
    element).  Worst error / bound measured on a B200 (1000 W): 0.0055."""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(B + d)
    x = torch.randn(B, d, device="cuda", generator=g)
    w = torch.randn(F, d, device="cuda", generator=g) / d ** 0.5
    b = torch.randn(F, device="cuda", generator=g) * 0.1
    a, wp = ops.pack_activations(x, None, 1), ops.pack_encoder(w, b, 1)
    got = ops.encode_dense(a, wp, B, F, d, 1)
    A, W = a[:B].double(), wp[:F].double()
    ref = A @ W.t()
    bound = C * U * (d + 3) * (A.abs() @ W.abs().t())
    _within(got, ref, bound, f"encode_dense {B}x{d}->{F}")


# ------------------------------------------------------------------------------------------------
# 2. K4 at nb_tile = 8 with training-like data
# ------------------------------------------------------------------------------------------------
def _skewed_entries(B, F, k, seed):
    """k distinct features per row: eight hot features in feature tile 1 fire in ~97 % of rows (a
    (tile, 64-row chunk) cell then holds ~500 entries), a power law over the rest, and feature tiles
    3..9 never fire.  About a third of the entries are inactive (value <= 0)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    weight = torch.rand(F, device="cuda", generator=g) ** 4
    weight[3 * 128:10 * 128] = -1.0
    scores = torch.rand(B, F, device="cuda", generator=g) * weight
    hot = torch.arange(8, device="cuda") * 16 + 128
    scores[:, hot] += 2.0 * (torch.rand(B, 8, device="cuda", generator=g) < 0.97)
    idx = scores.topk(k, dim=1).indices.to(torch.int32)
    del scores
    val = torch.randn(B, k, device="cuda", generator=g) + 0.5
    dpre = torch.randn(B, k, device="cuda", generator=g) * (val > 0)
    return idx, val, dpre


@pytest.mark.parametrize("d", [512, 1024, 1536])
@pytest.mark.parametrize("k", [32, 128, 256])
@pytest.mark.parametrize("B,F", [(1000, 8320), (16384, 8192)])
def test_wgrad_gemm_nb_tile8_skewed(B, F, k, d):
    """bucket_by_tile + wgrad_gemm_ (and its split-K slab form with det_ws) at the widths whose N tile is
    8 x 64 (two pipeline stages, a second MMA at N = 256, all 512 TMEM columns), on a ragged batch with
    an odd feature-tile count (8320 = 65 x 128) and on a 16 384-row batch with an even one.
    Worst error / bound measured on a B200 (1000 W), over all cases: 0.25 (dpre values), 0.23 (activations),
    the same with det_ws."""
    ops = _ops()
    idx, val, dpre = _skewed_entries(B, F, k, seed=B + F + k + d)
    g = torch.Generator(device="cuda").manual_seed(d)
    R = torch.randn(B, d, device="cuda", generator=g).to(torch.bfloat16)
    buckets = ops.bucket_by_tile(idx, val, dpre, F)
    n_chunks, n_ft = ops.bucket_cells(B, F)
    offs = buckets.offsets.view(n_chunks, n_ft + 1).long()
    active = int((val > 0).sum())
    assert torch.equal(offs[:, 0].cpu(), torch.arange(n_chunks) * 64 * k)
    assert int((offs[:, -1] - offs[:, 0]).sum()) == active
    assert bool((offs[:, 1:] >= offs[:, :-1]).all())
    cells = offs[:, 1:n_ft + 1] - offs[:, :n_ft]
    assert int(cells.max()) > 256, "no crowded cell"
    assert bool((cells[:, 3:10] == 0).all()), "dead tiles hold entries"

    Rd = R.double()
    act = (val > 0)
    nnz = torch.zeros(F, device="cuda", dtype=torch.float64).index_add_(
        0, idx[act].long(), torch.ones(active, device="cuda", dtype=torch.float64))
    ws_bytes = ops.wgrad_gemm_workspace(B, F, d)
    det_ws = torch.empty(max(ws_bytes // 4, 1), dtype=torch.float32, device="cuda")
    init = torch.randn(F, d, device="cuda", generator=g) * 0.1
    go = torch.tensor(1.5, device="cuda")
    for values_d, values, alpha, name in ((buckets.dpre, dpre, 1.0, "dpre"),
                                          (buckets.act, val.clamp_min(0), 0.25, "act")):
        S = torch.zeros(B, F, dtype=torch.float64, device="cuda")
        S.scatter_(1, idx.long(), (values * act).to(torch.bfloat16).double())
        scale = 1.5 * alpha
        ref = init.double() + scale * (S.t() @ Rd)
        absprod = init.double().abs() + abs(scale) * (S.abs().t() @ Rd.abs())
        del S
        bound = C * U * (nnz + 3).unsqueeze(1) * absprod
        outs = []
        for ws in (None, det_ws, det_ws):
            out = init.clone()
            ops.wgrad_gemm_(out, R, B, d, buckets, values_d, go, alpha, det_ws=ws)
            outs.append(out)
        torch.cuda.synchronize()
        _within(outs[0], ref, bound, f"K4 {name} {B}x{d} F={F} k={k}")
        _within(outs[1], ref, bound, f"K4 det {name} {B}x{d} F={F} k={k}")
        assert torch.equal(outs[1], outs[2]), "det_ws form differs between two calls"


# ------------------------------------------------------------------------------------------------
# 3. K23 above 65 536 features (stamps in global memory) and at d = 512 / 1024
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d,F", [(512, 81920), (1024, 81920), (1024, 8192)])
@pytest.mark.parametrize("k", [32, 128, 256])
@pytest.mark.parametrize("det", [False, True])
def test_k23_wide_f_matches_float64(d, F, k, det):
    """The test_decode_backward_fused recipe (tensor form at k = 32, team form at 128 / 256), default and
    deterministic, evaluated in float64 with per-element bounds.  The deterministic form's fixed-point
    sums add their quantum per addend (db_enc 2^-31 |s|, db_dec 2^-29 |s| per row).
    Worst error / bound measured on a B200 (1000 W), over all cases: resid 0.025, dpre 1.3e-3, db_enc 0.19
    (0.24 deterministic), db_dec 1.4e-3."""
    ops = _ops()
    B = 1000
    g = torch.Generator(device="cuda").manual_seed(d + F + k)
    x = torch.randn(B, d, device="cuda", generator=g)
    b_pre = torch.randn(d, device="cuda", generator=g) * 0.05
    b_dec = torch.randn(d, device="cuda", generator=g) * 0.02
    w_dec = torch.randn(F, d, device="cuda", generator=g)
    w_dec = (w_dec / w_dec.norm(dim=1, keepdim=True)).to(torch.bfloat16)
    idx = torch.rand(B, F, device="cuda", generator=g).topk(k, dim=1).indices.to(torch.int32)
    val = torch.randn(B, k, device="cuda", generator=g).abs() + 0.1
    val[::3, 0] = -val[::3, 0]                          # relu-masked entries contribute nothing
    val[1::7, k - 1] = -val[1::7, k - 1]                # ... also in the last warp's tail
    grad_out, coef = 0.5, 2.0 / (B * d)
    s = coef * grad_out
    assert ops.decode_backward_supported(d, k, True, deterministic=det)
    out = dict(stats=torch.zeros(3, dtype=torch.int64, device="cuda"),
               last=torch.zeros(F, dtype=torch.int64, device="cuda"),
               resid=torch.empty(B, d, device="cuda"),
               resid_bf=torch.empty(B, d, dtype=torch.bfloat16, device="cuda"),
               dbe=torch.zeros(F, device="cuda"), dbd=torch.zeros(d, device="cuda"),
               dpre=torch.empty(B, k, device="cuda"))
    ops.decode_backward(x, w_dec, b_dec, b_pre, idx, val, torch.tensor(grad_out, device="cuda"), coef,
                        resid=out["resid"], resid_bf16=out["resid_bf"], stats=out["stats"],
                        last_activated=out["last"], step_count=torch.tensor(41, dtype=torch.int64, device="cuda"),
                        d_b_enc=out["dbe"], d_b_dec=out["dbd"], dpre_val=out["dpre"],
                        det_ws=torch.zeros(F + d + 1, dtype=torch.int64, device="cuda") if det else None)
    torch.cuda.synchronize()
    tag = f"K23{' det' if det else ''} d={d} F={F} k={k}"
    fired = val > 0
    rows = w_dec.double()[idx.long()]                                  # [B, k, d]
    h = torch.relu(val).to(torch.bfloat16).double()
    terms = h.unsqueeze(-1) * rows
    resid_ref = terms.sum(1) + b_dec.double() + b_pre.double() - x.double()
    abs_r = terms.abs().sum(1) + b_dec.double().abs() + b_pre.double().abs() + x.double().abs()
    _within(out["resid"], resid_ref, C * U * (k + 3) * abs_r, tag + " resid")
    assert torch.equal(out["resid_bf"], out["resid"].to(torch.bfloat16))
    # dv uses the bf16 residual the kernel rounded (the operand K4 reads)
    prod = out["resid_bf"].double().unsqueeze(1) * rows                # [B, k, d]
    dv_ref = s * prod.sum(-1) * fired
    _within(out["dpre"], dv_ref, C * U * (d + 2) * abs(s) * prod.abs().sum(-1), tag + " dpre")
    del prod, rows, terms
    # the cross-row sums, over the kernel's own per-row outputs
    dp = out["dpre"].double()
    flat = idx.reshape(-1).long()
    dbe_ref = torch.zeros(F, dtype=torch.float64, device="cuda").index_add_(0, flat, dp.reshape(-1))
    dbe_abs = torch.zeros(F, dtype=torch.float64, device="cuda").index_add_(0, flat, dp.abs().reshape(-1))
    n_f = torch.zeros(F, dtype=torch.float64, device="cuda").index_add_(0, flat, fired.reshape(-1).double())
    bound_e = C * U * (n_f + 2) * dbe_abs + (n_f * abs(s) * 2.0 ** -31 if det else 0.0)
    _within(out["dbe"], dbe_ref, bound_e, tag + " db_enc")
    r = out["resid"].double()
    bound_d = C * U * (B + 2) * abs(s) * r.abs().sum(0) + (B * abs(s) * 2.0 ** -29 if det else 0.0)
    _within(out["dbd"], s * r.sum(0), bound_d, tag + " db_dec")
    sse = out["stats"][:1].view(torch.float64).item()
    sse_ref = (r ** 2).sum().item()
    assert abs(sse - sse_ref) <= 1e-6 * sse_ref + (B * 2.0 ** -21 if det else 0.0), (sse, sse_ref)
    assert out["stats"][1].item() == int(fired.sum())
    want_last = torch.zeros(F, dtype=torch.int64, device="cuda")
    want_last[idx[fired].long()] = 42
    assert torch.equal(out["last"], want_last)
