"""deterministic=True at 32 < k <= 256: the team-of-warps K23 with fixed-point (int64) sums, the route
that sends the deterministic step through it for every such k (33..64 included, whatever
WSAE_WIDE_K23 says), and bit-reproducible training on top.  Each layer has its own test, so a failure
names one piece."""

import threading

import pytest
import torch

from oracle import topk_sae_oracle as O


def _ops():
    from whisper_sae_b200 import ops
    return ops


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


# ------------------------------------------------------------------------------------------------
# 1. routing (no device needed)
# ------------------------------------------------------------------------------------------------
# (d, k, bf16 decoder, deterministic route, default route - as test_gpu_wide_k.py::test_routing pins it)
_ROUTES = [
    (384, 32, True, True, True),
    (384, 33, True, True, False),
    (384, 48, True, True, False),
    (384, 64, True, True, False),
    (384, 65, True, True, True),
    (768, 256, True, True, True),
    (384, 257, True, False, False),
    (392, 48, True, False, False),
    (392, 128, True, False, False),
    (384, 48, False, False, False),
    (384, 128, False, False, False),
]


@pytest.mark.parametrize("wide_env", [None, "0", "1"])
@pytest.mark.parametrize("d,k,bf16,det,default", _ROUTES)
def test_deterministic_route(d, k, bf16, det, default, wide_env, monkeypatch):
    monkeypatch.delenv("WSAE_FUSED_DECODE", raising=False)
    if wide_env is None:
        monkeypatch.delenv("WSAE_WIDE_K23", raising=False)
    else:
        monkeypatch.setenv("WSAE_WIDE_K23", wide_env)
    ops = _ops()
    assert ops.decode_backward_supported(d, k, bf16, deterministic=True) == det
    # the default mode is untouched: WSAE_WIDE_K23=1 alone moves 33..64 onto the team form
    want = default or (wide_env == "1" and bf16 and d % 128 == 0 and 32 < k <= 64)
    assert ops.decode_backward_supported(d, k, bf16, deterministic=False) == want
    assert ops.decode_backward_supported(d, k, bf16) == want


# ------------------------------------------------------------------------------------------------
# 2. K23 team form with det_ws against the same call without it
# ------------------------------------------------------------------------------------------------
_K23_F = {384: 3072, 768: 6144, 1280: 4096}
_U = 2.0 ** -24          # fp32 unit roundoff


@pytest.mark.gpu
@pytest.mark.parametrize("xdtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("d", [384, 768, 1280])
@pytest.mark.parametrize("k", [33, 64, 65, 128, 256])
def test_k23_wide_deterministic_form(k, d, xdtype):
    """The fp32 target goes through wsae_decode_backward_det (direct), the bf16 one through
    wsae_decode_backward_typed (slot).  Per-row outputs are bit-identical to the default form's; the
    three cross-row sums differ from its float atomics by at most the fixed-point rounding plus the
    float summation error of the default form, bounded per element (n addends, A = sum of |addend|):
      db_enc[f]: n * |s| * 2^-31 + (n + 2) * 2^-24 * A     (addends dot, scale 2^30; A = sum |dv|)
      db_dec[c]: B * |s| * 2^-29 + (B + 2) * 2^-24 * |s| * sum_rows |resid[:, c]|   (<= B block partials, 2^28)
      SSE:       B * 2^-21 + 1e-12 * SSE                                           (<= B block partials, 2^20)"""
    ops = _ops()
    B, F = 301, _K23_F[d]
    torch.manual_seed(k + d)
    state = O.init_state(d, F)
    b_pre = (torch.randn(d) * 0.05).cuda()
    b_dec = (torch.randn(d) * 0.02).cuda()
    w_enc = state["encoder.weight"].cuda()
    w_used = state["decoder.weight"].t().contiguous().to(torch.bfloat16).cuda()
    x = O.synthetic_activations(B, d, seed=3 * B + d).cuda().to(xdtype)
    pre = (x.float() - b_pre) @ w_enc.t() + state["encoder.bias"].cuda()
    val, idx = torch.topk(pre, k, dim=-1)
    val[::3, 0] = -val[::3, 0].abs()                    # relu-masked entries contribute nothing
    val[1::7, k - 1] = -val[1::7, k - 1].abs()          # ... also in the last warp's tail
    idx32, val = idx.to(torch.int32).contiguous(), val.contiguous()
    grad_out, coef = 0.5, 2.0 / (B * d)
    s = coef * grad_out

    def run(det, x=x, idx32=idx32, val=val):
        out = dict(stats=torch.zeros(3, dtype=torch.int64, device="cuda"),
                   last=torch.zeros(F, dtype=torch.int64, device="cuda"),
                   resid=torch.empty(B, d, device="cuda"),
                   resid_bf=torch.empty(B, d, dtype=torch.bfloat16, device="cuda"),
                   dbe=torch.zeros(F, device="cuda"), dbd=torch.zeros(d, device="cuda"),
                   dpre=torch.empty(B, k, device="cuda"))
        kw = dict(resid=out["resid"], resid_bf16=out["resid_bf"], stats=out["stats"], last_activated=out["last"],
                  step_count=torch.tensor(41, dtype=torch.int64, device="cuda"), d_b_enc=out["dbe"],
                  d_b_dec=out["dbd"], dpre_val=out["dpre"],
                  det_ws=torch.zeros(F + d + 1, dtype=torch.int64, device="cuda") if det else None)
        if xdtype == torch.float32:
            tgt, slot = x, False
        else:
            tgt, slot = torch.tensor([x.data_ptr()], dtype=torch.int64, device="cuda"), True
        ops.decode_backward(tgt, w_used, b_dec, b_pre, idx32, val, torch.tensor(grad_out, device="cuda"), coef,
                            target_is_slot=slot, x_dtype=xdtype, **kw)
        torch.cuda.synchronize()
        out["sse"] = out["stats"][:1].view(torch.float64).item()
        return out

    ref, det, det2 = run(False), run(True), run(True)
    for n in ("dpre", "resid", "resid_bf", "last"):
        assert torch.equal(det[n], ref[n]), n
    assert det["stats"][1].item() == ref["stats"][1].item() == int((val > 0).sum())
    assert torch.equal(det["last"] > 0, torch.zeros(F, dtype=torch.bool, device="cuda").index_fill_(
        0, idx[val > 0], True))

    fired = (val > 0).float()
    n_f = torch.zeros(F, device="cuda").index_add_(0, idx.reshape(-1), fired.reshape(-1)).double()
    a_f = torch.zeros(F, device="cuda").index_add_(0, idx.reshape(-1), ref["dpre"].abs().reshape(-1)).double()
    tol_e = n_f * abs(s) * 2.0 ** -31 + (n_f + 2) * _U * a_f
    assert ((det["dbe"].double() - ref["dbe"].double()).abs() <= tol_e).all(), "db_enc"
    assert (det["dbe"] != 0).sum() > 0.5 * (n_f > 0).sum()
    tol_d = B * abs(s) * 2.0 ** -29 + (B + 2) * _U * abs(s) * ref["resid"].double().abs().sum(0)
    assert ((det["dbd"].double() - ref["dbd"].double()).abs() <= tol_d).all(), "db_dec"
    assert abs(det["sse"] - ref["sse"]) <= B * 2.0 ** -21 + 1e-12 * ref["sse"], (det["sse"], ref["sse"])

    # run to run: bit-identical
    for n in ("dbe", "dbd", "dpre", "resid_bf"):
        assert torch.equal(det[n], det2[n]), n
    assert det["sse"] == det2["sse"]

    # order independence of db_enc: the same rows in another order (each feature's addends are integers)
    perm = torch.randperm(B, device="cuda")
    detp = run(True, x=x[perm].contiguous(), idx32=idx32[perm].contiguous(), val=val[perm].contiguous())
    assert torch.equal(detp["dbe"], det["dbe"])
    assert torch.equal(detp["dpre"], det["dpre"][perm])


# ------------------------------------------------------------------------------------------------
# 3. trainer: two deterministic runs are bit-identical
# ------------------------------------------------------------------------------------------------
def _trainer(tmp_path, tag, d, F, k, B, **kw):
    from whisper_sae_b200.config import TrainingConfig
    from whisper_sae_b200.sae import SAETrainer, TopKSAE

    torch.manual_seed(42)
    sae = TopKSAE(d, F, k=k, dead_feature_threshold=10_000)
    cfg = TrainingConfig(batch_size=B, use_amp=True, num_workers=0, learning_rate=1e-3, warmup_steps=2)
    tr = SAETrainer(sae, cfg, device="cuda", run_dir=tmp_path / tag, **kw)
    tr.setup_scheduler(100)
    return tr


def _state(tr):
    torch.cuda.synchronize()
    st = {n: t.detach().clone() for n, t in tr.model.state_dict().items()}
    for i, p in enumerate(tr.model.parameters()):
        s = tr.optimizer.state[p]
        st[f"m{i}"], st[f"v{i}"] = s["exp_avg"].clone(), s["exp_avg_sq"].clone()
    return st


@pytest.mark.gpu
@pytest.mark.parametrize("rows,d,F,k", [
    (75776, 384, 3072, 48), (75776, 384, 3072, 64), (75776, 384, 3072, 128), (75776, 384, 3072, 256),
    (75776, 768, 6144, 128), (2048, 1280, 40960, 128),
    (512, 384, 3072, 128),          # dense K1
])
def test_deterministic_wide_k_is_bit_reproducible(rows, d, F, k, tmp_path, monkeypatch):
    """test_gpu_fullsize.py::test_deterministic_mode_is_bit_reproducible at 32 < k <= 256.  Against the
    default mode (float atomics in arrival order; K2 + K3 at k <= 64): the first step, from the same
    weights, agrees to 1e-5 in the loss with the same fired set; after 5 steps the weights are within
    the wide-k float-atomic tolerance of test_gpu_wide_k.py, 5e-3 rel-L2.  Measured on a B200 (1000 W),
    largest over the four parameters: k = 48 5.7e-4, k = 64 5.1e-4 (against K2 + K3), k = 128 6.9e-6,
    k = 256 1.1e-5 (384 -> 3072); 3.4e-5 (768 -> 6144), 1.0e-4 (1280 -> 40960), 5.6e-7 (512 rows)."""
    monkeypatch.delenv("WSAE_WIDE_K23", raising=False)
    steps = 5
    x = O.synthetic_activations(2 * rows, d, seed=21).cuda()

    def run(deterministic, tag):
        tr = _trainer(tmp_path, tag, d, F, k, rows, deterministic=deterministic)
        ms = [tr.train_step(x[:rows])]
        fired0 = tr.model.feature_last_activated.clone()
        ms += [tr.train_step(x[(s % 2) * rows:(s % 2 + 1) * rows]) for s in range(1, steps)]
        gs = tr._graphs[rows]
        assert gs.graph is not None and gs.det == deterministic
        return tr, [(m.loss, m.l0, m.dead_feature_ratio) for m in ms], fired0, _state(tr)

    ta, la, fa, sa = run(True, "a")
    _, lb, _, sb = run(True, "b")
    assert la == lb, "deterministic mode: losses differ between two runs"
    for n in sa:
        assert torch.equal(sa[n], sb[n]), f"deterministic mode: {n} differs between two runs"
    ga = ta._graphs[rows]
    assert ga.in_place and ga._x is None and ga.state.resid is None      # K23 (team form), not K2 + K3
    assert not ga.row_step
    tc, lc, fc, sc = run(False, "c")
    if k <= 64:          # the default mode keeps K2 + K3 at 33..64
        assert tc._graphs[rows].state.resid is not None
    assert la[0][0] == pytest.approx(lc[0][0], rel=1e-5) and la[0][1] == lc[0][1]
    assert torch.equal(fa, fc)
    for n in ("encoder.weight", "decoder.weight", "encoder.bias", "decoder.bias"):
        rel = _rel(sa[n], sc[n])
        assert rel < 5e-3, f"{n}: deterministic vs default rel-L2 {rel:.2e}"


@pytest.mark.gpu
def test_deterministic_wide_k_needs_d_multiple_of_128(tmp_path):
    tr = _trainer(tmp_path, "d392", 392, 3072, 128, 4096, deterministic=True)
    with pytest.raises(RuntimeError, match=r"d % 128 == 0 and k <= 256"):
        tr.train_step(O.synthetic_activations(4096, 392, seed=1).cuda())


# ------------------------------------------------------------------------------------------------
# 4. inputs: half-precision batches, IndexedBatch, two emulated ranks
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("k", [48, 128])
@pytest.mark.parametrize("indexed", [False, True])
def test_deterministic_wide_k_half_is_bit_identical(dtype, k, indexed, tmp_path, monkeypatch):
    """test_gpu_half_inputs.py::test_trainer_deterministic_half_is_bit_identical at k = 48 and 128: a
    half batch, read in place, trains exactly as its fp32 copy."""
    from whisper_sae_b200.data.feature_cache import ResidentBatches

    monkeypatch.delenv("WSAE_WIDE_K23", raising=False)
    B, d, F, steps = 8192, 384, 3072, 6
    xh = O.synthetic_activations(B * 2, d, seed=B + k).cuda().to(dtype)
    runs = {}
    for name, x in (("half", xh), ("fp32", xh.float())):
        tr = _trainer(tmp_path, name, d, F, k, B, deterministic=True)
        if indexed:
            batches = []
            while len(batches) < steps:
                batches += [b[0] for b in ResidentBatches(x, B, True, "cuda", seed=5)]
            batches = batches[:steps]
        else:
            batches = [x[(s % 2) * B:(s % 2 + 1) * B] for s in range(steps)]
        ms = [tr.train_step(b) for b in batches]
        runs[name] = (tr, ms, _state(tr))
    (th, mh, sh), (tf, mf, sf) = runs["half"], runs["fp32"]
    assert [(m.loss, m.l0, m.dead_feature_ratio) for m in mh] == [(m.loss, m.l0, m.dead_feature_ratio) for m in mf]
    for n in sf:
        assert torch.equal(sh[n], sf[n]), n
    gh = th._graphs[B]
    assert gh.det and gh.graph is not None and gh.x_dtype == dtype
    assert gh._x is None, "a device half batch must be read in place, not staged"


@pytest.mark.gpu
def test_deterministic_wide_k_two_ranks(tmp_path):
    """Two emulated ranks (replicated exchange, summed in rank order) with deterministic=True at
    k = 128, run twice: losses and consolidated weights are bit-identical between the runs and
    between the ranks."""
    from whisper_sae_b200.sae import parallel

    k, B, d, F, steps = 128, 8192, 384, 3072, 5
    x = O.synthetic_activations(B * steps, d, seed=17).cuda()

    def run(tag):
        comms = parallel.ThreadCommunicator.make(2)
        ranks = [_trainer(tmp_path, f"{tag}{r}", d, F, k, B // 2, data_parallel=True, dp_comm=c,
                          deterministic=True) for r, c in enumerate(comms)]
        got = [[None] * steps for _ in range(2)]
        errors = []

        def work(r):
            try:
                torch.cuda.set_device(0)
                for s in range(steps):
                    a, b = parallel.shard_rows(B, 2, r)
                    got[r][s] = ranks[r].train_step(x[s * B + a:s * B + b])
            except Exception as e:  # noqa: BLE001
                errors.append(e)
                comms[r].shared.barrier.abort()

        ts = [threading.Thread(target=work, args=(r,)) for r in range(2)]
        [t.start() for t in ts]
        [t.join() for t in ts]
        assert not errors, errors
        ts = [threading.Thread(target=ranks[r].consolidate_weights) for r in range(2)]
        [t.start() for t in ts]
        [t.join() for t in ts]
        for tr in ranks:
            gs = tr._graphs[B // 2]
            assert gs.det and not gs.shard and gs.in_place
        return [[m.loss for m in g] for g in got], [_state(tr) for tr in ranks]

    l1, s1 = run("a")
    l2, s2 = run("b")
    assert l1[0] == l1[1] == l2[0] == l2[1]
    for n in s1[0]:
        assert torch.equal(s1[0][n], s1[1][n]), ("ranks", n)
        assert torch.equal(s1[0][n], s2[0][n]), ("runs", n)
        assert torch.equal(s2[0][n], s2[1][n]), ("ranks, run 2", n)
