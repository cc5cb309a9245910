"""Half-precision activation matrices (bf16 / fp16) as a first-class input of the graphed bf16 step.

A bf16 or fp16 value converts to fp32 exactly, and the kernels convert at the load and then run the
fp32 arithmetic.  So everything here is checked against the same computation on ``Xh.float()``: bit for
bit wherever the fp32 path is deterministic, and to float-atomic summation-order noise where it is not.
Each layer has its own test, so a failure names one piece."""

import threading

import pytest
import torch

from oracle import topk_sae_oracle as O

HALF = [torch.bfloat16, torch.float16]


def _ops():
    from whisper_sae_b200 import ops
    return ops


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def _slot(t):
    return torch.tensor([t.data_ptr()], dtype=torch.int64, device="cuda")


# ------------------------------------------------------------------------------------------------
# 1. routing and dtype codes (no device needed)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,ok", [(torch.float32, True), (torch.bfloat16, True), (torch.float16, True),
                                      (torch.float64, False), (torch.int32, False), (torch.int64, False)])
def test_graph_ok_accepts_half_batches(dtype, ok):
    from whisper_sae_b200.data.feature_cache import IndexedBatch
    from whisper_sae_b200.sae import TopKSAE
    from whisper_sae_b200.sae.training import SAETrainer

    class _Stub:         # _graph_ok reads these attributes only
        cuda_graph = True
        model = TopKSAE(384, 3072, k=32)
    assert SAETrainer._graph_ok(_Stub(), torch.zeros(4, 384, dtype=dtype)) == ok
    if dtype.is_floating_point:
        batch = IndexedBatch(torch.zeros(16, 384, dtype=dtype), torch.arange(4))
        assert SAETrainer._graph_ok(_Stub(), batch) == ok


def test_dtype_codes_match_the_layernorm_convention():
    ops = _ops()
    assert ops._LN_DTYPES == {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}
    for dt, code in ops._LN_DTYPES.items():
        assert ops._x_dtype_code(dt) == code
    with pytest.raises(RuntimeError):
        ops._x_dtype_code(torch.float64)


# ------------------------------------------------------------------------------------------------
# 2. kernels: K0, K23, the row step, LayerNorm
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("d", [384, 392])
def test_k0_pack_half_matches_fp32(dtype, d):
    ops = _ops()
    B, N = 1000, 3000
    xh = O.synthetic_activations(N, d, seed=d).cuda().to(dtype)
    x32 = xh.float()
    b_pre = (0.1 * torch.randn(d, generator=torch.Generator().manual_seed(1))).cuda()
    perm = torch.randperm(N, device="cuda")[:B]
    for rows in (None, perm):
        rs = None if rows is None else _slot(rows)
        a = ops.pack_activations_at(_slot(xh), B, d, b_pre, rows_at=rs, x_dtype=dtype)
        b = ops.pack_activations_at(_slot(x32), B, d, b_pre, rows_at=rs)
        assert torch.equal(a.view(torch.int16), b.view(torch.int16))
    with pytest.raises(RuntimeError):          # the multi-term pack reads fp32 only
        ops.pack_activations(xh, b_pre, 3)


def _k23(x, rows_at, dtype, w, b_dec, b_pre, idx, val, F, det):
    ops = _ops()
    B, k = idx.shape
    d = w.shape[1]
    out = dict(resid_bf=torch.empty(B, d, dtype=torch.bfloat16, device="cuda"),
               stats=torch.zeros(3, dtype=torch.int64, device="cuda"),
               last=torch.zeros(F, dtype=torch.int64, device="cuda"),
               dbe=torch.zeros(F, device="cuda"), dbd=torch.zeros(d, device="cuda"),
               dpre=torch.empty(B, k, device="cuda"))
    step = torch.tensor([6], dtype=torch.int64, device="cuda")
    det_ws = torch.zeros(F + d + 1, dtype=torch.int64, device="cuda") if det else None
    ops.decode_backward(_slot(x), w, b_dec, b_pre, idx, val, None, 1e-3, resid=None, resid_bf16=out["resid_bf"],
                        stats=out["stats"], last_activated=out["last"], step_count=step, d_b_enc=out["dbe"],
                        d_b_dec=out["dbd"], dpre_val=out["dpre"], target_is_slot=True, rows_at=rows_at,
                        det_ws=det_ws, x_dtype=dtype)
    torch.cuda.synchronize()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("form,d,k,det", [("warp", 392, 32, False), ("tensor", 384, 32, False),
                                          ("team", 384, 128, False), ("det", 384, 32, True)])
def test_k23_half_matches_fp32(dtype, form, d, k, det):
    B, N, F = 4096, 6000, 3072
    g = torch.Generator(device="cuda").manual_seed(d + k)
    xh = O.synthetic_activations(N, d, seed=k).cuda().to(dtype)
    x32 = xh.float()
    w = (torch.randn(F, d, device="cuda", generator=g) / d ** 0.5).to(torch.bfloat16)
    b_dec = 0.1 * torch.randn(d, device="cuda", generator=g)
    b_pre = 0.1 * torch.randn(d, device="cuda", generator=g)
    idx = torch.rand(B, F, device="cuda", generator=g).topk(k, dim=1).indices.to(torch.int32)
    val = torch.randn(B, k, device="cuda", generator=g)            # some entries do not fire
    rows = torch.randperm(N, device="cuda", generator=g)[:B]
    rs = _slot(rows)
    a = _k23(xh, rs, dtype, w, b_dec, b_pre, idx, val, F, det)
    b = _k23(x32, rs, torch.float32, w, b_dec, b_pre, idx, val, F, det)
    assert torch.equal(a["resid_bf"].view(torch.int16), b["resid_bf"].view(torch.int16))
    assert torch.equal(a["dpre"], b["dpre"])
    assert torch.equal(a["last"], b["last"]) and int(a["stats"][1]) == int(b["stats"][1])
    sse_a, sse_b = (o["stats"][:1].view(torch.float64).item() for o in (a, b))
    if det:       # every sum is order-independent: all outputs bit-identical
        assert sse_a == sse_b
        assert torch.equal(a["dbe"], b["dbe"]) and torch.equal(a["dbd"], b["dbd"])
    else:         # float atomics in arrival order
        assert sse_a == pytest.approx(sse_b, rel=1e-6)
        assert _rel(a["dbe"], b["dbe"]) < 1e-6 and _rel(a["dbd"], b["dbd"]) < 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("B", [128, 512])
def test_row_step_half_matches_fp32(dtype, B):
    ops = _ops()
    d, F, k = 384, 3072, 32
    g = torch.Generator(device="cuda").manual_seed(B)
    xh = O.synthetic_activations(B, d, seed=B).cuda().to(dtype)
    pre = torch.randn(B, F, device="cuda", generator=g)
    w_enc = torch.randn(F, d, device="cuda", generator=g) / d ** 0.5
    w = (torch.randn(F, d, device="cuda", generator=g) / d ** 0.5).to(torch.bfloat16)
    b_dec = 0.1 * torch.randn(d, device="cuda", generator=g)
    b_pre = 0.1 * torch.randn(d, device="cuda", generator=g)
    outs = []
    for x in (xh, xh.float()):
        o = dict(stats=torch.zeros(3, dtype=torch.int64, device="cuda"),
                 last=torch.zeros(F, dtype=torch.int64, device="cuda"),
                 dbe=torch.zeros(F, device="cuda"), dbd=torch.zeros(d, device="cuda"),
                 dwe=torch.zeros(F, d, device="cuda"), dwd=torch.zeros(F, d, device="cuda"),
                 dbp=torch.zeros(d, device="cuda"), resid=torch.empty(B, d, device="cuda"),
                 dpre=torch.empty(B, k, device="cuda"))
        step = torch.tensor([3], dtype=torch.int64, device="cuda")
        o["idx"], o["val"] = ops.row_step(pre, x, w, b_dec, b_pre, None, 1e-3, k, stats=o["stats"],
                                          last_activated=o["last"], step_count=step, d_b_enc=o["dbe"],
                                          d_b_dec=o["dbd"], d_w_enc=o["dwe"], d_w_decT=o["dwd"], resid=o["resid"],
                                          dpre_val=o["dpre"], w_enc=w_enc, d_b_pre=o["dbp"])
        torch.cuda.synchronize()
        outs.append(o)
    a, b = outs
    for n in ("idx", "val", "resid", "dpre", "last"):
        assert torch.equal(a[n], b[n]), n
    assert int(a["stats"][1]) == int(b["stats"][1])
    for n in ("dwe", "dwd", "dbe", "dbd", "dbp"):
        assert _rel(a[n], b[n]) < 1e-6, n


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("in_dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_layernorm_half_output_is_fp32_rounded(dtype, in_dtype):
    ops = _ops()
    rows, d = 1500, 384
    g = torch.Generator().manual_seed(7)
    x = (torch.randn(rows, d, generator=g) * 3 + 0.5).to(in_dtype).cuda()
    gamma = (1 + 0.2 * torch.randn(d, generator=g)).cuda()
    beta = (0.3 * torch.randn(d, generator=g)).cuda()
    ref = torch.empty(rows, d, device="cuda")
    ops.layernorm_rows_(x, gamma, beta, 1e-5, ref)
    out = torch.zeros(rows + 4, d, dtype=dtype, device="cuda")
    ops.layernorm_rows_(x, gamma, beta, 1e-5, out, row0=2)
    assert torch.equal(out[2:2 + rows], ref.to(dtype))
    assert not out[:2].any() and not out[2 + rows:].any()


# ------------------------------------------------------------------------------------------------
# 3. trainer
# ------------------------------------------------------------------------------------------------
def _trainer(tmp_path, tag, d, F, k, B, **kw):
    from whisper_sae_b200.config import TrainingConfig
    from whisper_sae_b200.sae import SAETrainer, TopKSAE

    use_amp = kw.pop("use_amp", True)
    torch.manual_seed(3)
    sae = TopKSAE(d, F, k=k, dead_feature_threshold=4)
    cfg = TrainingConfig(batch_size=B, use_amp=use_amp, num_workers=0, learning_rate=1e-3, warmup_steps=2)
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
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("B,d,F", [(8192, 384, 3072), (2048, 768, 6144)])
@pytest.mark.parametrize("indexed", [False, True])
def test_trainer_deterministic_half_is_bit_identical(dtype, B, d, F, indexed, tmp_path):
    from whisper_sae_b200.data.feature_cache import ResidentBatches

    steps = 10
    xh = O.synthetic_activations(B * 2, d, seed=B).cuda().to(dtype)
    runs = {}
    for name, x in (("half", xh), ("fp32", xh.float())):
        tr = _trainer(tmp_path, name, d, F, 32, B, deterministic=True)
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
    gh, gf = th._graphs[B], tf._graphs[B]
    assert gh.det and gh.graph is not None and gh.x_dtype == dtype
    assert gh._x is None, "a device half batch must be read in place, not staged"
    assert gh.kernels_per_replay == gf.kernels_per_replay


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("case", ["k32", "k128", "rows128", "k64", "fp32grade"])
def test_trainer_default_mode_half_matches_fp32(dtype, case, tmp_path):
    # (rows, k, trainer options, loss tolerance after step 0, weight rel-L2 tolerance).  The default mode
    # sums gradients with float atomics in arrival order, and AdamW's early steps turn last-bit differences
    # in near-zero gradients into lr-sized weight differences - two fp32 runs of the same step differ too.
    # Measured on a B200 (1000 W) over 10 steps, two fp32 runs / bf16 against fp32, worst loss rel:
    # k = 32 2.3e-6 / 1.8e-6, k = 64 3.0e-6 / 2.6e-5, k = 128 1.4e-5 / 7.7e-5 (weights 8.4e-4 / 1.8e-3),
    # 128 rows 0 / 0, fp32-grade 0 / 7e-7.  So the first step, which starts from the same weights,
    # must agree to 1e-5 everywhere, and the later ones to a few times the measured spread.
    B, k, kw, loss_tol, tol = {"k32": (75776, 32, {}, 1e-5, 1e-3), "k128": (4096, 128, {}, 3e-4, 5e-3),
                               "rows128": (128, 32, {}, 1e-5, 1e-3), "k64": (4096, 64, {}, 1e-4, 1e-3),
                               "fp32grade": (4096, 32, {"use_amp": False}, 1e-5, 1e-3)}[case]
    steps = 10
    xh = O.synthetic_activations(B * 2, 384, seed=k).cuda().to(dtype)
    runs = {}
    for name, x in (("half", xh), ("fp32", xh.float())):
        tr = _trainer(tmp_path, name, 384, 3072, k, B, **dict(kw))
        runs[name] = (tr, [tr.train_step(x[(s % 2) * B:(s % 2 + 1) * B]) for s in range(steps)])
    (th, mh), (tf, mf) = runs["half"], runs["fp32"]
    gh = th._graphs[B]
    staged = case in ("k64", "fp32grade")
    assert (gh._x is not None) == staged and gh.x_dtype == (torch.float32 if staged else dtype)
    if case == "rows128":
        assert gh.row_step
    assert mh[0].loss == pytest.approx(mf[0].loss, rel=1e-5) and mh[0].l0 == mf[0].l0
    for a, b in zip(mh, mf):
        assert a.loss == pytest.approx(b.loss, rel=loss_tol)
    assert torch.equal(th.model.feature_last_activated, tf.model.feature_last_activated)
    for (n, p), (_, q) in zip(th.model.named_parameters(), tf.model.named_parameters()):
        assert _rel(p, q) < tol, (n, _rel(p, q))


@pytest.mark.gpu
def test_trainer_two_ranks_bf16_match_fp32(tmp_path):
    from whisper_sae_b200.sae import parallel

    k, B, steps = 128, 4096, 10
    xh = O.synthetic_activations(B * steps, 384, seed=17).cuda().to(torch.bfloat16)
    results = {}
    for name, x in (("bf16", xh), ("fp32", xh.float())):
        comms = parallel.ThreadCommunicator.make(2)
        ranks = [_trainer(tmp_path, f"{name}{r}", 384, 3072, k, B, data_parallel=True, dp_comm=c)
                 for r, c in enumerate(comms)]
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
        results[name] = (ranks, got)
    (rh, gh), (rf, gf) = results["bf16"], results["fp32"]
    assert gh[0][0].loss == pytest.approx(gf[0][0].loss, rel=1e-5)
    assert rh[0]._graphs[B // 2].x_dtype == torch.bfloat16 and rh[0]._graphs[B // 2]._x is None
    for r in range(2):
        assert torch.equal(rh[r].model.feature_last_activated, rf[r].model.feature_last_activated)
        for (n, p), (_, q) in zip(rh[r].model.named_parameters(), rf[r].model.named_parameters()):
            assert _rel(p, q) < 1e-3, (r, n, _rel(p, q))


@pytest.mark.gpu
def test_host_bf16_batches_equal_device_bf16(tmp_path):
    """train_epoch copies pinned host batches to the device in their own dtype; a host batch handed to
    train_step directly is staged into a bf16 buffer.  Both train like the device batches, bit for bit."""
    B, steps = 4096, 6
    xh = O.synthetic_activations(B * steps, 384, seed=29).to(torch.bfloat16)
    host = [[xh[s * B:(s + 1) * B].pin_memory()] for s in range(steps)]
    dev = [[b[0].cuda()] for b in host]
    runs = {}
    for name in ("epoch_host", "epoch_dev", "step_host"):
        tr = _trainer(tmp_path, name, 384, 3072, 32, B, deterministic=True)
        if name == "step_host":
            ms = [tr.train_step(b[0]) for b in host]
        else:
            ms = tr.train_epoch(host if name == "epoch_host" else dev)
        runs[name] = (tr, ms, _state(tr))
    _, md, sd = runs["epoch_dev"]
    for name in ("epoch_host", "step_host"):
        tr, ms, st = runs[name]
        assert [m.loss for m in ms] == [m.loss for m in md], name
        for n in sd:
            assert torch.equal(st[n], sd[n]), (name, n)
        assert tr._graphs[B]._x is None
    assert runs["step_host"][0]._graphs[B]._xh[torch.bfloat16].dtype == torch.bfloat16   # 2 bytes per element


@pytest.mark.gpu
def test_alternating_dtypes_capture_one_graph_each(tmp_path):
    B = 4096
    x = O.synthetic_activations(B, 384, seed=31).cuda()
    tr = _trainer(tmp_path, "alt", 384, 3072, 32, B)
    for s in range(10):
        tr.train_step(x if s % 2 == 0 else x.to(torch.bfloat16))
    gs = tr._graphs[B]
    assert gs.captures == 2, gs.captures
    assert gs.x_dtype == torch.bfloat16 and torch.float32 in gs._captured


# ------------------------------------------------------------------------------------------------
# 4. extraction into half-precision caches
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_extract_and_cache_features_bf16(tmp_path):
    import json

    from tests.test_hooks import _build, _fx
    from whisper_sae_b200.config import DataConfig, WhisperConfig as WCfg
    from whisper_sae_b200.data import FeatureCache, extract_and_cache_features

    fx = _fx()
    model, x = _build(fx["recipe"])
    caches = {}
    for dtype in (torch.float32, torch.bfloat16):
        cache = FeatureCache(tmp_path / str(dtype), WCfg(), DataConfig())
        loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(x), batch_size=2)
        extract_and_cache_features(model, None, loader, cache, encoder_layers=[0, 2], decoder_layers=[1],
                                   device="cuda", dtype=dtype)
        caches[dtype] = cache
    for comp, layer in (("encoder", 0), ("encoder", 2), ("decoder", 1)):
        f32, m32 = caches[torch.float32].load(comp, layer)
        f16, m16 = caches[torch.bfloat16].load(comp, layer)
        assert f16.dtype == torch.bfloat16 and torch.equal(f16, f32.to(torch.bfloat16))
        a = json.loads(m32.to_json())
        b = json.loads(m16.to_json())
        a.pop("created_at"), b.pop("created_at")
        assert a == b and len(json.loads(m16.to_json())) == 8
