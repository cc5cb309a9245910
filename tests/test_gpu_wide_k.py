"""TopK SAEs with k > 64: the chunked K1 route, the team-of-warps K23 (32 < k <= 256), the wiring that
routes to them, and k > 256 falling through to K3's scatter.  Each layer has its own test, so a
failure names one piece."""

import threading

import pytest
import torch

from oracle import topk_sae_oracle as O


def _ops():
    from whisper_sae_b200 import ops
    return ops


# ------------------------------------------------------------------------------------------------
# 1. routing (no device needed)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,d,F,k,bf16,k1,k23,graph", [
    (75776, 384, 3072, 32, True, "fused", True, True),
    (75776, 384, 3072, 64, True, "fused", False, True),     # 33..64 keeps K2 + K3 by default
    (75776, 384, 3072, 65, True, "chunked", True, True),
    (75776, 768, 6144, 256, True, "chunked", True, True),
    (75776, 384, 3072, 257, True, "chunked", False, False),
    (75776, 384, 3072, 512, True, "chunked", False, False),
    (512, 384, 3072, 128, True, "dense", True, True),         # small batch: the dense form, any k
    (4096, 392, 3072, 128, True, "chunked", False, True),     # d % 128 != 0: K2 + K3
    (4096, 384, 3072, 128, False, "chunked", False, True),    # fp32 decoder: K2 + K3
    (2176, 1280, 65536, 128, True, "chunked", True, True),    # F beyond one select's shared memory: slices
    (4096, 1280, 81920, 128, True, "chunked", True, True),
    (512, 1280, 81920, 128, True, "chunked", True, True),     # small batch, but too wide for "dense"
    (4096, 384, 3002, 100, True, "chunked", True, True),      # F % 4 != 0: the scratch has a row pitch
    (2176, 1280, 65536, 64, True, "fused", False, True),       # k <= 64 keeps the fused route
])
def test_routing(B, d, F, k, bf16, k1, k23, graph, monkeypatch):
    monkeypatch.delenv("WSAE_WIDE_K23", raising=False)
    monkeypatch.delenv("WSAE_FUSED_DECODE", raising=False)
    from whisper_sae_b200.sae import TopKSAE
    from whisper_sae_b200.sae.training import SAETrainer

    ops = _ops()
    assert ops.encode_route(B, F, k) == k1
    if k > ops.ENCODE_FUSED_MAX_K:      # the fused epilogue cannot run k > 64, with or without an F-split
        assert ops.encode_route(B, F, k, nsplit=4) == "chunked"
        for Bx, Fx in [(1, 3072), (1024, 49153), (1025, 3002), (75776, 393216), (100, 131072)]:
            assert ops.encode_route(Bx, Fx, k) != "fused"
    assert ops.decode_backward_supported(d, k, bf16) == k23
    if k > 256:      # the bf16 backward then scatters through K3 instead of bucketing for K4
        assert ops.bucket_supported(F, k) == (k < 266)
    else:
        assert ops.bucket_supported(F, k)

    class _Stub:         # _graph_ok reads these attributes only
        cuda_graph = True
        model = TopKSAE(d, 256, k=min(k, 256))
    _Stub.model.k = k
    _Stub.model.hidden_dim = F
    assert SAETrainer._graph_ok(_Stub(), torch.zeros(2, d)) == graph


def test_routing_wide_k23_switch(monkeypatch):
    ops = _ops()
    monkeypatch.setenv("WSAE_WIDE_K23", "1")
    assert ops.decode_backward_supported(384, 33, True) and ops.decode_backward_supported(384, 64, True)
    assert ops.decode_backward_supported(384, 32, True)            # the k <= 32 kernels are unchanged
    assert not ops.decode_backward_supported(392, 64, True)


def test_chunk_rows():
    ops = _ops()
    for B, F, k in [(75776, 3072, 128), (75776, 6144, 256), (2176, 40960, 65), (5000, 49152, 128),
                    (100, 3072, 65), (4096, 81920, 128), (4096, 3002, 100), (75776, 393216, 256)]:
        r = ops.encode_chunk_rows(B, F, k)
        assert r % 128 == 0 and r >= 128 and r <= (B + 127) // 128 * 128
        assert r == 128 or ops.encode_chunk_scratch_floats(F, k, r) * 4 <= 40 << 20
    assert ops.encode_chunk_scratch_floats(49152, 256, 128) == 128 * 49152             # one slice: no lists
    assert ops.encode_chunk_scratch_floats(3002, 65, 128) == 128 * 3004                 # row pitch
    assert ops.encode_chunk_scratch_floats(81920, 128, 256) == 256 * (81920 + 2 * 2 * 128)


# ------------------------------------------------------------------------------------------------
# 2. K1, chunked
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("B,d,F", [(5000, 384, 3072), (2176, 1280, 40960)])
@pytest.mark.parametrize("k", [65, 128, 256])
def test_k1_chunked_matches_unchunked_dense(B, d, F, k):
    """Bit for bit what one unchunked wsae_encode_topk_dense call returns on the same packed operands;
    in fp32-grade mode the selected sets are torch.topk's except at documented near-ties."""
    from whisper_sae_b200 import _lib
    ops = _ops()
    assert ops.encode_route(B, F, k) == "chunked"
    assert (B + ops.encode_chunk_rows(B, F, k) - 1) // ops.encode_chunk_rows(B, F, k) >= 2
    torch.manual_seed(B + k)
    state = O.init_state(d, F)
    state["b_pre"] = torch.randn(d) * 0.05
    x = O.synthetic_activations(B, d, seed=B + d).cuda()
    st = {n: t.cuda() for n, t in state.items() if t.is_floating_point()}
    lib = _lib.load()
    for terms in (1, 6):
        a = ops.pack_activations(x, st["b_pre"], terms)
        w = ops.pack_encoder(st["encoder.weight"], st["encoder.bias"], terms)
        ps = ops.packed_shape(d, terms)
        idx, val = ops.encode_topk(a, w, B, F, d, terms, k)
        pre = torch.empty(B, F, device="cuda")
        ref_v = torch.empty(B, k, device="cuda")
        ref_i = torch.empty(B, k, dtype=torch.int32, device="cuda")
        _lib.check(lib.wsae_encode_topk_dense(a.data_ptr(), w.data_ptr(), B, a.shape[0], F, w.shape[0], ps.kp,
                                              ps.used_cols, k, pre.data_ptr(), ref_v.data_ptr(), ref_i.data_ptr(),
                                              ops._stream()), "wsae_encode_topk_dense")
        torch.cuda.synchronize()
        assert torch.equal(idx, ref_i) and torch.equal(val, ref_v), f"terms={terms}"
        if terms == 6:      # the fp32 statement, evaluated in float64 so that its own rounding drops out
            want = ((x - st["b_pre"]).double() @ st["encoder.weight"].double().t() + st["encoder.bias"].double())
            scale = want.abs().max().item()
            got = torch.sort(idx.long(), -1).values
            ref = torch.sort(torch.topk(want, k, dim=-1).indices, -1).values
            bad = (got != ref).any(-1).cpu()
            ties = O.near_tie_rows(want.float().cpu(), k, 1e-5 * scale)
            assert not (bad & ~ties).any(), int((bad & ~ties).sum())
            # values: fp32 accumulation of 6 * d split-bf16 products (1.2e-5 of the row scale at d = 1280)
            torch.testing.assert_close(val.double(), want.gather(-1, idx.long()), rtol=1e-5, atol=3e-5 * scale)
        del pre


# ------------------------------------------------------------------------------------------------
# 3. K23, team-of-warps form, against the oracle
# ------------------------------------------------------------------------------------------------
_K23_F = {384: 3072, 512: 4096, 768: 6144, 1024: 8192, 1280: 4096}


@pytest.mark.gpu
@pytest.mark.parametrize("d", [384, 512, 768, 1024, 1280])
@pytest.mark.parametrize("k", [33, 64, 65, 128, 256])
def test_k23_wide_matches_oracle(k, d):
    """The test_decode_backward_fused recipe (tests/test_gpu_sparse.py) at 32 < k <= 256 on a ragged
    batch, directly and through the _rows_at slot form with a permutation."""
    ops = _ops()
    B, F = 301, _K23_F[d]
    torch.manual_seed(k + d)
    state = O.init_state(d, F)
    state["b_pre"] = torch.randn(d) * 0.05
    state["decoder.bias"] = torch.randn(d) * 0.02
    state["decoder.weight"] = state["decoder.weight"].to(torch.bfloat16).float()
    st = {n: t.cuda() for n, t in state.items() if t.is_floating_point()}
    x = O.synthetic_activations(B, d, seed=3 * B + d).cuda()
    pre = (x - st["b_pre"]) @ st["encoder.weight"].t() + st["encoder.bias"]
    val, idx = torch.topk(pre, k, dim=-1)
    val[::3, 0] = -val[::3, 0].abs()                    # relu-masked entries contribute nothing
    val[1::7, k - 1] = -val[1::7, k - 1].abs()          # ... also in the last warp's tail
    w_decT = st["decoder.weight"].t().contiguous()      # [F, d], exactly bf16-representable
    rows = w_decT[idx]                                  # [B, k, d]
    h_bf = torch.relu(val).to(torch.bfloat16).float()
    recon = (h_bf.unsqueeze(-1) * rows).sum(1) + st["decoder.bias"] + st["b_pre"]
    resid_ref = recon - x
    grad_out, coef = 0.5, 2.0 / (B * d)
    g = resid_ref * (coef * grad_out)
    dv_ref = (g.unsqueeze(1) * rows).sum(-1) * (val > 0)
    dbe_ref = torch.zeros(F, device="cuda").index_add_(0, idx.reshape(-1), dv_ref.reshape(-1))
    w_used = w_decT.to(torch.bfloat16)
    idx32 = idx.to(torch.int32).contiguous()
    val = val.contiguous()

    perm = torch.randperm(B, device="cuda")
    x_src = torch.empty_like(x)
    x_src[perm] = x                                     # batch row r is row perm[r] of x_src
    slot = torch.tensor([x_src.data_ptr()], dtype=torch.int64, device="cuda")
    rows_slot = torch.tensor([perm.data_ptr()], dtype=torch.int64, device="cuda")

    def run(form):
        out = dict(stats=torch.zeros(3, dtype=torch.int64, device="cuda"),
                   last=torch.zeros(F, dtype=torch.int64, device="cuda"),
                   resid=torch.empty(B, d, device="cuda"),
                   resid_bf=torch.empty(B, d, dtype=torch.bfloat16, device="cuda"),
                   dbe=torch.zeros(F, device="cuda"), dbd=torch.zeros(d, device="cuda"),
                   dpre=torch.empty(B, k, device="cuda"))
        kw = dict(resid=out["resid"], resid_bf16=out["resid_bf"], stats=out["stats"], last_activated=out["last"],
                  step_count=torch.tensor(41, dtype=torch.int64, device="cuda"), d_b_enc=out["dbe"],
                  d_b_dec=out["dbd"], dpre_val=out["dpre"])
        tgt = x if form == "direct" else slot
        ops.decode_backward(tgt, w_used, st["decoder.bias"], st["b_pre"], idx32, val,
                            torch.tensor(grad_out, device="cuda"), coef, target_is_slot=form != "direct",
                            rows_at=rows_slot if form == "rows_at" else None, **kw)
        torch.cuda.synchronize()
        return out

    def close(a, b, name, rtol=2e-5, arel=2e-6):
        scale = b.abs().max().item() + 1e-30
        torch.testing.assert_close(a, b, rtol=rtol, atol=arel * scale, msg=lambda m: f"{name}: {m}")

    for form in ("direct", "rows_at"):
        o = run(form)
        torch.testing.assert_close(o["resid"], resid_ref, rtol=1e-5, atol=2e-6)
        assert torch.equal(o["resid_bf"], o["resid"].to(torch.bfloat16))
        raw = o["stats"].cpu()
        assert raw[:1].view(torch.float64).item() == pytest.approx((resid_ref.double() ** 2).sum().item(), rel=1e-6)
        assert raw[1].item() == int((val > 0).sum())
        want_last = torch.zeros(F, dtype=torch.int64, device="cuda")
        want_last[idx[val > 0]] = 42
        assert torch.equal(o["last"], want_last)
        close(o["dpre"], dv_ref, "dpre", rtol=2e-2, arel=4e-3)
        close(o["dbe"], dbe_ref, "db_enc", rtol=2e-2, arel=4e-3)
        close(o["dbd"], g.sum(0), "db_dec")
        g_bf = o["resid_bf"].float() * (coef * grad_out)
        dv_bf = (g_bf.unsqueeze(1) * rows).sum(-1) * (val > 0)
        close(o["dpre"], dv_bf, "dpre vs bf16-residual reference", rtol=1e-4, arel=1e-5)


# ------------------------------------------------------------------------------------------------
# 4. module step (autograd node) and 6. k > 256
# ------------------------------------------------------------------------------------------------
def _dense_reference(sae, x, k):
    """bf16-mode loss, fired set and dense fp32 gradients with torch ops (test_gpu_fullsize.py)."""
    w = {n: p.detach() for n, p in sae.named_parameters()}
    B, D = x.shape
    F = w["encoder.bias"].numel()
    with torch.no_grad():
        xc = x - w["b_pre"]
        pre = xc.to(torch.bfloat16).float() @ w["encoder.weight"].to(torch.bfloat16).float().t() + w["encoder.bias"]
        v, i = torch.topk(pre, k, dim=1)
        wd = w["decoder.weight"].t().to(torch.bfloat16).float()
        hidden = torch.zeros(B, F, device="cuda").scatter_(1, i, torch.relu(v))
        resid = hidden.to(torch.bfloat16).float() @ wd + w["decoder.bias"] + w["b_pre"] - x
        g = resid * (2.0 / (B * D))
        dpre = torch.zeros(B, F, device="cuda").scatter_(1, i, (g @ wd.t()).gather(1, i) * (v > 0))
        fired = torch.zeros(F, dtype=torch.bool, device="cuda")
        fired[i[v > 0]] = True
        grads = {"encoder.weight": dpre.t() @ xc, "encoder.bias": dpre.sum(0), "decoder.bias": g.sum(0),
                 "decoder.weight": (hidden.t() @ g).t()}
        return (resid ** 2).mean().item(), fired, grads


@pytest.mark.gpu
@pytest.mark.parametrize("k", [128, 256])
def test_module_step_wide_k(k):
    from whisper_sae_b200.sae import TopKSAE

    B, D, F = 4096, 384, 3072
    torch.manual_seed(5)
    sae = TopKSAE(D, F, k=k).cuda().train()
    x = O.synthetic_activations(B, D, seed=k).cuda()
    loss_ref, fired_ref, g_ref = _dense_reference(sae, x, k)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = sae(x)
    assert out.loss.item() == pytest.approx(loss_ref, rel=1e-4)
    out.loss.backward()
    assert torch.equal(sae.feature_last_activated > 0, fired_ref)
    for n, p in sae.named_parameters():
        if n == "b_pre":
            continue
        rel = ((p.grad - g_ref[n]).norm() / g_ref[n].norm()).item()
        assert rel < 2e-2, (n, rel)


@pytest.mark.gpu
def test_train_step_k_above_256_runs(tmp_path):
    """k = 512: eager autograd, K2 + K3 scatter (the K4 bucketing's shared memory stops at ~265)."""
    from whisper_sae_b200.config import TrainingConfig
    from whisper_sae_b200.sae import SAETrainer, TopKSAE

    B, D, F, k = 4096, 384, 3072, 512
    torch.manual_seed(6)
    sae = TopKSAE(D, F, k=k)
    tr = SAETrainer(sae, TrainingConfig(batch_size=B, use_amp=True, num_workers=0), device="cuda",
                    run_dir=tmp_path)
    x = O.synthetic_activations(B, D, seed=9).cuda()
    loss_ref, _, _ = _dense_reference(sae, x, k)
    m = tr.train_step(x)
    assert not tr._graphs
    assert m.loss == pytest.approx(loss_ref, rel=2e-2)
    assert 0 < m.l0 <= k
    for p in sae.parameters():
        assert torch.isfinite(p).all()


# ------------------------------------------------------------------------------------------------
# 5. trainer: graphed == eager, two emulated ranks == one device
# ------------------------------------------------------------------------------------------------
def _trainer(tmp_path, tag, k, **kw):
    from whisper_sae_b200.config import TrainingConfig
    from whisper_sae_b200.sae import SAETrainer, TopKSAE

    torch.manual_seed(3)
    sae = TopKSAE(384, 3072, k=k, dead_feature_threshold=4)
    cfg = TrainingConfig(batch_size=4096, use_amp=True, num_workers=0, learning_rate=1e-3, warmup_steps=2)
    tr = SAETrainer(sae, cfg, device="cuda", run_dir=tmp_path / tag, **kw)
    tr.setup_scheduler(100)
    return tr


@pytest.mark.gpu
def test_trainer_graphed_matches_eager_k128(tmp_path):
    k, B, steps = 128, 4096, 10
    x = O.synthetic_activations(B * steps, 384, seed=13).cuda()
    runs = {}
    for graphed in (True, False):
        tr = _trainer(tmp_path, f"g{int(graphed)}", k, cuda_graph=graphed)
        runs[graphed] = (tr, [tr.train_step(x[s * B:(s + 1) * B]) for s in range(steps)])
    (tg, mg), (te, me) = runs[True], runs[False]
    assert tg._graphs[B].graph is not None and not te._graphs
    assert mg[0].loss == pytest.approx(me[0].loss, rel=1e-5)
    assert mg[0].l0 == me[0].l0
    # both runs sum their gradients with float atomics in arrival order, and AdamW's early steps move an
    # element by ~lr whatever the size of its gradient: last-bit differences in near-zero gradients become
    # lr-sized weight differences (1.4e-3 - 1.7e-3 rel-L2 after 10 steps, measured)
    for (n, p), (_, q) in zip(tg.model.named_parameters(), te.model.named_parameters()):
        rel = ((p - q).norm() / q.norm()).item()
        assert rel < 5e-3, (n, rel)
    assert int(tg.model.step_count) == int(te.model.step_count) == steps
    assert torch.equal(tg.model.feature_last_activated, te.model.feature_last_activated)


@pytest.mark.gpu
def test_trainer_two_ranks_match_one_device_k128(tmp_path):
    from whisper_sae_b200.sae import parallel

    k, B, steps = 128, 4096, 10
    x = O.synthetic_activations(B * steps, 384, seed=17).cuda()
    single = _trainer(tmp_path, "single", k)
    ref = [single.train_step(x[s * B:(s + 1) * B]) for s in range(steps)]
    comms = parallel.ThreadCommunicator.make(2)
    ranks = [_trainer(tmp_path, f"rank{r}", k, data_parallel=True, dp_comm=c) for r, c in enumerate(comms)]
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
    assert got[0][0].loss == pytest.approx(ref[0].loss, rel=1e-5)
    for s in range(steps):
        assert got[0][s].l0 == got[1][s].l0
    ts = [threading.Thread(target=ranks[r].consolidate_weights) for r in range(2)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    for r in range(2):
        m = ranks[r].model
        assert int(m.step_count) == steps
        assert torch.equal(m.feature_last_activated, single.model.feature_last_activated)
        for (n, p), (_, q) in zip(m.named_parameters(), single.model.named_parameters()):
            rel = ((p - q).norm() / q.norm()).item()
            assert rel < 1e-3, (r, n, rel)


# ------------------------------------------------------------------------------------------------
# 7. consumers of the sparse encoder
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_consumers_k128():
    from oracle.feature_topk_oracle import TrackerOracle
    from whisper_sae_b200.analysis.feature_viz import collect_top_activations
    from whisper_sae_b200.sae import TopKSAE

    B, D, F, k = 2048, 384, 3072, 128
    torch.manual_seed(7)
    sae = TopKSAE(D, F, k=k, dead_feature_threshold=3).cuda()
    x = O.synthetic_activations(B, D, seed=23).cuda()

    # collect_top_activations: the tracker holds what the CPU tracker oracle holds for the same code
    tracker = collect_top_activations(sae, [x[:1024], x[1024:]], num_features=F, k=5)
    idx, val = sae._sparse_encode(x)
    hidden = torch.zeros(B, F, device="cuda").scatter_(1, idx.long(), torch.relu(val)).cpu()
    oracle = TrackerOracle(F, 5)
    oracle.update(hidden[:1024].numpy(), list(range(1024)))
    oracle.update(hidden[1024:].numpy(), list(range(1024, B)))
    assert tracker.total_activations == oracle.total_activations
    for f in range(0, F, 97):
        want = sorted(oracle.heaps[f], key=lambda e: (-e[0], -e[1]))
        got = tracker.get_top_examples(f)
        assert [e.sample_idx for e in got] == [e[2] for e in want], f
        assert [e.activation_value for e in got] == pytest.approx([e[0] for e in want], rel=1e-6), f

    # resample_dead_features (eval mode: the forward inside stamps nothing): the i-th dead feature gets
    # the i-th highest-error row, L2-normalised, as encoder row and decoder column, bias 0
    sae.eval()
    with torch.no_grad():
        sae.step_count.fill_(10)
        sae.feature_last_activated.zero_()
        sae.feature_last_activated[: F // 2] = 10
        w_enc0 = sae.encoder.weight.detach().clone()
        sae(x)
        errors = (sae._last_sparse.resid.float() ** 2).sum(-1)
    n = sae.resample_dead_features(x, num_resample=50)
    assert n == 50
    dead = torch.arange(F // 2, F // 2 + 50, device="cuda")
    assert torch.equal(sae.encoder.weight[: F // 2], w_enc0[: F // 2])
    top = torch.topk(errors, 50).indices
    torch.testing.assert_close(sae.encoder.weight[dead], torch.nn.functional.normalize(x[top], dim=-1))
    torch.testing.assert_close(sae.decoder.weight[:, dead].t(), sae.encoder.weight[dead])
    assert (sae.encoder.bias[dead] == 0).all()
    assert (sae.feature_last_activated[dead] == 10).all()
