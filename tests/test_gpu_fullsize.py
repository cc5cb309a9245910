"""Full-size (BASELINE.json configs[1] bench shape: 75776 x 384 -> 3072, k = 32) checks through
size-independent properties, with torch-on-GPU as the checker where the CPU oracle would take
minutes: TopK optimality, exact sparsity, value = recomputed pre-activation, decode/loss identity,
unit-norm decoder, counter invariants."""

import pytest
import torch

from oracle import topk_sae_oracle as O

pytestmark = pytest.mark.gpu

B, D, F, K = 75776, 384, 3072, 32


def _state():
    torch.manual_seed(42)
    return O.init_state(D, F)


def test_fullsize_topk_is_optimal_and_exact():
    from whisper_sae_b200 import ops

    st = _state()
    x = O.synthetic_activations(B, D, seed=1234).cuda()
    w, b = st["encoder.weight"].cuda(), st["encoder.bias"].cuda()
    a = ops.pack_activations(x, None, 1)
    wp = ops.pack_encoder(w, b, 1)
    idx, val = ops.encode_topk(a, wp, B, F, D, 1, K)
    torch.cuda.synchronize()
    assert idx.shape == (B, K) and int(idx.min()) >= 0 and int(idx.max()) < F
    srt = torch.sort(idx, dim=1).values
    assert bool((srt[:, 1:] != srt[:, :-1]).all())                      # k distinct features per row
    # checker: the same bf16-rounded operands, fp32 accumulate (torch matmul), exact fp32 bias
    xq, wq = x.to(torch.bfloat16).float(), w.to(torch.bfloat16).float()
    worst_gap, worst_val = 0.0, 0.0
    for r0 in range(0, B, 8192):
        pre = xq[r0:r0 + 8192] @ wq.t() + b
        scale = pre.abs().max().item()
        got = pre.gather(1, idx[r0:r0 + 8192].long())
        worst_val = max(worst_val, ((got - val[r0:r0 + 8192]).abs().max() / scale).item())
        kth = torch.topk(pre, K + 1, dim=1).values
        # every selected value >= the true (k+1)-th largest (up to accumulation-order noise) ...
        worst_gap = max(worst_gap, ((kth[:, K:K + 1] - val[r0:r0 + 8192]).max() / scale).item())
        # ... and the selected sum equals the optimal top-k sum
        assert torch.allclose(val[r0:r0 + 8192].sum(1), kth[:, :K].sum(1), rtol=1e-5, atol=1e-4 * scale)
    assert worst_val <= 2e-6, worst_val            # values = recomputed pre-activations
    assert worst_gap <= 2e-6, worst_gap            # nothing outside the set beats anything inside


def test_fullsize_train_step_invariants(tmp_path):
    from whisper_sae_b200.config import TrainingConfig
    from whisper_sae_b200.sae import SAETrainer, TopKSAE

    torch.manual_seed(42)
    sae = TopKSAE(D, F, k=K, dead_feature_threshold=10_000)
    cfg = TrainingConfig(batch_size=B, use_amp=True, num_workers=0)
    tr = SAETrainer(sae, cfg, device="cuda", run_dir=tmp_path)
    tr.setup_scheduler(1000)
    x = O.synthetic_activations(2 * B, D, seed=7).cuda()
    w0 = {n: p.detach().clone() for n, p in sae.named_parameters()}

    def torch_forward(w, xb):
        """bf16-mode forward with torch ops on the given weights: loss, l0, fired set."""
        with torch.no_grad():
            pre = (xb - w["b_pre"]).to(torch.bfloat16).float() @ w["encoder.weight"].to(torch.bfloat16).float().t() \
                + w["encoder.bias"]
            v, i = torch.topk(pre, K, dim=1)
            wd = w["decoder.weight"].t().to(torch.bfloat16).float()       # [F, d] bf16 shadow
            recon = torch.zeros(B, D, device="cuda")
            for j in range(K):
                recon += torch.relu(v[:, j:j + 1]).to(torch.bfloat16).float() * wd[i[:, j]]
            recon += w["decoder.bias"] + w["b_pre"]
            fired = torch.zeros(F, dtype=torch.bool, device="cuda")
            fired[i[v > 0]] = True
            return ((recon - xb) ** 2).mean().item(), float((v > 0).sum()) / B, fired

    def torch_grads(w, xb):
        """Dense fp32 statement of the step's gradients (same bf16 operand roundings in the forward)."""
        with torch.no_grad():
            xc = xb - w["b_pre"]
            pre = xc.to(torch.bfloat16).float() @ w["encoder.weight"].to(torch.bfloat16).float().t() + w["encoder.bias"]
            v, i = torch.topk(pre, K, dim=1)
            del pre
            wd = w["decoder.weight"].t().to(torch.bfloat16).float()
            hidden = torch.zeros(B, F, device="cuda").scatter_(1, i, torch.relu(v))
            g = (hidden.to(torch.bfloat16).float() @ wd + w["decoder.bias"] + w["b_pre"] - xb) * (2.0 / (B * D))
            dpre = torch.zeros(B, F, device="cuda").scatter_(1, i, (g @ wd.t()).gather(1, i) * (v > 0))
            return {"encoder.weight": dpre.t() @ xc, "encoder.bias": dpre.sum(0), "decoder.bias": g.sum(0),
                    "decoder.weight": (hidden.t() @ g).t()}

    g_ref = torch_grads(w0, x[:B])
    loss_ref, l0_ref, fired_ref = torch_forward(w0, x[:B])
    m1 = tr.train_step(x[:B])
    # the FIRST AdamW step moves every element by ~lr * sign(gradient): where the reference gradient is not
    # tiny, the weights must have moved against it - a wrong row, a dropped or misplaced gradient tile at the
    # benchmark's own shape shows up here (the digests above cannot see it)
    for n in ("encoder.weight", "encoder.bias", "decoder.bias"):
        delta = sae.state_dict()[n].detach() - w0[n]
        gr = g_ref[n]
        big = gr.abs() > 1e-2 * gr.abs().max()
        agree = (torch.sign(delta[big]) == -torch.sign(gr[big])).double().mean().item()
        assert big.sum() > 0.01 * gr.numel() and agree > 0.999, (n, agree, int(big.sum()))
    # and the gradient the step left in .grad is the reference gradient (bf16 operands in K4: 2e-2)
    for n in ("encoder.weight", "decoder.weight", "encoder.bias", "decoder.bias"):
        got = dict(sae.named_parameters())[n].grad
        rel = ((got - g_ref[n]).norm() / g_ref[n].norm()).item()
        assert rel < 2e-2, (n, rel)
    del g_ref
    assert m1.loss == pytest.approx(loss_ref, rel=1e-4)
    assert m1.l0 == pytest.approx(l0_ref, abs=1e-3)
    assert int(sae.step_count) == 1
    assert torch.equal(sae.feature_last_activated > 0, fired_ref)         # fired set bit-exact
    assert m1.dead_feature_ratio == 0.0
    w1 = {n: p.detach().clone() for n, p in sae.named_parameters()}
    loss2_ref, l02_ref, fired2_ref = torch_forward(w1, x[B:])
    m2 = tr.train_step(x[B:])                                             # CUDA-graph capture / replay path
    assert m2.loss == pytest.approx(loss2_ref, rel=1e-4) and int(sae.step_count) == 2
    assert m2.l0 == pytest.approx(l02_ref, abs=1e-3)
    assert torch.equal(sae.feature_last_activated == 2, fired2_ref)
    norms = sae.decoder.weight.norm(dim=0)
    torch.testing.assert_close(norms, torch.ones(F, device="cuda"), atol=1e-5, rtol=0)
    for n, p in sae.named_parameters():
        assert torch.isfinite(p).all() and not torch.equal(p, w0[n]), n


@pytest.mark.parametrize("shape", [(75776, 384, 3072), (8192, 768, 6144), (2048, 1280, 40960), (16384, 512, 4096),
                                   (8192, 1024, 8192)])
def test_deterministic_mode_is_bit_reproducible(shape, tmp_path):
    """SAETrainer(deterministic=True): two runs of the bf16 graphed step from the same state on the
    same batches are BIT-identical (losses, every parameter, AdamW moments, counters) - split-K
    partials and cross-row sums are added in a fixed / order-independent way (wsae_*_det) instead of
    float atomics in arrival order.  The default mode must agree with it to accumulation-order noise."""
    from whisper_sae_b200.config import TrainingConfig
    from whisper_sae_b200.sae import SAETrainer, TopKSAE

    rows, d, f = shape
    steps = 5
    x = O.synthetic_activations(2 * rows, d, seed=21).cuda()

    def run(deterministic: bool, tag: str):
        torch.manual_seed(42)
        sae = TopKSAE(d, f, k=K, dead_feature_threshold=10_000)
        cfg = TrainingConfig(batch_size=rows, use_amp=True, num_workers=0, learning_rate=1e-3, warmup_steps=2)
        tr = SAETrainer(sae, cfg, device="cuda", run_dir=tmp_path / tag, deterministic=deterministic)
        tr.setup_scheduler(100)
        losses = [tr.train_step(x[(s % 2) * rows:(s % 2 + 1) * rows]).loss for s in range(steps)]
        torch.cuda.synchronize()
        state = {n: t.detach().clone() for n, t in sae.state_dict().items()}
        for i, p in enumerate(sae.parameters()):
            st = tr.optimizer.state[p]
            state[f"m{i}"], state[f"v{i}"] = st["exp_avg"].clone(), st["exp_avg_sq"].clone()
        assert tr._graphs[rows].graph is not None and tr._graphs[rows].det == deterministic
        return losses, state

    la, sa = run(True, "a")
    lb, sb = run(True, "b")
    assert la == lb, "deterministic mode: losses differ between two runs"
    for n in sa:
        assert torch.equal(sa[n], sb[n]), f"deterministic mode: {n} differs between two runs"
    lc, sc = run(False, "c")
    for a, c in zip(la, lc):
        assert a == pytest.approx(c, rel=1e-5)
    assert torch.equal(sa["feature_last_activated"], sc["feature_last_activated"])
    for n in ("encoder.weight", "decoder.weight"):
        rel = ((sa[n] - sc[n]).norm() / sc[n].norm()).item()
        assert rel < 1e-3, f"{n}: deterministic vs default rel-L2 {rel:.2e}"


@pytest.mark.parametrize("rows,d,f,k", [
    pytest.param(75776, 768, 6144, K, id="75776-768-6144"),
    pytest.param(37888, 1280, 40960, K, id="37888-1280-40960"),
    pytest.param(16384, 512, 4096, 32, id="base-16384-512-4096-k32"),
    pytest.param(16384, 512, 4096, 128, id="base-16384-512-4096-k128"),
    pytest.param(16384, 1024, 8192, 64, id="medium-16384-1024-8192-k64"),      # K2 + K3 + K4
    pytest.param(4096, 1280, 81920, 128, id="large-4096-1280-81920-k128"),     # chunked K1 in column slices
    pytest.param(2048, 1024, 65536, 256, id="medium-2048-1024-65536-k256"),
])
def test_fullsize_step_gradients_small_and_large_v3(rows, d, f, k, tmp_path):
    """BASELINE configs 3 / 4 at the bench's own batch sizes, and the Whisper base / medium widths and
    more than 65 536 features at k up to 256: loss, L0, fired set and the five gradient tensors of ONE
    graphed bf16 step against a dense fp32 statement with the same bf16 operand roundings in the forward
    (the golden traces at these widths are 256-row batches)."""
    from whisper_sae_b200.config import TrainingConfig
    from whisper_sae_b200.sae import SAETrainer, TopKSAE

    torch.manual_seed(42)
    sae = TopKSAE(d, f, k=k, dead_feature_threshold=10_000)
    tr = SAETrainer(sae, TrainingConfig(batch_size=rows, use_amp=True, num_workers=0), device="cuda", run_dir=tmp_path)
    tr.setup_scheduler(1000)
    x = O.synthetic_activations(rows, d, seed=17).cuda()
    w = {n: p.detach().clone() for n, p in sae.named_parameters()}
    with torch.no_grad():
        xc = x - w["b_pre"]
        pre = xc.to(torch.bfloat16).float() @ w["encoder.weight"].to(torch.bfloat16).float().t() + w["encoder.bias"]
        v, i = torch.topk(pre, k, dim=1)
        del pre
        wd = w["decoder.weight"].t().to(torch.bfloat16).float()
        hidden = torch.zeros(rows, f, device="cuda").scatter_(1, i, torch.relu(v))
        resid = hidden.to(torch.bfloat16).float() @ wd + w["decoder.bias"] + w["b_pre"] - x
        loss_ref = (resid ** 2).mean().item()
        g = resid * (2.0 / (rows * d))
        dpre = torch.zeros(rows, f, device="cuda").scatter_(1, i, (g @ wd.t()).gather(1, i) * (v > 0))
        ref = {"encoder.weight": dpre.t() @ xc, "encoder.bias": dpre.sum(0), "decoder.bias": g.sum(0),
               "decoder.weight": (hidden.t() @ g).t()}
        ref["b_pre"] = ref["decoder.bias"] - ref["encoder.bias"] @ w["encoder.weight"]
        fired = torch.zeros(f, dtype=torch.bool, device="cuda")
        fired[i[v > 0]] = True
        l0_ref = float((v > 0).sum()) / rows
        del hidden, dpre, resid, g
    m = tr.train_step(x)
    assert rows in tr._graphs          # the step ran the graphed route's kernels (the first call is not captured)
    assert m.loss == pytest.approx(loss_ref, rel=1e-4)
    assert m.l0 == pytest.approx(l0_ref, abs=1e-3)
    assert torch.equal(sae.feature_last_activated > 0, fired)
    for n, p in sae.named_parameters():
        rel = ((p.grad - ref[n]).norm() / ref[n].norm().clamp_min(1e-30)).item()
        # db_pre = db_dec - db_enc . W_enc is a difference of nearly cancelling sums: looser
        assert rel < (1e-1 if n == "b_pre" else 2e-2), (n, rel)
