"""Transcoder / crosscoder variants of the hot path (BASELINE config 5) on the fused CUDA path,
against golden vectors produced by the live reference (oracle/make_golden_variants.py:
tests/golden/variants.pt and variants_crosscoder.pt)."""

import pytest
import torch

from tests.conftest import load_golden

pytestmark = pytest.mark.gpu


def _inputs(seed, *shape):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def _close(a, b, name, rtol=2e-5, arel=2e-6):
    scale = b.abs().max().item() + 1e-30
    torch.testing.assert_close(a.detach().cpu().float(), b, rtol=rtol, atol=arel * scale,
                               msg=lambda m: f"{name}: {m}")


def _build_transcoder(fx, precision):
    from whisper_sae_b200.sae.transcoder import SkipTranscoder, TopKTranscoder

    r = fx["recipe"]
    cls = SkipTranscoder if r["skip"] else TopKTranscoder
    m = cls(r["d_in"], r["d_out"], r["F"], k=r["k"], precision=precision)
    m.load_state_dict(fx["state"])
    return m.cuda().train()


@pytest.mark.parametrize("name", ["transcoder_64_64_128_k8", "transcoder_96_64_256_k16", "skip_64_64_128_k8"])
def test_transcoder_fp32_matches_reference(name):
    fx = load_golden("variants")[name]
    r = fx["recipe"]
    m = _build_transcoder(fx, "fp32")
    x = _inputs(r["seed"] + 10, r["B"], r["d_in"]).cuda()
    y = _inputs(r["seed"] + 11, r["B"], r["d_out"]).cuda()
    out = m(x, y)
    out.loss.backward()
    assert out.loss.item() == pytest.approx(fx["loss"], rel=1e-5)
    assert out.reconstruction_loss is out.loss and out.sparsity_loss.item() == 0.0
    assert out.l0.item() == fx["l0"]
    _close(out.predicted, fx["predicted"], "predicted", rtol=1e-4, arel=1e-5)
    _close(out.hidden, fx["hidden"], "hidden", rtol=1e-4, arel=1e-5)
    for n, p in m.named_parameters():
        _close(p.grad, fx["grads"][n], n, rtol=1e-4, arel=1e-5)
    assert torch.equal(m.feature_last_activated.cpu(), fx["feature_last_activated"])   # bit-exact
    assert int(m.step_count) == fx["step_count"]
    assert len(out) == 6 and out[2] is out.loss        # tuple-like, like the reference NamedTuple


def test_transcoder_bf16_within_tolerance():
    fx = load_golden("variants")["transcoder_96_64_256_k16"]
    r = fx["recipe"]
    m = _build_transcoder(fx, "bf16")
    out = m(_inputs(r["seed"] + 10, r["B"], r["d_in"]).cuda(), _inputs(r["seed"] + 11, r["B"], r["d_out"]).cuda())
    out.loss.backward()
    assert out.loss.item() == pytest.approx(fx["loss"], rel=2e-2)
    assert out.l0.item() == fx["l0"]
    g, ref = m.encoder.weight.grad.cpu(), fx["grads"]["encoder.weight"]
    assert (g - ref).norm() <= 5e-2 * ref.norm()


def test_skip_transcoder_init_and_identity_skip():
    """transcoder.py:300-319 zero init; tests/test_transcoder.py:272-292 identity skip => pred == input."""
    from whisper_sae_b200.sae.transcoder import SkipTranscoder, create_transcoder

    m = SkipTranscoder(64, 64, 128, k=8, precision="fp32").cuda()
    assert float(m.decoder.weight.abs().sum()) == 0 and float(m.skip.weight.abs().sum()) == 0
    m.normalize_decoder_weights()                      # zero columns stay zero (1e-12 clamp)
    assert float(m.decoder.weight.abs().sum()) == 0
    with torch.no_grad():
        m.skip.weight.copy_(torch.eye(64))
    x = torch.randn(16, 64, device="cuda")
    out = m(x, x)
    torch.testing.assert_close(out.predicted, x, rtol=1e-5, atol=1e-6)
    assert out.loss.item() < 1e-10
    assert isinstance(create_transcoder(64, 64, 128, k=8), SkipTranscoder)
    assert type(create_transcoder(64, 64, 128, k=8, use_skip=False)).__name__ == "TopKTranscoder"


def test_transcoder_resample_and_training_step():
    from whisper_sae_b200.sae.transcoder import TopKTranscoder

    torch.manual_seed(0)
    m = TopKTranscoder(64, 64, 128, k=8, dead_feature_threshold=0, precision="fp32").cuda().train()
    x, y = torch.randn(32, 64, device="cuda"), torch.randn(32, 64, device="cuda")
    opt = torch.optim.Adam(m.parameters(), lr=1e-2)
    first = None
    for _ in range(30):
        out = m(x, y)
        opt.zero_grad()
        out.loss.backward()
        opt.step()
        m.normalize_decoder_weights()
        first = first if first is not None else out.loss.item()
    assert out.loss.item() < first
    torch.testing.assert_close(m.decoder.weight.norm(dim=0), torch.ones(128, device="cuda"), atol=1e-5, rtol=0)
    n_dead = int(m.get_dead_features().sum())
    assert m.resample_dead_features(x, y, num_resample=10) == min(n_dead, 10)


def _build_crosscoder(r, precision, state=None):
    from whisper_sae_b200.sae.crosscoder import TopKCrossLayerCrosscoder

    torch.manual_seed(r["seed"])          # same torch calls as the reference constructor => same init
    li = r["layer_indices"] if r["layer_indices"] != list(range(r["L"])) else None
    m = TopKCrossLayerCrosscoder(r["d"], r["L"], r["F"], k=r["k"], layer_indices=li, precision=precision)
    if state is not None:
        for n, v in state.items():                     # constructor reproduces the reference init
            torch.testing.assert_close(m.state_dict()[n], v, rtol=0, atol=0)
    return m.cuda().train()


@pytest.mark.parametrize("name", ["crosscoder_64x4_128_k8", "crosscoder_subset_64x2_128_k8"])
def test_crosscoder_fp32_matches_reference(name):
    fx = load_golden("variants_crosscoder")[name]
    r = fx["recipe"]
    m = _build_crosscoder(r, "fp32", fx["state"])
    acts = {li: _inputs(r["seed"] + 20 + i, r["B"], r["d"]).cuda() for i, li in enumerate(r["layer_indices"])}
    out = m(acts)
    out.loss.backward()
    assert out.loss.item() == pytest.approx(fx["loss"], rel=1e-5)
    assert out.l0.item() == fx["l0"]
    _close(out.hidden, fx["hidden"], "hidden", rtol=1e-4, arel=1e-5)
    for li, v in fx["per_layer_loss"].items():
        assert out.per_layer_loss[li].item() == pytest.approx(v, rel=1e-5)
        assert out.reconstructed[li].shape == (r["B"], r["d"])
    for n, p in m.named_parameters():
        _close(p.grad, fx["grads"][n], n, rtol=1e-4, arel=1e-5)
    assert torch.equal(m.feature_last_activated.cpu(), fx["feature_last_activated"])
    m.normalize_decoder_weights()
    torch.testing.assert_close(m.get_decoder_norms(), torch.ones(r["F"], device="cuda"), atol=1e-5, rtol=0)


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("bf16", 2e-2)])
def test_crosscoder_whisper_tiny_shape(precision, tol, monkeypatch):
    """tests/test_crosscoder.py:421-436 shape (BASELINE config 5): d=384, 4 layers, 3072 features, k=32."""
    fx = load_golden("variants_crosscoder")["crosscoder_tiny_384x4_3072_k32"]
    r = fx["recipe"]
    m = _build_crosscoder(r, precision)
    acts = {li: _inputs(r["seed"] + 20 + i, r["B"], r["d"]).cuda() for i, li in enumerate(r["layer_indices"])}
    out = m(acts)
    out.loss.backward()
    assert out.loss.item() == pytest.approx(fx["loss"], rel=tol)
    assert out.l0.item() == 32.0 == fx["l0"]
    assert out.hidden.shape == (r["B"], r["F"])
    for n, p in m.named_parameters():
        g, dg = p.grad.detach().cpu(), fx["grads"][n]
        if precision == "fp32":
            assert abs(g.double().abs().sum().item() - dg["abs_sum"]) <= 5e-4 * dg["abs_sum"] + 1e-9
            torch.testing.assert_close(g.reshape(-1)[::997], dg["sample"], rtol=1e-3,
                                       atol=1e-5 * dg["sample"].abs().max().item() + 1e-12)
        else:
            # bf16 against the fp32 golden: the TopK sets differ where bf16 rounding reorders near ties, which
            # moves whole weight-gradient rows (measured on a B200: rel L2 0.112 W_enc, 0.066 W_dec, 9e-4 b_enc)
            sample = dg["sample"].double()
            rel = ((g.reshape(-1)[::997].double() - sample).norm() / sample.norm()).item()
            assert rel <= (0.15 if n in ("W_enc", "W_dec") else tol), (n, rel)
    if precision == "bf16":
        # d = 4 x 384 = 1536 runs K4 at nb_tile = 8 (two stages, a second MMA at N = 256, all 512 TMEM
        # columns): its weight gradients must be those of K3's scatter on the same step (measured on a
        # B200: rel L2 2.4e-3 W_enc, 2.5e-3 W_dec; both are bf16 products summed in different orders)
        monkeypatch.setenv("WSAE_WGRAD", "scatter")
        m2 = _build_crosscoder(r, precision)
        m2(acts).loss.backward()
        for n, p in m2.named_parameters():
            ref, got = p.grad.detach().double(), dict(m.named_parameters())[n].grad.detach().double()
            rel = ((got - ref).norm() / ref.norm()).item()
            assert rel <= 1e-2, (n, rel)


@pytest.mark.parametrize("kind", ["transcoder", "skip", "crosscoder"])
def test_graphed_variant_step_follows_the_hand_stepped_trajectory(kind):
    """GraphedVariantStep (whole step in one CUDA graph) == the reference's hand-written step
    (forward, backward, AdamW, renorm; tests/test_transcoder.py / test_crosscoder.py of the reference)
    launched eagerly: same kernels, so losses agree to accumulation-order noise, dead-feature
    counters exactly, over more steps than the eager + capture calls."""
    from whisper_sae_b200.sae import (GraphedVariantStep, SkipTranscoder, TopKCrossLayerCrosscoder,
                                      TopKTranscoder, make_optimizer)

    d, F, k, B, L, steps = 128, 1024, 16, 512, 3, 6

    def build():
        torch.manual_seed(5)
        if kind == "crosscoder":
            return TopKCrossLayerCrosscoder(d, L, F, k=k).cuda().train()
        cls = SkipTranscoder if kind == "skip" else TopKTranscoder
        return cls(d, d, F, k=k).cuda().train()

    def batch(s):
        if kind == "crosscoder":
            return ({li: _inputs(100 * s + li, B, d).cuda() for li in range(L)},)
        return (_inputs(2 * s, B, d).cuda(), _inputs(2 * s + 1, B, d).cuda())

    ref, ref_opt = build(), None
    ref_opt = make_optimizer(ref, lr=1e-3)
    ref_losses = []
    for s in range(steps):
        with torch.amp.autocast("cuda", dtype=torch.bfloat16):
            out = ref(*batch(s))
        ref_opt.zero_grad()
        out.loss.backward()
        ref_opt.step()
        ref.normalize_decoder_weights()
        ref_losses.append(out.loss.item())

    m = build()
    stepper = GraphedVariantStep(m, make_optimizer(m, lr=1e-3))
    got = [stepper(*batch(s)) for s in range(steps)]
    assert stepper._graph is not None and stepper.calls == steps
    for s, (r, g) in enumerate(zip(ref_losses, got)):
        assert g.loss.item() == pytest.approx(r, rel=2e-3), f"step {s}"
        assert 0 < g.l0.item() <= k
    assert torch.equal(m.feature_last_activated, ref.feature_last_activated)
    assert int(m.step_count) == steps
    for (n, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        rel = ((p - q).norm() / (q.norm() + 1e-12)).item()
        assert rel < 2e-2, f"{n}: rel-L2 {rel:.2e}"
    with pytest.raises(RuntimeError):
        GraphedVariantStep(m, torch.optim.AdamW(m.parameters(), lr=1e-3))
