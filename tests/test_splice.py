"""Splicing TopK SAEs into Whisper's forward pass (sae/splice.py, csrc/wsae_splice.cu).

The statement the kernels are held to (include/wsae.h): for a layer output row h with mean mu, biased
variance var and r = rsqrt(var + eps),
    x      = (h - mu) * r * gamma + beta
    (i, v) = TopK_k(pack(x - b_pre) . W'^T)                       (K1, unchanged)
    a_j    = relu(v_j), rounded to bf16; W_dec rows from the bf16 shadow
    recon  = sum_j a_j W_dec[i_j] + b_dec + b_pre
    recon' = sum_j gain[i_j] a_j W_dec[i_j] + b_dec + b_pre + steer
    replace: h' = mu + ((recon' - beta) / gamma) / r          error: h' = h + ((recon' - recon) / gamma) / r
``splice_oracle`` below is that statement in float64.

CPU: the validation errors the splice raises before any launch, and the oracle's two fixed points.
GPU:
* ``wsae_splice_pack`` is bit-identical to ``pack_activations(layernorm_rows(h), b_pre, 1)``, and K1 on it
  selects what ``TopKSAE._sparse_encode`` selects on the extracted activations.
* ``wsae_splice_decode`` against the oracle run on the same (idx, val), bf16 decoder rows, bf16-rounded
  activations and (mu, r), per element within
      bound = 2 * [ (k + 4) * u * (S + |beta|) / |gamma * r| + 4 * u * (|t| + |mu| + |h|) ] + u_T * |h'|
  where u = 2^-24, u_T the unit roundoff of h's dtype (2^-24, 2^-8, 2^-11), S = |b_dec| + |b_pre| + |steer|
  + sum_j (1 + |gain_j|) a_j |W_dec[i_j]| (the magnitudes the two fp32 accumulations add), and t the
  inverse-LayerNorm term ((recon' - beta) / gamma / r or (recon' - recon) / gamma / r).
  Measured on a B200 (1000 W): worst |err| / bound 0.98-0.997 per (k, F); the u_T * |h'| term, which
  round-to-nearest into bf16 / fp16 reaches, sets it.
* Exact: error mode without an intervention returns h bit for bit (-0.0 included); l0 and the feature
  counts equal torch.bincount of idx[val > 0]; mse equals TopKSAE.forward's reconstruction_loss (bf16 mode)
  on the extracted activations up to summation order; the SAEs' state_dict is unchanged.
* End to end on a seeded random-init whisper-tiny-shaped model (fp32 and fp16) with non-trivial final
  LayerNorm affine parameters, splices on encoder layers 0 and 2 and decoder layer 1.
"""

from __future__ import annotations

import numpy as np
import pytest
import torch

U32 = 2.0 ** -24
U_DTYPE = {torch.float32: 2.0 ** -24, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}


# ---------------------------------------------------------------- float64 statement
def splice_oracle(h, idx, val, w_dec, b_dec, b_pre, mode, gamma=None, beta=None, eps=1e-5, gain=None,
                  steer=None, mu=None, r=None):
    """h' in float64 (torch tensors on any device).  ``w_dec`` [F, d] (feature-major), ``idx`` / ``val``
    [N, k] with (-inf, -1) padding.  gamma None: no LayerNorm (x = h, identity inverse).  mu / r: given
    (per row), or computed from h."""
    f64 = lambda t: None if t is None else torch.as_tensor(t).to(torch.float64)   # noqa: E731
    h = f64(h)
    ln = gamma is not None
    if ln:
        if mu is None:
            mu = h.mean(1)
            r = 1.0 / torch.sqrt(((h - mu[:, None]) ** 2).mean(1) + eps)
        mu, r, gamma, beta = f64(mu)[:, None], f64(r)[:, None], f64(gamma), f64(beta)
    idx = torch.as_tensor(idx).long()
    val = f64(val)
    fired = (idx >= 0) & (val > 0)
    a = torch.where(fired, val, torch.zeros_like(val))
    safe = torch.where(fired, idx, torch.zeros_like(idx))
    g = torch.ones_like(a) if gain is None else f64(gain)[safe]
    W = f64(w_dec)[safe]                                           # [N, k, d]
    bias = f64(b_dec) + (0.0 if b_pre is None else f64(b_pre))
    recon = torch.bmm(a[:, None, :], W)[:, 0] + bias
    delta = torch.bmm(((g - 1.0) * a)[:, None, :], W)[:, 0] + (0.0 if steer is None else f64(steer))
    if mode == "replace":
        rp = recon + delta
        return mu + ((rp - beta) / gamma) / r if ln else rp
    return h + (delta / gamma) / r if ln else h + delta


def test_oracle_replace_with_an_exact_reconstruction_returns_h():
    g = torch.Generator().manual_seed(0)
    N, d, k = 6, 16, 3
    h = torch.randn(N, d, generator=g, dtype=torch.float64) * 2 + 0.3
    gamma = 1 + 0.2 * torch.randn(d, generator=g, dtype=torch.float64)
    beta = 0.1 * torch.randn(d, generator=g, dtype=torch.float64)
    mu = h.mean(1)
    r = 1 / torch.sqrt(((h - mu[:, None]) ** 2).mean(1) + 1e-5)
    x = (h - mu[:, None]) * r[:, None] * gamma + beta
    b_dec = torch.randn(d, generator=g, dtype=torch.float64)
    b_pre = torch.randn(d, generator=g, dtype=torch.float64)
    w_dec = torch.randn(N + 2, d, generator=g, dtype=torch.float64)
    w_dec[:N] = x - b_dec - b_pre                     # feature n reconstructs row n exactly
    idx = torch.full((N, k), -1)
    val = torch.full((N, k), float("-inf"), dtype=torch.float64)
    idx[:, 0], val[:, 0] = torch.arange(N), 1.0
    idx[:, 1], val[:, 1] = N, -0.5                    # negative pre-activation: relu drops it
    out = splice_oracle(h, idx, val, w_dec, b_dec, b_pre, "replace", gamma, beta)
    torch.testing.assert_close(out, h, rtol=1e-12, atol=1e-12)


def test_oracle_error_without_intervention_returns_h():
    g = torch.Generator().manual_seed(1)
    N, d, F, k = 5, 24, 40, 4
    h = torch.randn(N, d, generator=g, dtype=torch.float64)
    idx = torch.stack([torch.randperm(F, generator=g)[:k] for _ in range(N)])
    val = torch.randn(N, k, generator=g, dtype=torch.float64)
    w_dec = torch.randn(F, d, generator=g, dtype=torch.float64)
    gamma = 1 + 0.1 * torch.randn(d, generator=g, dtype=torch.float64)
    beta = torch.randn(d, generator=g, dtype=torch.float64)
    args = (h, idx, val, w_dec, torch.randn(d, generator=g), torch.randn(d, generator=g), "error")
    assert torch.equal(splice_oracle(*args, gamma, beta), h)
    assert torch.equal(splice_oracle(*args, gamma, beta, gain=torch.ones(F)), h)
    assert torch.equal(splice_oracle(*args), h)                        # without the LayerNorm


# ---------------------------------------------------------------- CPU: validation
def _tiny_model(d_model=64, device="cpu", seed=3):
    from transformers import WhisperConfig, WhisperForConditionalGeneration
    cfg = WhisperConfig(d_model=d_model, encoder_layers=3, decoder_layers=2, encoder_attention_heads=2,
                        decoder_attention_heads=2, encoder_ffn_dim=128, decoder_ffn_dim=128, num_mel_bins=80,
                        max_source_positions=40, max_target_positions=16, vocab_size=200, decoder_start_token_id=1,
                        pad_token_id=0, bos_token_id=1, eos_token_id=2)
    torch.manual_seed(seed)
    return WhisperForConditionalGeneration(cfg).eval().to(device)


def test_validation_errors_raise_before_any_launch():
    from whisper_sae_b200.sae import (ReLUSAE, TopKCrossLayerCrosscoder, TopKSAE, TopKTranscoder,
                                      WhisperSAESplice)
    model = _tiny_model()
    sae = TopKSAE(64, 256, k=8)
    with pytest.raises(ValueError, match="mode"):
        WhisperSAESplice(model, {("encoder", 0): sae}, mode="ablate")
    for bad in [("encoderx", 0), ("encoder", 3), ("decoder", -1), ("encoder", "0"), "encoder.0", ("encoder",)]:
        with pytest.raises(ValueError, match="site"):
            WhisperSAESplice(model, {bad: sae})
    with pytest.raises(TypeError, match="out of scope"):
        WhisperSAESplice(model, {("encoder", 0): TopKTranscoder(64, 64, 256, k=8)})
    with pytest.raises(TypeError, match="out of scope"):
        WhisperSAESplice(model, {("encoder", 0): TopKCrossLayerCrosscoder(64, 2, 256, k=8)})
    with pytest.raises(TypeError, match="TopKSAE"):
        WhisperSAESplice(model, {("encoder", 0): ReLUSAE(64, 256)})
    with pytest.raises(ValueError, match="input_dim"):
        WhisperSAESplice(model, {("decoder", 1): TopKSAE(128, 256, k=8)})
    odd = _tiny_model(d_model=60)
    with pytest.raises(ValueError, match="% 8"):
        WhisperSAESplice(odd, {("encoder", 0): TopKSAE(60, 256, k=8)})
    with torch.no_grad():
        model.model.decoder.layer_norm.weight[5] = 0.0
    with pytest.raises(ValueError, match="zero weight"):
        WhisperSAESplice(model, {("decoder", 0): sae})
    WhisperSAESplice(model, {("encoder", 0): sae})                              # the encoder's is fine
    WhisperSAESplice(model, {("decoder", 0): sae}, apply_layer_norm=False)      # no inverse needed

    splice = WhisperSAESplice(model, {("encoder", 1): sae}, mode="error")
    with pytest.raises(ValueError, match="gain"):
        splice.set_intervention(("encoder", 1), gain=torch.ones(256, dtype=torch.float64))
    with pytest.raises(ValueError, match="gain"):
        splice.set_intervention(("encoder", 1), gain=torch.ones(255))
    with pytest.raises(ValueError, match="steer"):
        splice.set_intervention(("encoder", 1), steer=torch.zeros(64, 1))
    with pytest.raises(KeyError):
        splice.set_intervention(("encoder", 2), gain=torch.ones(256))
    splice.set_intervention(("encoder", 1), gain=torch.ones(256), steer=torch.zeros(64))
    splice.clear_interventions()
    with pytest.raises(RuntimeError, match="dtype"):
        splice._splice(splice._sites[("encoder", 1)], torch.zeros(2, 64, dtype=torch.float64))
    with pytest.raises(RuntimeError, match="CUDA"):                 # CPU model: refused before any launch
        with splice:
            pass
    assert not splice.active


# ---------------------------------------------------------------- GPU: wsae_splice_pack
def _ln_params(d, seed):
    g = torch.Generator().manual_seed(seed)
    gamma = (1 + 0.2 * torch.randn(d, generator=g)).cuda()
    beta = (0.3 * torch.randn(d, generator=g)).cuda()
    b_pre = (0.2 * torch.randn(d, generator=g)).cuda()
    return gamma, beta, b_pre


@pytest.mark.gpu
@pytest.mark.parametrize("d", [384, 512, 768, 1024, 1280])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_splice_pack_is_the_extraction_pack_bit_for_bit(d, dtype):
    from whisper_sae_b200 import ops
    from whisper_sae_b200.sae import TopKSAE
    gamma, beta, b_pre = _ln_params(d, d)
    eps = 1e-5
    for N in (1, 127, 1500, 12000):
        g = torch.Generator(device="cuda").manual_seed(N + d)
        h = (torch.randn(N, d, device="cuda", generator=g) * 3 + 0.5).to(dtype)
        h[0, :5] = 0.0
        a, rs = ops.splice_pack(h, gamma, beta, eps, b_pre)
        x = torch.empty(N, d, device="cuda")
        ops.layernorm_rows_(h, gamma, beta, eps, x)
        ref = ops.pack_activations(x, b_pre, 1)
        assert a.shape == ref.shape and torch.equal(a.view(torch.int16), ref.view(torch.int16)), (N, d, dtype)
        h64 = h.double()
        mu64 = h64.mean(1)
        r64 = 1 / torch.sqrt(((h64 - mu64[:, None]) ** 2).mean(1) + eps)
        # a fp32 sum of d terms: relative to the row's mean magnitude
        assert ((rs[:, 0].double() - mu64).abs() <= 1e-6 * h64.abs().mean(1)).all()
        assert ((rs[:, 1].double() - r64).abs() <= 1e-6 * r64).all()
        if N == 1500:
            torch.manual_seed(d)
            sae = TopKSAE(d, 8 * d, k=32, precision="bf16").cuda()
            with torch.no_grad():
                sae.b_pre.copy_(b_pre)
            w = ops.pack_encoder(sae.encoder.weight.detach().contiguous(), sae.encoder.bias.detach(), 1)
            idx, val = ops.encode_topk(a, w, N, 8 * d, d, 1, 32)
            ridx, rval = sae._sparse_encode(x)
            assert torch.equal(idx, ridx) and torch.equal(val.view(torch.int32), rval.view(torch.int32))


# ---------------------------------------------------------------- GPU: wsae_splice_decode vs float64
def _decode_case(N, d, F, k, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    idx = torch.rand(N, F, device="cuda", generator=g).argsort(dim=1)[:, :k].to(torch.int32).contiguous()
    val = torch.randn(N, k, device="cuda", generator=g) + 0.3
    half = k // 2
    idx[0, half:], val[0, half:] = -1, float("-inf")          # a row K1 padded
    val[1, :] = -1.0                                           # a row with nothing positive
    w = (0.1 * torch.randn(F, d, device="cuda", generator=g))
    w_bf = w.to(torch.bfloat16).contiguous()
    b_dec = 0.1 * torch.randn(d, device="cuda", generator=g)
    return idx.contiguous(), val.contiguous(), w_bf, b_dec


@pytest.mark.gpu
@pytest.mark.parametrize("k,F", [(1, 3072), (32, 3072), (64, 3072), (128, 3072), (256, 3072),
                                 (1, 40960), (32, 40960), (64, 40960), (128, 40960), (256, 40960)])
def test_splice_decode_matches_float64(k, F):
    from whisper_sae_b200 import ops
    d = 384 if F == 3072 else 1280
    N = 200
    idx, val, w_bf, b_dec = _decode_case(N, d, F, k, seed=k * 7 + F)
    gamma, beta, b_pre = _ln_params(d, k)
    eps = 1e-5
    # the intervention features: ones the rows selected
    feats = torch.unique(idx[2:40, 0].long())[:16]
    gains = {"none": None}
    gains["ablate16"] = torch.ones(F, device="cuda")
    gains["ablate16"][feats] = 0.0
    gains["amp3"] = torch.ones(F, device="cuda")
    gains["amp3"][feats] = 3.0
    steer = 0.7 * w_bf[feats[0]].float()                       # clamp feature feats[0] to 0.7 with gain 0
    fired = (idx >= 0) & (val > 0)
    a_bf = torch.where(fired, val, 0).to(torch.bfloat16).double()
    safe = torch.where(fired, idx, 0).long()
    W64 = w_bf.double()
    absW = W64[safe].abs()                                     # [N, k, d]
    worst = 0.0
    for dtype in (torch.float32, torch.bfloat16, torch.float16):
        gh = torch.Generator(device="cuda").manual_seed(k + F)
        h = (torch.randn(N, d, device="cuda", generator=gh) * 2 + 0.4).to(dtype)
        _, rs = ops.splice_pack(h, gamma, beta, eps, b_pre)
        mu, r = rs[:, 0].double(), rs[:, 1].double()
        h64 = h.double()
        for mode in ("replace", "error"):
            for gname, gain in gains.items():
                for st in (None, steer):
                    if st is not None:
                        gain = (gains["ablate16"] if gain is None else gain).clone()
                        gain[feats[0]] = 0.0
                    out = ops.splice_decode(h, rs, gamma, beta, w_bf, b_dec, b_pre, idx, val, mode=mode,
                                            gain=gain, steer=st)
                    want = splice_oracle(h64, idx, a_bf, W64, b_dec, b_pre, mode, gamma, beta, gain=gain, steer=st,
                                         mu=mu, r=r)
                    g_sel = torch.ones_like(a_bf) if gain is None else gain.double()[safe]
                    S = (b_dec.double().abs() + b_pre.double().abs() + (0 if st is None else st.double().abs())
                         + torch.bmm(((1 + g_sel.abs()) * a_bf)[:, None, :], absW)[:, 0])
                    gr = (gamma.double()[None, :] * r[:, None]).abs()
                    t = want - (mu[:, None] if mode == "replace" else h64)
                    bound = 2 * ((k + 4) * U32 * (S + beta.double().abs()) / gr
                                 + 4 * U32 * (t.abs() + mu.abs()[:, None] + h64.abs())) + U_DTYPE[dtype] * want.abs()
                    ratio = float(((out.double() - want).abs() / bound).max())
                    assert ratio <= 1.0, (dtype, mode, gname, st is not None, ratio)
                    worst = max(worst, ratio)
                    if mode == "error" and gain is None and st is None:
                        assert torch.equal(out, h)
    print(f"splice_decode k={k} F={F}: worst |err| / bound = {worst:.3g}")


# ---------------------------------------------------------------- GPU: exact checks
@pytest.mark.gpu
def test_splice_exact_identities_and_statistics():
    from whisper_sae_b200 import ops
    from whisper_sae_b200.sae import TopKSAE
    d, F, k, N = 384, 3072, 32, 1500
    gamma, beta, b_pre = _ln_params(d, 5)
    torch.manual_seed(7)
    sae = TopKSAE(d, F, k=k, precision="bf16").cuda().eval()
    with torch.no_grad():
        sae.b_pre.copy_(b_pre)
        sae.decoder.bias.normal_(0, 0.05)
    g = torch.Generator(device="cuda").manual_seed(9)
    h = torch.randn(N, d, device="cuda", generator=g) * 2 + 0.4
    h[3, :7] = -0.0
    h[4, :7] = 0.0
    a, rs = ops.splice_pack(h, gamma, beta, 1e-5, sae.b_pre.detach())
    w = ops.pack_encoder(sae.encoder.weight.detach().contiguous(), sae.encoder.bias.detach(), 1)
    idx, val = ops.encode_topk(a, w, N, F, d, 1, k)
    w_bf = ops.cast_bf16(sae.decoder.weight.detach().t().contiguous())
    stats = torch.zeros(3, dtype=torch.int64, device="cuda")
    x_sum = torch.zeros(d, dtype=torch.float64, device="cuda")
    fc = torch.zeros(F, dtype=torch.int64, device="cuda")
    for dtype in (torch.float32, torch.bfloat16, torch.float16):
        hd = h.to(dtype)
        out = ops.splice_decode(hd, rs, gamma, beta, w_bf, sae.decoder.bias.detach(), sae.b_pre.detach(), idx, val,
                                mode="error", stats=stats if dtype == torch.float32 else None)
        assert torch.equal(out.view(torch.int8), hd.view(torch.int8)), dtype       # -0.0 included
        out = ops.splice_decode(hd, None, None, None, w_bf, sae.decoder.bias.detach(), sae.b_pre.detach(), idx, val,
                                mode="error")
        assert torch.equal(out.view(torch.int8), hd.view(torch.int8)), dtype
    stats.zero_()
    ops.splice_decode(h, rs, gamma, beta, w_bf, sae.decoder.bias.detach(), sae.b_pre.detach(), idx, val,
                      mode="replace", stats=stats, x_sum=x_sum, feature_count=fc)
    want_fc = torch.bincount(idx[val > 0].long(), minlength=F)
    assert torch.equal(fc, want_fc)
    assert int(stats[2]) == int((val > 0).sum())
    x = torch.empty(N, d, device="cuda")
    ops.layernorm_rows_(h, gamma, beta, 1e-5, x)
    with torch.no_grad():
        ref = sae(x)
    sse = float(stats[:1].view(torch.float64))
    assert abs(sse / (N * d) - float(ref.reconstruction_loss)) <= 1e-5 * float(ref.reconstruction_loss)
    torch.testing.assert_close(x_sum, x.double().sum(0), rtol=1e-6, atol=1e-6 * N)
    sumsq = float(stats[1:2].view(torch.float64))
    assert abs(sumsq - float((x.double() ** 2).sum())) <= 1e-6 * sumsq


# ---------------------------------------------------------------- GPU: end to end
def _whisper_tiny(dtype):
    from transformers import WhisperConfig, WhisperForConditionalGeneration
    cfg = WhisperConfig(d_model=384, encoder_layers=4, decoder_layers=4, encoder_attention_heads=6,
                        decoder_attention_heads=6, encoder_ffn_dim=1536, decoder_ffn_dim=1536, num_mel_bins=80,
                        max_source_positions=1500, max_target_positions=448, vocab_size=1000,
                        decoder_start_token_id=1, pad_token_id=0, bos_token_id=1, eos_token_id=2)
    torch.manual_seed(21)
    model = WhisperForConditionalGeneration(cfg).eval()
    with torch.no_grad():
        g = torch.Generator().manual_seed(22)
        for ln in (model.model.encoder.layer_norm, model.model.decoder.layer_norm):
            ln.weight.copy_(1.0 + 0.1 * torch.randn(ln.weight.shape, generator=g))
            ln.bias.copy_(0.1 * torch.randn(ln.bias.shape, generator=g))
    x = torch.randn(2, 80, 3000, generator=torch.Generator().manual_seed(23))
    return model.to("cuda", dtype), x.to("cuda", dtype)


def _reference_splice(h, ln, sae):
    """The statement as a plain PyTorch computation (replace mode, no intervention): extraction's LayerNorm,
    the SAE's own K1 selection, then the decode and the inverse LayerNorm in torch fp32."""
    from whisper_sae_b200 import ops
    d = h.shape[-1]
    h2 = h.reshape(-1, d).float()
    x = torch.empty_like(h2)
    ops.layernorm_rows_(h2, ln.weight.float(), ln.bias.float(), ln.eps, x)
    idx, val = sae._sparse_encode(x)
    fired = (idx >= 0) & (val > 0)
    a = torch.where(fired, val, 0).to(torch.bfloat16).float()
    W = sae.decoder.weight.detach().t().to(torch.bfloat16).float()[torch.where(fired, idx, 0).long()]
    recon = (a[:, :, None] * W).sum(1) + sae.decoder.bias.detach() + sae.b_pre.detach()
    mu = h2.mean(1, keepdim=True)
    r = torch.rsqrt(((h2 - mu) ** 2).mean(1, keepdim=True) + ln.eps)
    return (mu + ((recon - ln.bias.float()) / ln.weight.float()) / r).reshape(h.shape)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_splice_end_to_end_on_whisper_tiny(dtype):
    from whisper_sae_b200.sae import TopKSAE, WhisperSAESplice, evaluate_splice
    from whisper_sae_b200.sae.hooks import _hidden_of
    model, feats = _whisper_tiny(dtype)
    sites = [("encoder", 0), ("encoder", 2), ("decoder", 1)]
    saes = {}
    for i, s in enumerate(sites):
        torch.manual_seed(100 + i)
        saes[s] = TopKSAE(384, 3072, k=32, precision="bf16").cuda()
        with torch.no_grad():
            saes[s].b_pre.normal_(0, 0.1)
            saes[s].decoder.bias.normal_(0, 0.05)
    before = {s: {n: t.clone() for n, t in sae.state_dict().items()} for s, sae in saes.items()}
    ids = torch.tensor([[1, 5, 9, 13, 17, 21, 25, 29], [1, 7, 3, 11, 2, 0, 0, 0]], device="cuda")
    labels = torch.cat([ids[:, 1:], torch.full((2, 1), 2, device="cuda")], dim=1)
    labels[1, 5:] = -100

    with torch.no_grad():
        clean = model(input_features=feats, decoder_input_ids=ids).logits
        clean_gen = model.generate(feats, max_new_tokens=6, do_sample=False)
        splice = WhisperSAESplice(model, saes, mode="error")
        with splice:
            spliced = model(input_features=feats, decoder_input_ids=ids).logits
            gen = model.generate(feats, max_new_tokens=6, do_sample=False)
        assert torch.equal(spliced, clean) and torch.equal(gen, clean_gen)
        st = splice.stats(("encoder", 0))
        assert st.rows >= 2 * 1500 and st.feature_counts.shape == (3072,) and 0 < st.l0 <= 32
        assert splice.stats(("decoder", 1)).rows > 2 * 8      # teacher-forced rows + B x 1 generate steps
        assert torch.equal(model(input_features=feats, decoder_input_ids=ids).logits, clean)   # after __exit__

        # replace mode: every site's output against the plain PyTorch statement on the same input
        seen = {}

        def recorder(site, slot):
            def hook(m, i, o):
                seen.setdefault(site, {})[slot] = _hidden_of(o).detach().clone()
            return hook
        layers = {s: getattr(model.model, s[0]).layers[s[1]] for s in sites}
        pre = [layers[s].register_forward_hook(recorder(s, "h")) for s in sites]
        splice_r = WhisperSAESplice(model, saes, mode="replace")
        with splice_r:
            post = [layers[s].register_forward_hook(recorder(s, "out")) for s in sites]
            model(input_features=feats, decoder_input_ids=ids)
            for p in post:
                p.remove()
        for p in pre:
            p.remove()
        tol = 1e-4 if dtype == torch.float32 else 4e-3
        for s in sites:
            h, out = seen[s]["h"], seen[s]["out"]
            assert out.dtype == dtype and out.shape == h.shape
            ref = _reference_splice(h, getattr(model.model, s[0]).layer_norm, saes[s])
            torch.testing.assert_close(out.float(), ref, rtol=tol, atol=tol * float(ref.abs().max()))

        ev = evaluate_splice(model, feats, labels, splice)
        assert ev.ce_spliced == ev.ce_clean and ev.kl == 0.0 and not splice.active
        ev = evaluate_splice(model, feats, labels, splice_r)
        with splice_r:
            out = model(input_features=feats, labels=labels)
        assert ev.ce_spliced == float(out.loss)
        ce = torch.nn.functional.cross_entropy(out.logits.float().reshape(-1, out.logits.shape[-1]), labels.reshape(-1),
                                               ignore_index=-100)
        assert abs(float(ce) - ev.ce_spliced) <= 1e-3 * abs(ev.ce_spliced)
        assert ev.kl > 0 and np.isfinite(ev.ce_zero)
        assert ev.loss_recovered == pytest.approx((ev.ce_zero - ev.ce_spliced) / (ev.ce_zero - ev.ce_clean))

        if dtype == torch.float32:    # without the LayerNorm, and an ablation that changes the stream
            with WhisperSAESplice(model, saes, mode="error", apply_layer_norm=False):
                assert torch.equal(model(input_features=feats, decoder_input_ids=ids).logits, clean)
            gain = torch.ones(3072, device="cuda")
            gain[:1536] = 0.0
            with splice:
                splice.set_intervention(("encoder", 0), gain=gain)
                ablated = model(input_features=feats, decoder_input_ids=ids).logits
                splice.clear_interventions()
                assert torch.equal(model(input_features=feats, decoder_input_ids=ids).logits, clean)
            assert not torch.equal(ablated, clean)

    for s, sae in saes.items():
        for n, t in sae.state_dict().items():
            assert torch.equal(t, before[s][n]), (s, n)
