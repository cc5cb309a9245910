"""Pin the CPU oracle against golden vectors produced by the live reference
(oracle/make_golden.py).  CPU-only; runs in the build container and on the GPU box."""

import pytest
import torch

from oracle import topk_sae_oracle as O
from tests.conftest import load_golden

# the last two are BASELINE configs 3 / 4 (whisper-small 768->6144, large-v3 1280->40960)
CASES = ["small_64x256", "tiny_test_384x3072", "mid_128x1024_k32", "small_768x6144", "large_1280x40960"]


def _check_digest(t: torch.Tensor, dg: dict, rtol: float, atol: float = 1e-7):
    assert tuple(t.shape) == tuple(dg["shape"])
    td = t.double().reshape(-1)
    scale = max(dg["abs_sum"], 1e-30)
    assert abs(td.sum().item() - dg["sum"]) <= rtol * scale + atol
    assert abs(td.abs().sum().item() - dg["abs_sum"]) <= rtol * scale + atol
    sample = t.reshape(-1)[:: dg["sample_stride"]]
    torch.testing.assert_close(sample, dg["sample"], rtol=rtol * 50, atol=rtol * dg["abs_sum"] / td.numel())


def _run_oracle(fx):
    r = fx["recipe"]
    torch.manual_seed(r["model_seed"])
    state = O.init_state(r["d"], r["F"])
    opt = O.AdamWState()
    x_all = O.synthetic_activations(r["B"] * r["steps"], r["d"], r["data_seed"])
    lrs = O.lr_sequence(r["lr"], r["total_steps"], r["warmup"])
    results = []
    for s in range(r["steps"]):
        xb = x_all[s * r["B"]:(s + 1) * r["B"]]
        results.append(O.train_step(state, opt, xb, r["k"], lrs[s], gradient_clip=r["gradient_clip"],
                                    weight_decay=r["weight_decay"], dead_threshold=r["dead_threshold"]))
    return state, results, lrs


@pytest.mark.parametrize("name", CASES)
def test_init_matches_reference_rng(name):
    fx = load_golden(name)
    r = fx["recipe"]
    torch.manual_seed(r["model_seed"])
    state = O.init_state(r["d"], r["F"])
    for n, dg in fx["init_digest"].items():
        _check_digest(state[n], dg, rtol=1e-7)


@pytest.mark.parametrize("name", CASES)
def test_train_steps_match_reference(name):
    fx = load_golden(name)
    state, results, lrs = _run_oracle(fx)
    for s, (res, ref) in enumerate(zip(results, fx["per_step"])):
        assert res.loss == pytest.approx(ref["loss"], rel=2e-6), f"step {s}"
        assert res.l0 == pytest.approx(ref["l0"], rel=1e-6)
        assert res.dead_feature_ratio == pytest.approx(ref["dead_feature_ratio"], abs=1e-7)
        assert lrs[s] == pytest.approx(ref["lr_used"], rel=1e-9)
    # integer state is bit-exact
    assert torch.equal(state["feature_last_activated"], fx["final_counters"]["feature_last_activated"])
    assert int(state["step_count"]) == int(fx["final_counters"]["step_count"])
    for n in O.PARAM_ORDER:
        ref = fx["final_params"][n]
        if isinstance(ref, dict):
            _check_digest(state[n], ref, rtol=2e-6)
        else:
            torch.testing.assert_close(state[n], ref, rtol=2e-5, atol=2e-7)


@pytest.mark.parametrize("name", CASES)
def test_first_step_topk_and_grads(name):
    fx = load_golden(name)
    r = fx["recipe"]
    torch.manual_seed(r["model_seed"])
    state = O.init_state(r["d"], r["F"])
    xb = O.synthetic_activations(r["B"] * r["steps"], r["d"], r["data_seed"])[: r["B"]]
    fwd = O.forward(state, xb, r["k"], training=True)
    first = fx["first_step"]
    assert torch.equal(torch.sort(fwd.idx, -1).values.to(torch.int32), first["topk_idx_sorted"])
    assert fwd.loss.item() == pytest.approx(first["loss"], rel=2e-6)
    assert fwd.l0.item() == pytest.approx(first["l0"], rel=1e-6)
    grads = O.backward(state, xb, fwd)
    for n in O.PARAM_ORDER:
        ref = first["grads"][n]
        if isinstance(ref, dict):
            _check_digest(grads[n], ref, rtol=1e-5)
        else:
            torch.testing.assert_close(grads[n], ref, rtol=1e-4, atol=1e-9)


def test_dead_feature_counters_fixed_row():
    """The reference's exactly-4-alive scenario (tests/test_sae_model.py:251-294)."""
    fx = load_golden("dead_fixed_row")
    r = fx["recipe"]
    torch.manual_seed(r["model_seed"])
    state = O.init_state(r["d"], r["F"])
    x = torch.randn(1, r["d"], generator=torch.Generator().manual_seed(r["x_seed"]))
    for _ in range(r["steps"]):
        O.forward(state, x, r["k"], training=True)
    assert int(state["step_count"]) == fx["step_count"]
    assert torch.equal(state["feature_last_activated"], fx["feature_last_activated"])
    dead = O.dead_features(state, r["thr"])
    assert torch.equal(dead, fx["dead_mask"])
    assert int((~dead).sum()) == fx["num_alive"] == 4


RESAMPLE_CASES = ["resample_64x256", "resample_64x256_eval", "resample_384x3072", "resample_1280x40960"]


def resample_pre_state(r: dict) -> dict:
    """The state oracle/make_golden.py's resample cases start from (seeds only)."""
    torch.manual_seed(r["model_seed"])
    state = O.init_state(r["d"], r["F"])
    g = torch.Generator().manual_seed(r["counter_seed"])
    state["feature_last_activated"] = torch.randint(0, r["step_count"], (r["F"],), generator=g)
    state["step_count"] = torch.tensor(r["step_count"], dtype=torch.long)
    return state


@pytest.mark.parametrize("name", RESAMPLE_CASES)
def test_resample_dead_features_matches_reference(name):
    """model.py:197-257 on the live reference (fixture) vs the oracle restatement."""
    fx = load_golden(name)
    r = fx["recipe"]
    state = resample_pre_state(r)
    assert torch.equal(torch.where(O.dead_features(state, r["thr"]))[0], fx["dead_before"])
    x = O.synthetic_activations(r["rows"], r["d"], r["data_seed"])
    ret = O.resample_dead_features(state, x, r["k"], r["thr"], r["num_resample"], training=r["train_mode"])
    assert ret == fx["returned"]
    assert int(state["step_count"]) == fx["step_count"] == r["step_count"] + int(r["train_mode"])
    assert torch.equal(state["feature_last_activated"], fx["feature_last_activated"])   # bit-exact
    tgt = fx["written"]
    torch.testing.assert_close(state["encoder.weight"][tgt], fx["encoder_rows"], rtol=0, atol=0)
    torch.testing.assert_close(state["decoder.weight"][:, tgt].t(), fx["decoder_cols_T"], rtol=0, atol=0)
    assert (state["encoder.bias"][tgt] == 0).all()
    for n in O.PARAM_ORDER:
        _check_digest(state[n], fx["after_digest"][n], rtol=1e-7)


def test_dense_hidden_has_exactly_k_nonzeros():
    torch.manual_seed(0)
    state = O.init_state(64, 256)
    x = torch.randn(100, 64)
    fwd = O.forward(state, x, 8, training=False)
    hidden = O.dense_hidden(fwd, 256)
    assert ((hidden != 0).sum(-1) <= 8).all()
    assert (hidden >= 0).all()
    assert int(state["step_count"]) == 0  # eval mode leaves counters alone (model.py:174)


def test_backward_matches_reference_autograd_formula():
    """Oracle backward itself vs torch autograd on the reference's forward graph (sanity of the
    hand-derived gradient)."""
    torch.manual_seed(3)
    state = O.init_state(32, 64)
    state['b_pre'] = torch.randn(32) * 0.05
    x = O.synthetic_activations(20, 32, seed=103)
    fwd = O.forward(state, x, 4, training=False)
    p = {n: state[n].clone().requires_grad_(True) for n in O.PARAM_ORDER}
    xr = x.clone().requires_grad_(True)
    pre = (xr - p["b_pre"]) @ p["encoder.weight"].t() + p["encoder.bias"]
    v, i = torch.topk(pre, 4, dim=-1)
    hidden = torch.zeros_like(pre).scatter(-1, i, torch.relu(v))
    recon = hidden @ p["decoder.weight"].t() + p["decoder.bias"] + p["b_pre"]
    torch.nn.functional.mse_loss(recon, xr).backward()
    g = O.backward(state, x, fwd)
    for n in O.PARAM_ORDER:
        torch.testing.assert_close(g[n], p[n].grad, rtol=1e-4, atol=1e-8)
    torch.testing.assert_close(g["dx"], xr.grad, rtol=1e-4, atol=1e-8)




# ---- transcoder / crosscoder variants (oracle/variants_oracle.py vs live-reference fixtures) ----
VARIANT_CASES = ["transcoder_64_64_128_k8", "transcoder_96_64_256_k16", "skip_64_64_128_k8",
                 "crosscoder_64x4_128_k8", "crosscoder_subset_64x2_128_k8"]


def _variant_inputs(seed, *shape):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("name", VARIANT_CASES)
def test_variants_oracle_matches_reference(name):
    from oracle import variants_oracle as V

    fx = load_golden("variants_crosscoder" if name.startswith("crosscoder") else "variants")[name]
    r = fx["recipe"]
    if name.startswith("crosscoder"):
        acts = {li: _variant_inputs(r["seed"] + 20 + i, r["B"], r["d"]) for i, li in enumerate(r["layer_indices"])}
        out = V.crosscoder(fx["state"], acts, r["layer_indices"], r["k"])
        for li, v in fx["per_layer_loss"].items():
            assert out["per_layer_loss"][li] == pytest.approx(v, rel=1e-6)
    else:
        x = _variant_inputs(r["seed"] + 10, r["B"], r["d_in"])
        y = _variant_inputs(r["seed"] + 11, r["B"], r["d_out"])
        out = V.transcoder(fx["state"], x, y, r["k"])
        torch.testing.assert_close(out["predicted"], fx["predicted"], rtol=1e-5, atol=1e-6)
    assert out["loss"] == pytest.approx(fx["loss"], rel=1e-6)
    assert out["l0"] == fx["l0"]
    torch.testing.assert_close(out["hidden"], fx["hidden"], rtol=1e-5, atol=1e-6)
    for n, g in fx["grads"].items():
        torch.testing.assert_close(out["grads"][n], g, rtol=1e-5, atol=1e-7, msg=lambda m: f"{n}: {m}")
    want = torch.zeros_like(fx["feature_last_activated"])
    want[out["fired"]] = 1
    assert torch.equal(want, fx["feature_last_activated"]) and fx["step_count"] == 1
