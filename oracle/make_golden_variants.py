"""Golden vectors for the transcoder / crosscoder variants from the LIVE reference (build container
only; same rules as make_golden.py).  Writes tests/golden/variants.pt (transcoders) and
tests/golden/variants_crosscoder.pt (crosscoders), two files so that each stays under 1 MB.

    PYTHONDONTWRITEBYTECODE=1 python oracle/make_golden_variants.py
"""

from __future__ import annotations

import sys
from pathlib import Path

import torch

REF_SRC = Path("/root/reference/src")
ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(REF_SRC))
sys.dont_write_bytecode = True

from whisper_sae.sae.crosscoder import TopKCrossLayerCrosscoder  # noqa: E402  (reference)
from whisper_sae.sae.transcoder import SkipTranscoder, TopKTranscoder  # noqa: E402  (reference)

GOLDEN = ROOT / "tests" / "golden"


def _inputs(seed: int, *shape: int) -> torch.Tensor:
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def transcoder_case(name: str, skip: bool, d_in: int, d_out: int, F: int, k: int, B: int, seed: int) -> dict:
    torch.manual_seed(seed)
    cls = SkipTranscoder if skip else TopKTranscoder
    m = cls(d_in, d_out, F, k=k)
    if skip:   # the zero-initialised decoder/skip would make every gradient trivial: perturb them
        g = torch.Generator().manual_seed(seed + 1)
        with torch.no_grad():
            m.decoder.weight.copy_(torch.randn(d_out, F, generator=g) * 0.05)
            m.decoder.bias.copy_(torch.randn(d_out, generator=g) * 0.02)
            m.skip.weight.copy_(torch.randn(d_out, d_in, generator=g) * 0.05)
            m.skip.bias.copy_(torch.randn(d_out, generator=g) * 0.02)
    state = {n: v.clone() for n, v in m.state_dict().items()}
    x, y = _inputs(seed + 10, B, d_in), _inputs(seed + 11, B, d_out)
    m.train()
    out = m(x, y)
    out.loss.backward()
    return {"recipe": dict(name=name, skip=skip, d_in=d_in, d_out=d_out, F=F, k=k, B=B, seed=seed),
            "state": state, "loss": out.loss.item(), "l0": out.l0.item(),
            "hidden": out.hidden.detach().clone(), "predicted": out.predicted.detach().clone(),
            "grads": {n: p.grad.clone() for n, p in m.named_parameters()},
            "feature_last_activated": m.feature_last_activated.clone(), "step_count": int(m.step_count)}


def crosscoder_case(name: str, d: int, L: int, F: int, k: int, B: int, seed: int,
                    layer_indices: list[int] | None = None) -> dict:
    torch.manual_seed(seed)
    m = TopKCrossLayerCrosscoder(d, L, F, k=k, layer_indices=layer_indices)
    state = {n: v.clone() for n, v in m.state_dict().items()}
    acts = {li: _inputs(seed + 20 + i, B, d) for i, li in enumerate(m.layer_indices)}
    m.train()
    out = m(acts)
    out.loss.backward()
    return {"recipe": dict(name=name, d=d, L=L, F=F, k=k, B=B, seed=seed, layer_indices=list(m.layer_indices)),
            "state": state, "loss": out.loss.item(), "l0": out.l0.item(),
            "hidden": out.hidden.detach().clone(),
            "per_layer_loss": {li: v.item() for li, v in out.per_layer_loss.items()},
            "grads": {n: p.grad.clone() for n, p in m.named_parameters()},
            "feature_last_activated": m.feature_last_activated.clone(), "step_count": int(m.step_count)}


if __name__ == "__main__":
    torch.set_num_threads(8)
    cases = {
        # shapes of tests/test_transcoder.py:17-24 and tests/test_crosscoder.py:17-25,421-454
        "transcoder_64_64_128_k8": transcoder_case("transcoder_64_64_128_k8", False, 64, 64, 128, 8, 16, 3),
        "transcoder_96_64_256_k16": transcoder_case("transcoder_96_64_256_k16", False, 96, 64, 256, 16, 40, 4),
        "skip_64_64_128_k8": transcoder_case("skip_64_64_128_k8", True, 64, 64, 128, 8, 16, 5),
        "crosscoder_64x4_128_k8": crosscoder_case("crosscoder_64x4_128_k8", 64, 4, 128, 8, 16, 6),
        "crosscoder_subset_64x2_128_k8": crosscoder_case("crosscoder_subset_64x2_128_k8", 64, 2, 128, 8, 16, 7,
                                                         layer_indices=[1, 2]),
        "crosscoder_tiny_384x4_3072_k32": crosscoder_case("crosscoder_tiny_384x4_3072_k32", 384, 4, 3072, 32, 8, 8),
    }
    # keep the whisper-tiny fixture small: grads as digests
    big = cases["crosscoder_tiny_384x4_3072_k32"]
    big["state_seed_only"] = True
    for key in ("state", "hidden"):
        big.pop(key)
    big["grads"] = {n: {"sum": g.double().sum().item(), "abs_sum": g.double().abs().sum().item(),
                        "sample": g.reshape(-1)[::997].clone()} for n, g in big["grads"].items()}
    GOLDEN.mkdir(parents=True, exist_ok=True)
    torch.save({n: c for n, c in cases.items() if not n.startswith("crosscoder")}, GOLDEN / "variants.pt")
    torch.save({n: c for n, c in cases.items() if n.startswith("crosscoder")}, GOLDEN / "variants_crosscoder.pt")
    for n, c in cases.items():
        print(n, "loss", round(c["loss"], 6), "l0", c["l0"])
