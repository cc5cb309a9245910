"""CPU oracle for the transcoder / crosscoder variants of the hot path — TEST INFRASTRUCTURE ONLY
(same rules as topk_sae_oracle.py: imported by tests/ only; the product path never touches it).

Plain-tensor restatements (dense torch ops + autograd for the gradients) of

    /root/reference/src/whisper_sae/sae/transcoder.py   TopKTranscoder (:102-170), SkipTranscoder (:328-372)
    /root/reference/src/whisper_sae/sae/crosscoder.py   TopKCrossLayerCrosscoder (:326-379), decode (:171-188)

operating on ``state_dict``-shaped dicts.  Pinned by ``oracle/make_golden_variants.py`` (live
reference) -> ``tests/golden/variants{,_crosscoder}.pt`` -> ``tests/test_oracle_golden.py``.
"""

from __future__ import annotations

import torch
from torch import Tensor


def _topk_hidden(pre: Tensor, k: int) -> Tensor:
    vals, idx = torch.topk(pre, k, dim=-1)
    return torch.zeros_like(pre).scatter_(-1, idx, torch.relu(vals))


def transcoder(state: dict[str, Tensor], x: Tensor, y: Tensor, k: int, want_grads: bool = True) -> dict:
    """loss = mse(TopK(x W_enc^T + b_enc) W_dec^T + b_dec [+ x W_skip^T + b_skip], y)."""
    p = {n: v.clone().requires_grad_(v.is_floating_point()) for n, v in state.items()}
    hidden = _topk_hidden(x @ p["encoder.weight"].t() + p["encoder.bias"], k)
    pred = hidden @ p["decoder.weight"].t() + p["decoder.bias"]
    if "skip.weight" in p:
        pred = pred + x @ p["skip.weight"].t() + p["skip.bias"]
    loss = torch.nn.functional.mse_loss(pred, y)
    out = {"loss": loss.item(), "l0": (hidden > 0).float().sum(-1).mean().item(),
           "hidden": hidden.detach(), "predicted": pred.detach(), "fired": (hidden > 0).any(0)}
    if want_grads:
        loss.backward()
        out["grads"] = {n: v.grad.clone() for n, v in p.items() if v.requires_grad and v.grad is not None}
    return out


def crosscoder(state: dict[str, Tensor], acts: dict[int, Tensor], layer_indices: list[int], k: int,
               want_grads: bool = True) -> dict:
    """pre = sum_l x_l W_enc[l] + b_enc; recon_l = h W_dec[:, l] + b_dec[l]; loss = sum_l mean_l."""
    p = {n: v.clone().requires_grad_(v.is_floating_point()) for n, v in state.items()}
    pre = p["b_enc"].unsqueeze(0)
    for li, a in acts.items():
        pre = pre + a @ p["W_enc"][layer_indices.index(li)]
    hidden = _topk_hidden(pre, k)
    per_layer, recon = {}, {}
    loss = torch.zeros(())
    for i, li in enumerate(layer_indices):
        recon[li] = hidden @ p["W_dec"][:, i, :] + p["b_dec"][i]
        per_layer[li] = torch.mean((recon[li] - acts[li]) ** 2)
        loss = loss + per_layer[li]
    out = {"loss": loss.item(), "l0": (hidden > 0).float().sum(-1).mean().item(),
           "hidden": hidden.detach(), "reconstructed": {li: r.detach() for li, r in recon.items()},
           "per_layer_loss": {li: v.item() for li, v in per_layer.items()}, "fired": (hidden > 0).any(0)}
    if want_grads:
        loss.backward()
        out["grads"] = {n: v.grad.clone() for n, v in p.items() if v.requires_grad and v.grad is not None}
    return out
