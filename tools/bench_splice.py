"""Measure the fused SAE splice (sae/splice.py, csrc/wsae_splice.cu) on random-init Whisper encoders.

Models are built from seeds (nothing is downloaded) and run in fp16, the dtype Whisper is served in:
  * whisper-tiny shape:      d = 384, 4 encoder layers, SAE 384 -> 3072, spliced at encoder layer 2;
  * whisper-large-v3 shape:  d = 1280, 32 encoder layers, SAE 1280 -> 40960, spliced at encoder layer 16.
Input: 8 clips x 3000 mel frames (N = 8 x 1500 = 12 000 rows per spliced layer), k in {32, 128}.

Per (model, k), CUDA events, after warm-up:
  * clean encoder forward;
  * the forward with WhisperSAESplice in replace mode, and in error mode with 16 ablated features;
  * the same splice as a plain PyTorch hook (the reference module's arithmetic written out: LayerNorm,
    nn.Linear, torch.topk, scatter into a dense [N, F] code, dense decode, inverse LayerNorm, in fp32);
  * wsae_splice_pack and wsae_splice_decode alone on the layer's hidden rows, each launch timed after a
    256 MB write that evicts L2 (126 MB), with the bytes each must move computed from the shapes:
    pack reads N*d*sizeof(h) and writes Bp*Kp*2 + 8N (share of 7.7 TB/s HBM); decode gathers at least
    N*l0*d*2 bytes of decoder rows (share of the 16.2 TB/s L2 row-gather ceiling measured by
    tools/l2_gather_bench.cu, profiles/r2_l2_gather.json).
One JSON line per measurement to --out, each with the card name and power limit read in the same run.
"""

from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from whisper_sae_b200 import ops  # noqa: E402
from whisper_sae_b200.sae import TopKSAE, WhisperSAESplice  # noqa: E402
from whisper_sae_b200.sae.hooks import _hidden_of  # noqa: E402

HBM_BPS = 7.7e12
L2_GATHER_BPS = 16.2e12

SHAPES = {
    "tiny": dict(d_model=384, encoder_layers=4, encoder_attention_heads=6, encoder_ffn_dim=1536, F=3072, site=2),
    "large-v3": dict(d_model=1280, encoder_layers=32, encoder_attention_heads=20, encoder_ffn_dim=5120, F=40960,
                     site=16),
}


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power = (q[0].split(", ") + ["?"])[:2] if q else (torch.cuda.get_device_name(), "?")
    return {"card": name, "power_limit": power}


def build(shape: dict):
    from transformers import WhisperConfig, WhisperForConditionalGeneration
    cfg = WhisperConfig(d_model=shape["d_model"], encoder_layers=shape["encoder_layers"], decoder_layers=1,
                        encoder_attention_heads=shape["encoder_attention_heads"], decoder_attention_heads=2,
                        encoder_ffn_dim=shape["encoder_ffn_dim"], decoder_ffn_dim=256, num_mel_bins=80,
                        max_source_positions=1500, max_target_positions=448, vocab_size=1000,
                        decoder_start_token_id=1, pad_token_id=0, bos_token_id=1, eos_token_id=2)
    torch.manual_seed(0)
    model = WhisperForConditionalGeneration(cfg).eval()
    with torch.no_grad():
        g = torch.Generator().manual_seed(1)
        ln = model.model.encoder.layer_norm
        ln.weight.copy_(1.0 + 0.1 * torch.randn(ln.weight.shape, generator=g))
        ln.bias.copy_(0.1 * torch.randn(ln.bias.shape, generator=g))
    return model.to("cuda", torch.float16)


def time_ms(fn, warmup: int, reps: int) -> float:
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def time_cold_ms(fn, reps: int, scratch: torch.Tensor) -> float:
    """Mean time of one launch of fn, each after a write of ``scratch`` that evicts L2."""
    fn()
    total = 0.0
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        scratch.fill_(1)
        a.record()
        fn()
        b.record()
        b.synchronize()
        total += a.elapsed_time(b)
    return total / reps


def torch_splice_hook(sae: TopKSAE, ln):
    """The reference module's arithmetic as a PyTorch hook (replace mode, fp32)."""
    W_enc, b_enc = sae.encoder.weight.detach(), sae.encoder.bias.detach()
    W_dec, b_dec, b_pre = sae.decoder.weight.detach(), sae.decoder.bias.detach(), sae.b_pre.detach()
    gamma, beta, eps = ln.weight.detach().float(), ln.bias.detach().float(), ln.eps

    def hook(m, i, o):
        h = _hidden_of(o)
        h2 = h.reshape(-1, h.shape[-1]).float()
        x = torch.nn.functional.layer_norm(h2, (h2.shape[1],), gamma, beta, eps)
        pre = torch.nn.functional.linear(x - b_pre, W_enc, b_enc)
        v, i = torch.topk(pre, sae.k, dim=-1)
        hidden = torch.zeros_like(pre).scatter_(1, i, torch.relu(v))
        recon = torch.nn.functional.linear(hidden, W_dec, b_dec) + b_pre
        mu = h2.mean(1, keepdim=True)
        r = torch.rsqrt(((h2 - mu) ** 2).mean(1, keepdim=True) + eps)
        out = (mu + ((recon - beta) / gamma) / r).to(h.dtype).reshape(h.shape)
        return (out,) + tuple(o[1:]) if isinstance(o, tuple) else out
    return hook


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSONL file the measurements are appended to")
    ap.add_argument("--models", default="tiny,large-v3")
    ap.add_argument("--ks", default="32,128")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_splice needs a CUDA device")
    info = card()
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    feats = torch.randn(8, 80, 3000, generator=torch.Generator().manual_seed(2)).to("cuda", torch.float16)
    with out.open("a") as f, torch.no_grad():
        def emit(**rec):
            rec.update(info)
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + "\n")

        for name in args.models.split(","):
            shape = SHAPES[name]
            model = build(shape)
            enc = model.model.encoder
            d, F, layer = shape["d_model"], shape["F"], shape["site"]
            clean_ms = time_ms(lambda: enc(feats), args.warmup, args.reps)
            emit(model=name, what="clean_encoder_forward", ms=clean_ms)
            captured = {}
            hcap = enc.layers[layer].register_forward_hook(lambda m, i, o: captured.__setitem__("h", _hidden_of(o)))
            enc(feats)
            hcap.remove()
            h = captured["h"].reshape(-1, d).contiguous()
            N = h.shape[0]
            for k in (int(s) for s in args.ks.split(",")):
                torch.manual_seed(3)
                sae = TopKSAE(d, F, k=k, precision="bf16").cuda().eval()
                site = ("encoder", layer)
                rec = dict(model=name, d=d, F=F, k=k, rows=N)
                # each hooked forward is timed right after a clean one, so both see the same clocks
                sp = WhisperSAESplice(model, {site: sae}, mode="replace", collect_stats=False)
                rec["clean_ms"] = clean_ms = time_ms(lambda: enc(feats), args.warmup, args.reps)
                with sp:
                    ms = time_ms(lambda: enc(feats), args.warmup, args.reps)
                emit(what="splice_replace_forward", ms=ms, over_clean_ms=ms - clean_ms, **rec)
                gain = torch.ones(F, device="cuda")
                gain[torch.randperm(F, generator=torch.Generator().manual_seed(4))[:16].cuda()] = 0.0
                se = WhisperSAESplice(model, {site: sae}, mode="error", collect_stats=False)
                rec["clean_ms"] = clean_ms = time_ms(lambda: enc(feats), args.warmup, args.reps)
                with se:
                    se.set_intervention(site, gain=gain)
                    ms = time_ms(lambda: enc(feats), args.warmup, args.reps)
                emit(what="splice_error_ablate16_forward", ms=ms, over_clean_ms=ms - clean_ms, **rec)
                sst = WhisperSAESplice(model, {site: sae}, mode="replace", collect_stats=True)
                rec["clean_ms"] = clean_ms = time_ms(lambda: enc(feats), args.warmup, args.reps)
                with sst:
                    ms = time_ms(lambda: enc(feats), args.warmup, args.reps)
                    st = sst.stats(site)
                emit(what="splice_replace_forward_with_stats", ms=ms, over_clean_ms=ms - clean_ms,
                     l0=st.l0, fvu=st.fvu, **rec)
                rec["clean_ms"] = clean_ms = time_ms(lambda: enc(feats), args.warmup, args.reps)
                th = enc.layers[layer].register_forward_hook(torch_splice_hook(sae, model.model.encoder.layer_norm))
                ms = time_ms(lambda: enc(feats), args.warmup, args.reps)
                th.remove()
                emit(what="torch_hook_replace_forward", ms=ms, over_clean_ms=ms - clean_ms, **rec)

                # the two kernels alone, L2 evicted before each launch
                rec = dict(model=name, d=d, F=F, k=k, rows=N)
                ln = model.model.encoder.layer_norm
                gamma, beta = ln.weight.float(), ln.bias.float()
                b_pre = sae.b_pre.detach()
                a_packed, rs = ops.splice_pack(h, gamma, beta, ln.eps, b_pre)
                ps = ops.packed_shape(d, 1)
                Bp = a_packed.shape[0]
                pack_bytes = N * d * h.element_size() + Bp * ps.kp * 2 + 8 * N
                ms = time_cold_ms(lambda: ops.splice_pack(h, gamma, beta, ln.eps, b_pre, out=a_packed, row_stats=rs),
                                  50, scratch)
                emit(what="wsae_splice_pack", ms=ms, bytes=pack_bytes, tbps=pack_bytes / ms / 1e9,
                     hbm_share=pack_bytes / ms / 1e9 / (HBM_BPS / 1e12), **rec)
                w_packed = ops.pack_encoder(sae.encoder.weight.detach().contiguous(), sae.encoder.bias.detach(), 1)
                idx, val = ops.encode_topk(a_packed, w_packed, N, F, d, 1, k)
                w_bf = ops.cast_bf16(sae.decoder.weight.detach().t().contiguous())
                b_dec = sae.decoder.bias.detach()
                l0 = int((val > 0).sum()) / N
                out_h = torch.empty_like(h)
                for mode, g_ in (("replace", None), ("error", gain)):
                    ms = time_cold_ms(lambda: ops.splice_decode(h, rs, gamma, beta, w_bf, b_dec, b_pre, idx, val,
                                                                mode=mode, gain=g_, out=out_h), 50, scratch)
                    gather = N * l0 * d * 2 if mode == "replace" else 0
                    r = dict(what=f"wsae_splice_decode_{mode}", ms=ms, l0=l0, **rec)
                    if gather:
                        r.update(gather_bytes=gather, tbps=gather / ms / 1e9,
                                 l2_gather_share=gather / ms / 1e9 / (L2_GATHER_BPS / 1e12))
                    else:
                        r.update(note="error mode, 16 ablated features, no statistics: only ablated rows gathered")
                    emit(**r)
                del sae, sp, se, sst
            del model
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
