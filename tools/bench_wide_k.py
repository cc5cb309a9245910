"""Train-step time and per-kernel spans of TopK SAEs at k in {32, 64, 128, 256} (B200).

  python tools/bench_wide_k.py [--rows 75776] [--blocks 7] [--steps 10] [--out FILE]

For each shape (384 -> 3072, 768 -> 6144) and k: the graphed bf16 SAETrainer step (CUDA events around
--blocks blocks of --steps back-to-back steps after warm-up; the median block's time per step), and
CUDA-event spans of the two kernels wide k adds - K1 chunked (wsae_encode_topk_chunked) and the
team-of-warps K23 - on that step's own operands.  At k = 64 the step is also timed with
WSAE_WIDE_K23=1 (team-of-warps K23 instead of K2 + K3), alternating blocks of both settings in one
run.  K23's gathered bytes (B * k * d * 2) are reported against the measured L2 row-gather ceiling of
DESIGN.md section 4 (16.2 TB/s, profiles/r2_l2_gather.json).  The card's name and power limit are
printed beside the numbers.  Needs a GPU; there is no CPU fallback.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from oracle import topk_sae_oracle as O  # noqa: E402
from whisper_sae_b200 import ops  # noqa: E402
from whisper_sae_b200.config import TrainingConfig  # noqa: E402
from whisper_sae_b200.sae import SAETrainer, TopKSAE  # noqa: E402

L2_GATHER_CEILING_TBS = 16.2


def card() -> dict:
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # noqa: BLE001
        info["power_limit"] = f"unavailable ({e})"
    return info


def make_trainer(d: int, F: int, k: int, rows: int, run_dir: Path) -> SAETrainer:
    torch.manual_seed(0)
    sae = TopKSAE(d, F, k=k)
    cfg = TrainingConfig(batch_size=rows, use_amp=True, num_workers=0)
    tr = SAETrainer(sae, cfg, device="cuda", run_dir=run_dir)
    tr.setup_scheduler(10_000)
    return tr


def time_block(fn, steps: int) -> float:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def kernel_spans(tr: SAETrainer, x: torch.Tensor, reps: int) -> dict:
    """Median CUDA-event time of K1 (as routed) and of K23 (as routed) on this model's operands."""
    m = tr.model
    B, d = x.shape
    F, k = m.hidden_dim, m.k
    a = ops.pack_activations(x, m.b_pre.data, 1)
    w = ops.pack_encoder(m.encoder.weight.data, m.encoder.bias.data, 1)
    w_used = ops.cast_bf16(m.decoder.weight.data.t())
    out = {"k1_route": ops.encode_route(B, F, k)}
    idx, val = ops.encode_topk(a, w, B, F, d, 1, k)
    out["k1_ms"] = statistics.median(time_block(lambda: ops.encode_topk(a, w, B, F, d, 1, k), 1) for _ in range(reps))
    if not ops.decode_backward_supported(d, k, True) and k <= 64:
        return out
    resid_bf = torch.empty(B, d, dtype=torch.bfloat16, device="cuda")
    stats = torch.zeros(3, dtype=torch.int64, device="cuda")
    dbe, dbd = torch.zeros(F, device="cuda"), torch.zeros(d, device="cuda")
    dpre = torch.empty(B, k, device="cuda")
    one = torch.ones((), device="cuda")

    def k23():
        ops.decode_backward(x, w_used, m.decoder.bias.data, m.b_pre.data, idx, val, one, 1.0 / (B * d),
                            resid=None, resid_bf16=resid_bf, stats=stats, last_activated=m.feature_last_activated,
                            step_count=m.step_count, d_b_enc=dbe, d_b_dec=dbd, dpre_val=dpre)

    k23()
    ms = statistics.median(time_block(k23, 1) for _ in range(reps))
    gathered = B * k * d * 2
    out.update({"k23_form": "warp" if k <= 32 else "team", "k23_ms": ms, "k23_gather_GB": gathered / 1e9,
                "k23_gather_TBs": gathered / (ms * 1e-3) / 1e12,
                "k23_share_of_l2_gather_ceiling": gathered / (ms * 1e-3) / 1e12 / L2_GATHER_CEILING_TBS})
    return out


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rows", type=int, default=75776)
    ap.add_argument("--blocks", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--ks", default="32,64,128,256")
    ap.add_argument("--shapes", default="384x3072,768x6144")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wide_k.py measures on a CUDA device; none found")
    torch.cuda.set_device(0)
    lines = [{"card": card(), "rows": args.rows, "blocks": args.blocks, "steps_per_block": args.steps}]
    print(json.dumps(lines[0]), flush=True)
    tmp = Path(tempfile.mkdtemp(prefix="wsae_bench_wide_k_"))
    for shape in args.shapes.split(","):
        d, F = (int(v) for v in shape.split("x"))
        x = O.synthetic_activations(args.rows, d, seed=1).cuda()
        for k in (int(v) for v in args.ks.split(",")):
            arms = {"default": None}
            if k == 64:
                arms["WSAE_WIDE_K23=1"] = "1"
            trainers = {}
            for name, env in arms.items():
                if env is None:
                    os.environ.pop("WSAE_WIDE_K23", None)
                else:
                    os.environ["WSAE_WIDE_K23"] = env
                tr = make_trainer(d, F, k, args.rows, tmp / f"{d}_{k}_{len(trainers)}")
                for _ in range(args.warmup):        # eager step, capture, replays
                    tr.train_step(x)
                torch.cuda.synchronize()
                assert tr._graphs, "the step was not graphed"
                trainers[name] = tr
            times = {name: [] for name in arms}
            for _ in range(args.blocks):             # alternate the arms block by block
                for name, tr in trainers.items():
                    times[name].append(time_block(lambda tr=tr: tr.train_step(x), args.steps))
            os.environ.pop("WSAE_WIDE_K23", None)
            for name, tr in trainers.items():
                ms = statistics.median(times[name])
                rec = {"d": d, "F": F, "k": k, "arm": name, "step_ms": ms, "rows_per_s": args.rows / (ms * 1e-3),
                       "step_ms_blocks": times[name]}
                if name == "default":
                    rec.update(kernel_spans(tr, x, reps=max(5, args.blocks)))
                lines.append(rec)
                print(json.dumps(rec), flush=True)
            del trainers
            torch.cuda.empty_cache()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
