"""Train-step rate on fp32, bf16 and fp16 activation matrices, alternated on one card (B200).

  python tools/bench_half_inputs.py [--rows 75776] [--blocks 7] [--steps 10] [--out FILE]

A bf16 / fp16 batch is read in place by the graphed step (K0, K23 and the row step convert at the
load), so its results equal the fp32 step's on ``Xh.float()``; what changes is the bytes per row.  Legs,
each with one trainer per dtype (same initial weights) and the dtypes alternated block by block:
  1. the graphed step on a resident matrix of 4 batches, contiguous batches and IndexedBatch shuffled
     batches, at 384 -> 3072 (k = 32 and k = 128) and 768 -> 6144 (k = 32);
  2. the shipped 128-row YAML batch (the row step), 384 -> 3072, k = 32;
  3. e2e: pinned host batches through SAETrainer.train_epoch (H2D copy inside), 384 -> 3072, k = 32;
  4. CUDA-event spans of K0 (pack, slot form) and K23 (decode + backward, slot form) per dtype.
Each number is the median block's time per step (as bench.py reports it).  The card's name and power
limit are read in the same call and written first.  Needs a GPU; there is no CPU fallback.
"""

from __future__ import annotations

import argparse
import json
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
from whisper_sae_b200.data.feature_cache import IndexedBatch  # noqa: E402
from whisper_sae_b200.sae import SAETrainer, TopKSAE  # noqa: E402

DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}


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
    tr = SAETrainer(sae, TrainingConfig(batch_size=rows, use_amp=True, num_workers=0), device="cuda",
                    run_dir=run_dir)
    tr.setup_scheduler(1_000_000)
    return tr


def time_block(fn, steps: int) -> float:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn(steps)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def alternate(runners: dict, steps: int, blocks: int, warmup: int) -> dict:
    """{dtype name: median ms per step}, the dtypes alternated block by block."""
    for run in runners.values():
        run(warmup)
    torch.cuda.synchronize()
    times = {n: [] for n in runners}
    for _ in range(blocks):
        for n, run in runners.items():
            times[n].append(time_block(run, steps))
    return {n: (statistics.median(t), t) for n, t in times.items()}


def step_runner(tr: SAETrainer, batches: list):
    pos = [0]

    def run(count: int) -> None:
        for _ in range(count):
            tr.train_step(batches[pos[0] % len(batches)])
            pos[0] += 1
    return run


def epoch_runner(tr: SAETrainer, host_batches: list):
    pos = [0]

    def run(count: int) -> None:
        tr.train_epoch([[host_batches[(pos[0] + i) % len(host_batches)]] for i in range(count)])
        pos[0] += count
    return run


def resident_leg(d, F, k, rows, args, tmp, emit, indexed_too=True):
    x32 = O.synthetic_activations(4 * rows, d, seed=d + k).cuda()
    mats = {n: x32.to(dt) for n, dt in DTYPES.items()}
    forms = ["contiguous", "indexed"] if indexed_too else ["contiguous"]
    for form in forms:
        runners, trainers = {}, {}
        for n, m in mats.items():
            tr = trainers[n] = make_trainer(d, F, k, rows, tmp / f"{form}_{d}_{k}_{rows}_{n}")
            if form == "contiguous":
                batches = [m[i * rows:(i + 1) * rows] for i in range(4)]
            else:
                perm = torch.randperm(4 * rows, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
                batches = [IndexedBatch(m, perm[i * rows:(i + 1) * rows]) for i in range(4)]
            runners[n] = step_runner(tr, batches)
        res = alternate(runners, args.steps, args.blocks, args.warmup)
        for n, (ms, blocks) in res.items():
            gs = trainers[n]._graphs[rows]
            emit({"leg": "resident", "form": form, "d": d, "F": F, "k": k, "rows": rows, "dtype": n,
                  "step_ms": ms, "rows_per_s": rows / (ms * 1e-3), "step_ms_blocks": blocks,
                  "in_place": gs._x is None, "row_step": bool(gs.row_step),
                  "kernels_per_replay": gs.kernels_per_replay})
        del trainers, runners
        torch.cuda.empty_cache()
    return mats


def e2e_leg(d, F, k, rows, args, tmp, emit):
    x32 = O.synthetic_activations(4 * rows, d, seed=99)
    runners = {}
    for n, dt in DTYPES.items():
        host = [x32[i * rows:(i + 1) * rows].to(dt).pin_memory() for i in range(4)]
        runners[n] = epoch_runner(make_trainer(d, F, k, rows, tmp / f"e2e_{n}"), host)
    res = alternate(runners, args.steps, args.blocks, args.warmup)
    for n, (ms, blocks) in res.items():
        bpr = d * DTYPES[n].itemsize
        emit({"leg": "e2e_pinned_host", "d": d, "F": F, "k": k, "rows": rows, "dtype": n, "step_ms": ms,
              "rows_per_s": rows / (ms * 1e-3), "h2d_bytes_per_row": bpr,
              "h2d_GBs": rows * bpr / (ms * 1e-3) / 1e9, "step_ms_blocks": blocks})


def kernel_leg(d, F, k, rows, mats, reps, tmp, emit):
    """K0 and K23 spans (slot forms) on one model's operands, for each dtype of the same matrix."""
    tr = make_trainer(d, F, k, rows, tmp / "kernels")
    m = tr.model
    x32 = mats["fp32"][:rows]
    a = ops.pack_activations(x32, m.b_pre.data, 1)
    w = ops.pack_encoder(m.encoder.weight.data, m.encoder.bias.data, 1)
    w_used = ops.cast_bf16(m.decoder.weight.data.t())
    idx, val = ops.encode_topk(a, w, rows, F, d, 1, k)
    resid_bf = torch.empty(rows, d, dtype=torch.bfloat16, device="cuda")
    stats = torch.zeros(3, dtype=torch.int64, device="cuda")
    dbe, dbd = torch.zeros(F, device="cuda"), torch.zeros(d, device="cuda")
    dpre = torch.empty(rows, k, device="cuda")
    one = torch.ones((), device="cuda")
    kp = ops.packed_shape(d, 1).kp
    for n, dt in DTYPES.items():
        xm = mats[n][:rows]
        slot = torch.tensor([xm.data_ptr()], dtype=torch.int64, device="cuda")

        def k0(count, slot=slot, dt=dt):
            for _ in range(count):
                ops.pack_activations_at(slot, rows, d, m.b_pre.data, out=a, x_dtype=dt)

        def k23(count, slot=slot, dt=dt):
            for _ in range(count):
                ops.decode_backward(slot, w_used, m.decoder.bias.data, m.b_pre.data, idx, val, one, 1.0 / (rows * d),
                                    resid=None, resid_bf16=resid_bf, stats=stats,
                                    last_activated=m.feature_last_activated, step_count=m.step_count, d_b_enc=dbe,
                                    d_b_dec=dbd, dpre_val=dpre, target_is_slot=True, x_dtype=dt)
        for name, fn, nbytes in (("K0_pack", k0, rows * d * dt.itemsize + a.shape[0] * kp * 2),
                                 ("K23_decode_backward", k23, None)):
            fn(3)
            ms = statistics.median(time_block(fn, 20) for _ in range(reps))
            rec = {"leg": "kernel", "kernel": name, "d": d, "F": F, "k": k, "rows": rows, "dtype": n, "ms": ms,
                   "activation_bytes": rows * d * dt.itemsize}
            if nbytes is not None:
                rec.update({"hbm_bytes": nbytes, "hbm_TBs": nbytes / (ms * 1e-3) / 1e12})
            emit(rec)


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rows", type=int, default=75776)
    ap.add_argument("--blocks", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_half_inputs.py measures on a CUDA device; none found")
    torch.cuda.set_device(0)
    lines = []

    def emit(rec):
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    emit({"card": card(), "rows": args.rows, "blocks": args.blocks, "steps_per_block": args.steps})
    tmp = Path(tempfile.mkdtemp(prefix="wsae_bench_half_"))
    mats = resident_leg(384, 3072, 32, args.rows, args, tmp, emit)
    kernel_leg(384, 3072, 32, args.rows, mats, max(5, args.blocks), tmp, emit)
    del mats
    resident_leg(384, 3072, 128, args.rows, args, tmp, emit)
    resident_leg(768, 6144, 32, args.rows, args, tmp, emit)
    resident_leg(384, 3072, 32, 128, args, tmp, emit, indexed_too=False)
    e2e_leg(384, 3072, 32, args.rows, args, tmp, emit)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
