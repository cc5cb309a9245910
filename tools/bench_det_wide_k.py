"""Cost of deterministic=True at k in {32, 48, 64, 128, 256} (B200).

  python tools/bench_det_wide_k.py [--rows 75776] [--blocks 7] [--steps 10] [--out FILE]

For each shape (384 -> 3072, 768 -> 6144) and k: the graphed bf16 SAETrainer step in the default mode
and with deterministic=True, alternating blocks of --steps back-to-back steps of the two (CUDA events
around each block after warm-up; the median block's time per step).  Then, outside the timed window,
a torch.profiler pass over --steps replays of each arm gives the device time per step of every kernel,
so the difference between the arms is attributed kernel by kernel.  At k = 128 and 256 it also times
(CUDA events, median of --reps single calls, on the step's own operands) the team-of-warps K23 with
and without det_ws (the det form includes its det_finish launch) and the two K4 weight-gradient GEMMs
with and without the ordered split-K workspace.  The card's name and power limit are printed beside
the numbers.  Needs a GPU; there is no CPU fallback.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
from collections import defaultdict
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from oracle import topk_sae_oracle as O  # noqa: E402
from whisper_sae_b200 import ops  # noqa: E402
from whisper_sae_b200.config import TrainingConfig  # noqa: E402
from whisper_sae_b200.sae import SAETrainer, TopKSAE  # noqa: E402


def card() -> dict:
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # noqa: BLE001
        info["power_limit"] = f"unavailable ({e})"
    return info


def make_trainer(d: int, F: int, k: int, rows: int, run_dir: Path, deterministic: bool) -> SAETrainer:
    torch.manual_seed(0)
    sae = TopKSAE(d, F, k=k)
    cfg = TrainingConfig(batch_size=rows, use_amp=True, num_workers=0)
    tr = SAETrainer(sae, cfg, device="cuda", run_dir=run_dir, deterministic=deterministic)
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


def kernel_table(fn, steps: int, tmp: Path) -> dict:
    """Device microseconds per step of every kernel ``steps`` calls of ``fn`` launch (torch.profiler,
    kernel records of its trace; template arguments kept, so the two team-form instantiations differ)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    trace = tmp / "trace.json"
    prof.export_chrome_trace(str(trace))
    per = defaultdict(float)
    for ev in json.loads(trace.read_text()).get("traceEvents", []):
        if ev.get("cat") == "kernel":
            name = ev["name"].split("(")[0].replace("void ", "").replace("wsae::", "")
            per[name] += float(ev.get("dur", 0.0)) / steps
    trace.unlink()
    return dict(sorted(per.items(), key=lambda kv: -kv[1]))


def kernel_spans(tr: SAETrainer, x: torch.Tensor, reps: int) -> dict:
    """K23 (team form) and the two K4 GEMMs, each with and without its deterministic workspace."""
    m = tr.model
    B, d = x.shape
    F, k = m.hidden_dim, m.k
    a = ops.pack_activations(x, m.b_pre.data, 1)
    w = ops.pack_encoder(m.encoder.weight.data, m.encoder.bias.data, 1)
    w_used = ops.cast_bf16(m.decoder.weight.data.t())
    idx, val = ops.encode_topk(a, w, B, F, d, 1, k)
    resid_bf = torch.empty(B, d, dtype=torch.bfloat16, device="cuda")
    stats = torch.zeros(3, dtype=torch.int64, device="cuda")
    dbe, dbd = torch.zeros(F, device="cuda"), torch.zeros(d, device="cuda")
    dpre = torch.empty(B, k, device="cuda")
    one = torch.ones((), device="cuda")
    coef = 2.0 / (B * d)
    det_k23 = torch.zeros(F + d + 1, dtype=torch.int64, device="cuda")
    ws_bytes = ops.wgrad_gemm_workspace(B, F, d)
    det_k4 = torch.empty(max(ws_bytes // 4, 1), dtype=torch.float32, device="cuda")

    def k23(det: bool):
        # the int64 sums wrap harmlessly over the repetitions; only the time is kept
        ops.decode_backward(x, w_used, m.decoder.bias.data, m.b_pre.data, idx, val, one, coef,
                            resid=None, resid_bf16=resid_bf, stats=stats, last_activated=m.feature_last_activated,
                            step_count=m.step_count, d_b_enc=dbe, d_b_dec=dbd, dpre_val=dpre,
                            det_ws=det_k23 if det else None)

    k23(False)
    buckets = ops.bucket_by_tile(idx, val, dpre, F)
    g_enc, g_dec = torch.zeros(F, d, device="cuda"), torch.zeros(F, d, device="cuda")

    def k4(det: bool):
        ws = det_k4 if det and ws_bytes else None
        ops.wgrad_gemm_(g_enc, a, B, d, buckets, buckets.dpre, None, 1.0, det_ws=ws)
        ops.wgrad_gemm_(g_dec, resid_bf, B, d, buckets, buckets.act, one, coef, det_ws=ws)

    out = {"k23_entries": B * k, "k4_det_workspace_bytes": ws_bytes}
    for name, fn in (("k23_team", k23), ("k4_pair", k4)):
        for det in (False, True):
            fn(det)
        times = {False: [], True: []}
        for _ in range(reps):                      # alternate the two forms call by call
            for det in (False, True):
                times[det].append(time_block(lambda det=det: fn(det), 1))
        out[f"{name}_ms"] = statistics.median(times[False])
        out[f"{name}_det_ms"] = statistics.median(times[True])
    return out


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rows", type=int, default=75776)
    ap.add_argument("--blocks", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--ks", default="32,48,64,128,256")
    ap.add_argument("--span-ks", default="128,256")
    ap.add_argument("--shapes", default="384x3072,768x6144")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_det_wide_k.py measures on a CUDA device; none found")
    os.environ.pop("WSAE_WIDE_K23", None)      # the default mode's own routing (K2 + K3 at 33..64)
    torch.cuda.set_device(0)
    lines = [{"card": card(), "rows": args.rows, "blocks": args.blocks, "steps_per_block": args.steps}]
    print(json.dumps(lines[0]), flush=True)
    tmp = Path(tempfile.mkdtemp(prefix="wsae_bench_det_wide_k_"))
    span_ks = {int(v) for v in args.span_ks.split(",") if v}
    for shape in args.shapes.split(","):
        d, F = (int(v) for v in shape.split("x"))
        x = O.synthetic_activations(args.rows, d, seed=1).cuda()
        for k in (int(v) for v in args.ks.split(",")):
            trainers = {}
            for arm, det in (("default", False), ("deterministic", True)):
                tr = make_trainer(d, F, k, args.rows, tmp / f"{d}_{k}_{arm}", det)
                for _ in range(args.warmup):        # eager step, capture, replays
                    tr.train_step(x)
                torch.cuda.synchronize()
                gs = tr._graphs[args.rows]
                assert gs.graph is not None and gs.det == det, "the step was not graphed in this mode"
                trainers[arm] = tr
            times = {arm: [] for arm in trainers}
            for _ in range(args.blocks):             # alternate the arms block by block
                for arm, tr in trainers.items():
                    times[arm].append(time_block(lambda tr=tr: tr.train_step(x), args.steps))
            for arm, tr in trainers.items():
                ms = statistics.median(times[arm])
                gs = tr._graphs[args.rows]
                rec = {"d": d, "F": F, "k": k, "arm": arm, "step_ms": ms, "rows_per_s": args.rows / (ms * 1e-3),
                       "step_ms_blocks": times[arm], "k23": gs.state.resid is None,
                       "kernels_per_replay": gs.kernels_per_replay,
                       "kernel_us_per_step": kernel_table(lambda tr=tr: tr.train_step(x), args.steps, tmp)}
                lines.append(rec)
                print(json.dumps(rec), flush=True)
            if k in span_ks:
                rec = {"d": d, "F": F, "k": k, "arm": "spans"}
                rec.update(kernel_spans(trainers["default"], x, args.reps))
                lines.append(rec)
                print(json.dumps(rec), flush=True)
            del trainers
            torch.cuda.empty_cache()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
