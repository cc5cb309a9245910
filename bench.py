#!/usr/bin/env python
"""bench.py — activation rows/s of the TopK-SAE train step (BASELINE.json metric) on N B200s.

    python bench.py --gpus 1 --steps 50 --warmup 10
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # CPU arm: the UNMODIFIED reference trainer on the host cores

Headline workload (BASELINE.json configs[1]): whisper-tiny TopKSAE 384 -> 3072, k = 32,
hyper-parameters of configs/tiny_default.yaml (lr 1e-4, warm-up 1000, clip 1.0, AMP on => bf16
path), synthetic row-standardised Gaussian activations (SURVEY §8d).  One "step" = one
`SAETrainer.train_step` (pack, tcgen05 GEMM + fused TopK, sparse decode + MSE, sparse backward,
clip + AdamW, decoder renorm, counters, metrics).  The YAML batch (128) is launch-latency bound by
construction, so the headline batch is `--batch` (default 75776 = 4 waves of 148 x 128-row tiles;
config-legal: TrainingConfig.batch_size >= 1); the YAML-batch number is reported as `yaml_batch`.

Timing: `--steps` K is the number of timed steps of the headline value (and of the e2e leg).  They
run back to back after `--warmup` untimed ones and CUDA events on the launching stream cut them into
`--repeats` blocks (at most K; barrier + synchronize before and after, max over ranks per block);
the MEDIAN block's time per step is reported, min / max next to it - one straggler block cannot set
the number.  The defaults, 1250 steps in 25 blocks of 50 (about 1 s at 0.76 ms per step), keep the
timed window long against clock and scheduler noise.

`--dump-outputs DIR` writes what the timed path returned in its last timed step (the step's metrics
and the model state it left, bench.dump_outputs) as DIR/<name>.npy; the inputs are seeded, so two
builds run with the same arguments can be compared output for output.

N > 1: one process per GPU, each training an independent layer's SAE (4 encoder + 4 decoder layers
of whisper-tiny; no data-path collective), value = sum of rows/s, weak scaling.  The same JSON line
carries a `workloads` block: whisper-small 768->6144 and large-v3 1280->40960 (BASELINE configs[2],
[3]) on one GPU, and at N > 1 their batch-sharded data-parallel step (NCCL gradient exchange) at a
fixed batch per rank (weak) and at a fixed global batch (strong).
"""

from __future__ import annotations

import argparse
import contextlib
import dataclasses
import gc
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# Workloads (BASELINE.json configs): "tiny" = configs[1] (headline; N GPUs train N independent layer
# SAEs, no collective); "small-dp" / "large-dp" = configs[2] / [3]: one SAE, batch sharded over the
# ranks, gradients all-reduced with NCCL.
WORKLOADS = {
    "tiny": dict(label="whisper-tiny", d=384, expansion=8, k=32, dp=False, cfg="configs[1]", batch=75776),
    "small-dp": dict(label="whisper-small", d=768, expansion=8, k=32, dp=True, cfg="configs[2]", batch=75776),
    "large-dp": dict(label="whisper-large-v3", d=1280, expansion=32, k=32, dp=True, cfg="configs[3]",
                     batch=37888),
}
METRIC = "sae_train_step_activation_rows_per_sec"
UNIT = "rows/s"
REF_DIR = ROOT / "baseline" / "_ref"


def load_peaks() -> tuple[dict, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()), "measured (MEASURED_PEAKS.json)"
    # fallback stated by /opt/skills/guides/B200_PROFILING.md
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def load_l2_ceiling() -> tuple[float | None, str | None]:
    """Measured L2 row-gather ceiling (GB/s) from tools/l2_gather_bench (profiles/r2_l2_gather.json)."""
    p = ROOT / "profiles" / "r2_l2_gather.json"
    if p.exists():
        try:
            j = json.loads(p.read_text())
            return float(j["ceiling_gbs"]), "profiles/r2_l2_gather.json (tools/l2_gather_bench.cu)"
        except Exception:
            pass
    return None, None


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: an NVML polling thread (5 ms
    cadence, so even a 30 ms region gets several samples); falls back to `nvidia-smi -lms`."""

    _REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
                ("sw_power_cap", 0x4))

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.samples: list[tuple[float, float, int]] = []
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None
        self.proc = None
        self.lines: list[str] = []

    def _physical_index(self) -> int:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if self.gpu_index < len(ids) and ids[self.gpu_index].isdigit():
                return int(ids[self.gpu_index])
        return self.gpu_index

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self._nvml = pynvml
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def poll():
                while not self._stop.is_set():
                    try:
                        sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        try:
                            rs = int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                        except Exception:
                            rs = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                        self.samples.append((sm, mx, rs))
                    except Exception:
                        pass
                    self._stop.wait(0.005)

            self._thread = threading.Thread(target=poll, daemon=True)
            self._thread.start()
        except Exception:
            self._nvml = None
            try:
                fields = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                          "clocks_event_reasons.hw_thermal_slowdown,"
                          "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
                self.proc = subprocess.Popen(
                    ["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={fields}",
                     "--format=csv,noheader,nounits", "-lms", "100"],
                    stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self._thread = threading.Thread(target=self._pump, daemon=True)
                self._thread.start()
            except OSError:
                self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *exc):
        self._stop.set()
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        if self._thread is not None:
            self._thread.join(timeout=2)

    def summary(self) -> dict:
        if self.samples:
            sm = [x[0] for x in self.samples]
            reasons = set()
            for _, _, rs in self.samples:
                for name, bit in self._REASONS:
                    if rs & bit:
                        reasons.add(name)
            return {"sm_mhz": statistics.median(sm), "sm_min_mhz": min(sm),
                    "sm_max_mhz": self.samples[0][1], "reasons": sorted(reasons),
                    "samples": len(sm), "source": "nvml"}
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, flag in zip(names, parts[3:7]):
                if flag.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}


def bind_to_gpu_numa_node(local_rank: int) -> dict:
    """Pin this rank's host threads to the CPUs of the GPU's NUMA node BEFORE any pinned staging
    buffer is allocated (first-touch places the pages there), so N ranks do not all stream their
    H2D copies out of node 0.  Returns what was found for the bench line."""
    info: dict = {"numa_node": None, "cpus": None}
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = local_rank
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if local_rank < len(ids) and ids[local_rank].isdigit():
                idx = int(ids[local_rank])
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:          # nvml: 00000000:1b:00.0 -> sysfs: 0000:1b:00.0
            bus = bus[4:]
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text().strip())
        info["numa_node"] = node
        nodes = [p for p in Path("/sys/devices/system/node").glob("node[0-9]*")]
        info["numa_nodes_online"] = len(nodes)
        if node >= 0 and len(nodes) > 1:
            cpulist = Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip()
            cpus: set[int] = set()
            for part in cpulist.split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
            allowed = cpus & os.sched_getaffinity(0)
            if allowed:
                os.sched_setaffinity(0, allowed)
                info["cpus"] = cpulist
    except Exception as e:  # noqa: BLE001 - topology probing is best effort
        info["error"] = str(e)[:80]
    return info


def make_trainer(wl: dict, batch: int, device: str, layer_seed: int, use_amp: bool = True, cuda_graph=None,
                 data_parallel: bool = False, global_rows: int | None = None, deterministic: bool = False):
    from whisper_sae_b200.config import ExperimentConfig
    from whisper_sae_b200.sae import SAETrainer, create_sae

    cfg = ExperimentConfig.from_yaml(ROOT / "configs" / "tiny_default.yaml")
    cfg.training.batch_size = batch
    cfg.training.use_amp = use_amp
    cfg.sae.expansion_factor = wl["expansion"]
    cfg.sae.k = wl["k"]
    torch.manual_seed(cfg.training.seed + layer_seed)
    sae = create_sae(cfg.sae, wl["d"])
    run_dir = Path(tempfile.mkdtemp(prefix="wsae_bench_"))
    tr = SAETrainer(sae, cfg.training, device=device, run_dir=run_dir, cuda_graph=cuda_graph,
                    data_parallel=data_parallel, global_batch_rows=global_rows, deterministic=deterministic)
    tr.setup_scheduler(100_000)
    return tr, cfg


def synth(n_rows: int, d: int, seed: int) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n_rows, d, generator=g)
    return (x - x.mean(1, keepdim=True)) / x.std(1, unbiased=False, keepdim=True)


def _max_over_ranks(vals: list[float], dist_on: bool) -> list[float]:
    if not dist_on:
        return vals
    t = torch.tensor(vals, device="cuda", dtype=torch.float64)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return t.tolist()


def time_blocks(run_steps, steps: int, warmup: int, repeats: int, dist_on: bool) -> tuple[dict, int]:
    """Exactly `steps` timed steps after `warmup` untimed ones, run back to back and cut into
    min(`repeats`, `steps`) consecutive blocks of near-equal length by CUDA events on the launching
    stream; barrier + synchronize before the first block and after the last, max over ranks per block.
    Returns seconds PER STEP (median / min / max over the blocks) and this rank's kernel launches
    over the `steps` steps."""
    from whisper_sae_b200 import ops

    run_steps(0, warmup)
    torch.cuda.synchronize()
    nblk = max(1, min(repeats, steps))
    sizes = [steps // nblk + (i < steps % nblk) for i in range(nblk)]
    events = [torch.cuda.Event(enable_timing=True) for _ in range(nblk + 1)]
    if dist_on:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    l0 = ops.GPU_LAUNCHES
    events[0].record()
    pos = warmup
    for i, n in enumerate(sizes):
        run_steps(pos, n)
        events[i + 1].record()
        pos += n
    torch.cuda.synchronize()
    launches = ops.GPU_LAUNCHES - l0
    if dist_on:
        torch.distributed.barrier()
    secs = [events[i].elapsed_time(events[i + 1]) / 1e3 / n for i, n in enumerate(sizes)]
    secs = _max_over_ranks(secs, dist_on)
    srt = sorted(secs)
    return {"median": statistics.median(secs), "min": srt[0], "max": srt[-1], "blocks": nblk}, launches


def step_runner(tr, batches):
    """run(pos, count): `count` train steps on `batches` from index `pos`; run.last is the
    TrainingMetrics of the latest step."""
    n = len(batches)

    def run(pos: int, count: int) -> None:
        for i in range(count):
            run.last = tr.train_step(batches[(pos + i) % n])
    run.last = None
    return run


DUMP_LIMIT_BYTES = 60 << 20          # with the .npy headers, under 64 MB however counted


def dump_outputs(out_dir: Path, metrics, model) -> None:
    """What a caller of the timed path holds after its last step, one `out_dir/<name>.npy` each: the
    returned TrainingMetrics fields (float64) and the model's state_dict (float32; integer counters as
    float64).  Above DUMP_LIMIT_BYTES in all, every array over 1 MiB keeps the same fraction of its
    elements, at sorted flat indices drawn from a generator seeded with 0: the same elements on every
    run with the same shapes."""
    import numpy as np

    arrays = {k: np.array(v, dtype=np.float64) for k, v in dataclasses.asdict(metrics).items()}
    for name, t in model.state_dict().items():
        t = t.detach().cpu().contiguous()
        arrays[name] = (t.float() if t.is_floating_point() else t.double()).numpy()
    big = sorted(k for k, a in arrays.items() if a.nbytes > 1 << 20)
    big_bytes = sum(arrays[k].nbytes for k in big)
    small_bytes = sum(a.nbytes for a in arrays.values()) - big_bytes
    if small_bytes + big_bytes > DUMP_LIMIT_BYTES:
        frac = (DUMP_LIMIT_BYTES - small_bytes) / big_bytes
        for k in big:
            flat = arrays[k].reshape(-1)
            idx = torch.randperm(flat.size, generator=torch.Generator().manual_seed(0))[:int(flat.size * frac)]
            arrays[k] = flat[idx.sort().values.numpy()]
    out_dir.mkdir(parents=True, exist_ok=True)
    for k, a in arrays.items():
        np.save(out_dir / f"{k}.npy", a)


def epoch_runner(tr, host_batches):
    """Through the public loop `SAETrainer.train_epoch` fed with pinned HOST batches: every step's
    H2D copy (prefetched one batch ahead on a copy stream) and its metrics readback (32 bytes the
    counters kernel posts to the pinned host mailbox) are inside the timed region."""
    n = len(host_batches)

    def run(pos: int, count: int) -> None:
        tr.train_epoch([[host_batches[(pos + i) % n]] for i in range(count)])
    return run


def resident_loader_rate(tr, rows: torch.Tensor, batch: int, dev: str, epochs: int = 3) -> dict:
    """SURVEY 8(f) rank 2: the activation matrix lives in HBM behind the `FeatureCache.get_dataloader(
    device=...)` iterable (`ResidentBatches`, shuffled: every batch is an IndexedBatch = matrix + a
    slice of the epoch's device permutation, gathered inside K0 / K23) and is trained on through the
    public `SAETrainer.train_epoch`.  Rows/s over whole epochs, randperm included."""
    from whisper_sae_b200.data.feature_cache import ResidentBatches

    loader = ResidentBatches(rows, batch, True, dev, drop_last=True, seed=99)
    tr.train_epoch(loader)                      # warm-up epoch (captures the indexed graph)
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(epochs):
        tr.train_epoch(loader)
    end.record()
    torch.cuda.synchronize()
    sec = start.elapsed_time(end) / 1e3
    n = epochs * len(loader) * batch
    return {"value": n / sec, "unit": UNIT, "ms_per_step": 1e3 * sec / (epochs * len(loader)),
            "resident_rows": int(rows.shape[0]), "batches_per_epoch": len(loader), "epochs": epochs,
            "path": "FeatureCache.get_dataloader(device=...) -> ResidentBatches(shuffle=True) -> "
                    "SAETrainer.train_epoch; rows gathered by index inside K0/K23 (no index_select pass)"}


def variants_block(dev: str, rows: int = 16384, steps: int = 20) -> dict:
    """BASELINE.json configs[4]: TopK crosscoder over the 4 whisper-tiny encoder layers and the TopK /
    skip transcoders at 384 -> 3072, k = 32, B = 16384 (SURVEY 8(d) config 5).  The reference has no
    trainer for them (its tests step them by hand: forward, backward, optimizer step, renorm), so a
    step here is exactly that through the public modules under bf16 autocast with torch AdamW."""
    from whisper_sae_b200.sae import (GraphedVariantStep, SkipTranscoder, TopKCrossLayerCrosscoder,
                                      TopKTranscoder, make_optimizer)

    d, F, k, L = 384, 3072, 32, 4
    out = {}

    def timed(model, call, args, flops_per_row):
        opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.0, fused=True)

        def step():
            with torch.amp.autocast("cuda", dtype=torch.bfloat16):
                o = call()
            opt.zero_grad(set_to_none=False)
            o.loss.backward()
            opt.step()
            model.normalize_decoder_weights()
        for _ in range(5):
            step()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            step()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        # the same step captured into one CUDA graph (whisper_sae_b200.sae.GraphedVariantStep)
        stepper = GraphedVariantStep(model, make_optimizer(model))
        for _ in range(5):
            stepper(*args)
        torch.cuda.synchronize()
        a.record()
        for _ in range(steps):
            stepper(*args)
        b.record()
        torch.cuda.synchronize()
        gms = a.elapsed_time(b) / steps
        return {"value": rows / gms * 1e3, "unit": UNIT, "ms_per_step": gms, "batch_rows": rows,
                "gemm_tflops": flops_per_row * rows / gms / 1e9,
                "hand_stepped": {"value": rows / ms * 1e3, "ms_per_step": ms}}

    torch.manual_seed(7)
    acts = {li: synth(rows, d, seed=50 + li).to(dev) for li in range(L)}
    cc = TopKCrossLayerCrosscoder(d, L, F, k=k).to(dev)
    out["topk_crosscoder_4x384_3072"] = timed(cc, lambda: cc(acts), (acts,), 6 * L * d * F)
    del cc
    x, y = acts[0], acts[1]
    tc = TopKTranscoder(d, d, F, k=k).to(dev)
    out["topk_transcoder_384_384_3072"] = timed(tc, lambda: tc(x, y), (x, y), 6 * d * F)
    del tc
    sk = SkipTranscoder(d, d, F, k=k).to(dev)
    out["skip_transcoder_384_384_3072"] = timed(sk, lambda: sk(x, y), (x, y), 6 * d * F + 6 * d * d)
    del sk, acts
    torch.cuda.empty_cache()
    out["note"] = ("forward + backward + torch fused AdamW + decoder renorm through the public modules "
                   "(autograd node on the same K0/K1/K23/K4 kernels), bf16 autocast, device-resident inputs; "
                   "value = the step replayed as one CUDA graph (GraphedVariantStep), hand_stepped = the "
                   "same calls launched eagerly the way the reference's tests step these modules")
    return out


@contextlib.contextmanager
def serial_kernels():
    """The per-kernel profile runs the step WITHOUT the forked graph branches (WSAE_FORK=0): a kernel
    timed while it shares the SMs with a weight-gradient GEMM reads many times its own duration
    (b_pre gradient at 1280 -> 40960: 2.3 ms beside K4, ~0.1 ms alone)."""
    old = os.environ.get("WSAE_FORK")
    os.environ["WSAE_FORK"] = "0"
    try:
        yield
    finally:
        if old is None:
            os.environ.pop("WSAE_FORK", None)
        else:
            os.environ["WSAE_FORK"] = old


def kernel_profile(tr, batches, steps: int) -> dict:
    """Per-kernel CUDA-event spans of the eagerly launched step.  Each step is queued behind a ~3 ms
    device-side spin, so the host has enqueued the whole step (kernels and events) before the first
    kernel starts: the spans hold kernel time only, no host launch gaps (round 1 read K23 as 0.29 ms
    on boxes where the Python host fell behind the GPU, 0.22 ms where it did not)."""
    from whisper_sae_b200 import ops

    spin = int(3e-3 * 1.9e9)
    torch.cuda.synchronize()
    ops.PROFILE = ops.KernelProfile()
    for i in range(steps):
        torch.cuda._sleep(spin)
        tr.train_step(batches[i % len(batches)])
    summ = ops.PROFILE.summary()
    ops.PROFILE = None
    step_ms = sum(v["total_ms"] for v in summ.values()) / steps
    for v in summ.values():
        v["share_of_step"] = v["total_ms"] / (step_ms * steps)
        v["per_step"] = v["launches"] / steps
    summ["_step_ms"] = step_ms
    return summ


# dram__bytes_read.sum + dram__bytes_write.sum and lts__t_sectors.sum x 32 B per launch from `ncu --set
# full` of each workload's default batch (bf16): profiles/r2c_{tiny,small-dp,large-dp}_top3_ncu_full.txt
# (K1 = CTA-pair kernel, K4 averaged over its two launches); K23 = tensor form with the L2 eviction hints:
# profiles/r2d_{tiny,small-dp,large-dp}_k23_ncu_full.txt
NCU_TRAFFIC = {
    "tiny": {"wsae_encode_topk": (74.56e6, 1704.9e6), "wsae_decode_backward": (155.07e6, 2248.7e6),
             "wsae_wgrad_gemm": (88.89e6, 925.6e6)},
    "small-dp": {"wsae_encode_topk": (155.82e6, 6022.0e6), "wsae_decode_backward": (337.65e6, 4410.4e6),
                 "wsae_wgrad_gemm": (289.79e6, 3436.5e6)},
    "large-dp": {"wsae_encode_topk": (334.74e6, 23662.3e6), "wsae_decode_backward": (1421.41e6, 8744.3e6),
                 "wsae_wgrad_gemm": (1094.70e6, 17442.1e6)},
}
NCU_SOURCE = "profiles/r2c_{wl}_top3_ncu_full.txt"


def rooflines(prof: dict, wl_name: str, wl: dict, batch: int, peaks: dict, peak_src: str) -> tuple[dict, dict]:
    """(roofline of the dominant kernel, per-kernel table).  Dominant = largest total time per step.
    Algorithmic work per launch (DESIGN.md §4, SURVEY §8d):
      K1 encode_topk, K4 wgrad_gemm (x2 launches): 2*B*d*F FLOP, tensor bound;
      K23 decode_backward: COMPULSORY HBM bytes B*(d*4 + d*2 + k*12) + F*d*2 (x read, bf16 residual
        write, idx/val/dv, the bf16 decoder once) against HBM; its k*d*2 B/row decoder-row gather is
        served by L2 (the bf16 decoder is L2-resident for d <= 768), reported as `l2` against the
        measured L2 row-gather ceiling;
      elementwise kernels: their HBM bytes."""
    d, F, k = wl["d"], wl["d"] * wl["expansion"], wl["k"]
    kern = {n: v for n, v in prof.items() if not n.startswith("_")}
    l2_ceiling, l2_src = load_l2_ceiling()
    P = 2 * d * F + F + 2 * d
    table = {}
    for name, v in kern.items():
        t = v["avg_ms"] / 1e3
        if t <= 0:
            continue
        ncu = NCU_TRAFFIC.get(wl_name, {}).get(name) if batch == wl["batch"] else None
        e = {"avg_ms": round(v["avg_ms"], 4), "per_step": v["per_step"], "share_of_step": round(v["share_of_step"], 4)}
        if name in ("wsae_encode_topk", "wsae_wgrad_gemm"):
            tf = 2.0 * batch * d * F / t / 1e12
            e.update(bound="tensor", achieved=tf, unit="TFLOP/s", peak=peaks["bf16_tflops_sustained"],
                     frac=tf / peaks["bf16_tflops_sustained"], peak_burst=peaks["bf16_tflops"],
                     frac_burst=tf / peaks["bf16_tflops"])
        else:
            if name == "wsae_decode_backward":
                nbytes = batch * (d * 4 + d * 2 + k * 12) + F * d * 2
                gather = batch * k * d * 2
                e["l2"] = {"gather_bytes": gather, "achieved": gather / t / 1e9, "unit": "GB/s",
                           "peak": l2_ceiling, "frac": (gather / t / 1e9 / l2_ceiling) if l2_ceiling else None,
                           "peak_source": l2_src}
            elif name == "wsae_pack_activations":
                nbytes = batch * d * 4 + batch * ((d + 16 + 63) // 64 * 64) * 2
            elif name == "wsae_pack_encoder":
                nbytes = F * d * 4 + F * ((d + 16 + 63) // 64 * 64) * 2
            elif name == "wsae_cast_bf16":
                nbytes = F * d * 6
            elif name == "wsae_adamw_multi":
                nbytes = 28 * P
            elif name == "wsae_sumsq":
                nbytes = 4 * P
            elif name == "wsae_bucket_by_tile":
                nbytes = batch * k * (12 + 12)
            elif name == "wsae_bpre_grad":
                nbytes = F * d * 4
            else:
                nbytes = 0
            gbs = nbytes / t / 1e9
            e.update(bound="hbm", achieved=gbs, unit="GB/s", peak=peaks["hbm_gbs"], frac=gbs / peaks["hbm_gbs"])
        if ncu is not None:
            e["traffic"] = ncu[0]
            e["lts_bytes"] = ncu[1]
        table[name] = e
    top = max(table, key=lambda n: kern[n]["total_ms"])
    t = table[top]
    roof = {"kernel": top, "bound": t["bound"], "achieved": t["achieved"], "peak": t["peak"], "unit": t["unit"],
            "frac": t["frac"], "traffic": t.get("traffic"), "peak_source": peak_src,
            "launches_per_step": t["per_step"],
            "traffic_source": NCU_SOURCE.format(wl=wl_name) + " (dram bytes per launch)" if "traffic" in t else None}
    if t["bound"] == "tensor":
        roof["frac_burst"] = t["frac_burst"]
        roof["peak_burst"] = t["peak_burst"]
    return roof, table


# ------------------------------------------------------------------------------------ CPU arms
def _reference_modules():
    """The UNMODIFIED reference package installed by baseline/install_ref.sh (None if absent)."""
    if not (REF_DIR / "whisper_sae").exists():
        return None
    if str(REF_DIR) not in sys.path:
        sys.path.insert(0, str(REF_DIR))
    try:
        from whisper_sae.config import ExperimentConfig as RefExperimentConfig
        from whisper_sae.sae.model import create_sae as ref_create_sae
        from whisper_sae.sae.training import SAETrainer as RefSAETrainer
    except Exception:   # noqa: BLE001
        return None
    return RefExperimentConfig, ref_create_sae, RefSAETrainer


def reference_trainer(wl: dict, batch: int, threads: int):
    """Reference `SAETrainer` on the CPU (fp32: it disables AMP off-CUDA, sae/training.py:73-75),
    same YAML hyper-parameters, same seed recipe as the B200 arm."""
    mods = _reference_modules()
    if mods is None:
        return None
    RefExperimentConfig, ref_create_sae, RefSAETrainer = mods
    torch.set_num_threads(threads)
    cfg = RefExperimentConfig.from_yaml(ROOT / "configs" / "tiny_default.yaml")
    cfg.training.batch_size = batch
    cfg.sae.expansion_factor = wl["expansion"]
    cfg.sae.k = wl["k"]
    torch.manual_seed(cfg.training.seed)
    sae = ref_create_sae(cfg.sae, wl["d"])
    tr = RefSAETrainer(sae, cfg.training, device="cpu", run_dir=Path(tempfile.mkdtemp(prefix="wsae_ref_")))
    tr.setup_scheduler(100_000)
    return tr


def cpu_reference_rate(wl: dict, sample_rows: int, seconds_budget: float, threads: int) -> dict | None:
    """rows/s of the reference's own `SAETrainer.train_step` on the host cores, bounded sample."""
    tr = reference_trainer(wl, sample_rows, threads)
    if tr is None:
        return None
    x = synth(sample_rows * 2, wl["d"], seed=1234)
    tr.train_step(x[:sample_rows])                              # warm-up (thread pools, page faults)
    n, t0 = 0, time.perf_counter()
    while True:
        tr.train_step(x[(n % 2) * sample_rows:(n % 2 + 1) * sample_rows])
        n += 1
        el = time.perf_counter() - t0
        if el >= seconds_budget or n >= 200:
            break
    return {"value": sample_rows * n / el, "unit": UNIT, "cores": threads, "kind": "reference",
            "sample": f"{n} steps of the unmodified reference SAETrainer.train_step (baseline/_ref, device='cpu', "
                      f"fp32) on {sample_rows}-row batches ({el:.1f} s), torch {torch.__version__}"}


def cpu_oracle_rate(wl: dict, batch: int, seconds_budget: float, threads: int) -> dict:
    """rows/s of the CPU oracle port (sparse restatement of the reference algorithm, torch CPU fp32)."""
    from oracle import topk_sae_oracle as O

    d, F, k = wl["d"], wl["d"] * wl["expansion"], wl["k"]
    torch.set_num_threads(threads)
    torch.manual_seed(42)
    state = O.init_state(d, F)
    opt = O.AdamWState()
    lrs = O.lr_sequence(1e-4, 100_000, 1000)
    x = O.synthetic_activations(batch * 2, d, seed=1234)
    O.train_step(state, opt, x[:batch], k, lrs[0])          # warm-up (thread pools, page faults)
    n, t0 = 0, time.perf_counter()
    while True:
        O.train_step(state, opt, x[(n % 2) * batch:(n % 2 + 1) * batch], k, lrs[n + 1])
        n += 1
        el = time.perf_counter() - t0
        if el >= seconds_budget or n >= 200:
            break
    return {"value": batch * n / el, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{n} train steps of B={batch} rows ({el:.1f} s), oracle/topk_sae_oracle.py, "
                      f"torch {torch.__version__} CPU fp32"}


def run_reference_arm(args, wl: dict) -> None:
    """`--impl reference`: the reference's own CPU implementation of the path (unmodified
    `whisper_sae.sae.training.SAETrainer.train_step` from baseline/_ref; the oracle port only if that
    install is absent), all host threads, same config / metric / unit, bounded per-step sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    steps, warm = max(1, args.steps), max(0, args.warmup)
    budget = 150.0                                       # seconds of CPU work for warm + steps
    d, k = wl["d"], wl["k"]
    tr = reference_trainer(wl, args.batch, threads)
    kind = "reference" if tr is not None else "port"
    if tr is not None:
        probe_rows = min(args.batch, 4096)
        xp = synth(probe_rows, d, seed=99)
        tr.train_step(xp)
        t0 = time.perf_counter()
        tr.train_step(xp)
        rate = probe_rows / (time.perf_counter() - t0)
        rows = int(min(args.batch, max(1024, rate * budget / (steps + warm)) // 1024 * 1024))
        x = synth(rows * 2, d, seed=1234)

        def one(i):
            tr.train_step(x[(i % 2) * rows:(i % 2 + 1) * rows])
        impl_note = "unmodified reference SAETrainer.train_step (baseline/_ref, device='cpu', fp32, six dense GEMMs)"
    else:
        from oracle import topk_sae_oracle as O
        torch.set_num_threads(threads)
        torch.manual_seed(42)
        state, opt = O.init_state(d, d * wl["expansion"]), O.AdamWState()
        lrs = O.lr_sequence(1e-4, 100_000, 1000)
        rows = min(args.batch, 16384)
        x = O.synthetic_activations(rows * 2, d, seed=1234)

        def one(i):
            O.train_step(state, opt, x[(i % 2) * rows:(i % 2 + 1) * rows], k, lrs[i])
        impl_note = "oracle port (baseline/_ref not installed: run baseline/install_ref.sh)"
    for i in range(warm):
        one(i)
    t0 = time.perf_counter()
    for i in range(steps):
        one(warm + i)
    el = time.perf_counter() - t0
    value = rows * steps / el
    sample = (f"{steps} timed steps on {rows}-row batches (bounded sample of the {args.batch}-row "
              f"workload batch) on {threads} host threads: {impl_note}; units of an N-GPU job run "
              f"sequentially at this rate (scripts/train.py:338-342)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": 1e3 * el / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, wl, max(1, args.gpus)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(args, wl: dict, n_gpus: int) -> dict:
    d, F = wl["d"], wl["d"] * wl["expansion"]
    if wl["dp"] and n_gpus > 1:
        par = f"batch sharded over {n_gpus} GPUs, NCCL all-reduce of the gradient bucket"
    elif n_gpus > 1:
        par = "1 SAE (layer) per GPU, no data-path collective"
    else:
        par = "single GPU"
    return {
        "workload": f"{wl['label']} TopKSAE {d}->{F} k={wl['k']} train step "
                    f"(configs/tiny_default.yaml hyper-parameters; BASELINE.json {wl['cfg']})",
        "batch_rows_per_gpu": args.batch,
        "global_batch_rows": args.batch * n_gpus,
        "parallelism": par,
        "precision_mode": args.precision,
        "l2_policy": f"{args.resident_batches} distinct resident batches cycled "
                     f"({args.resident_batches * args.batch * d * 4 / 2**20:.0f} MiB > 126 MiB L2)",
    }


def side_workload(name: str, batch: int, dev: str, rank: int, world: int, steps_per_block: int, warmup: int,
                  repeats: int,
                  peaks: dict, peak_src: str, dp: bool, global_rows: int | None, profile: bool) -> dict:
    """One entry of the `workloads` block: the same step at another BASELINE config."""
    wl = WORKLOADS[name]
    dist_on = world > 1
    tr, _ = make_trainer(wl, batch, dev, layer_seed=0, data_parallel=dp, global_rows=global_rows)
    nb = 2
    rows = synth(nb * batch, wl["d"], seed=777 + rank)
    batches = [rows[i * batch:(i + 1) * batch].to(dev) for i in range(nb)]
    with ClockSampler(int(dev.split(":")[1])) as clocks:
        blk, launches = time_blocks(step_runner(tr, batches), steps_per_block * repeats, warmup, repeats, dist_on)
    n_ranks = world if dp else 1
    out = {"config": f"{wl['label']} TopKSAE {wl['d']}->{wl['d'] * wl['expansion']} k={wl['k']} "
                     f"(BASELINE.json {wl['cfg']}), {batch} rows per GPU x {n_ranks} GPU(s), bf16",
           "value": batch * n_ranks / blk["median"], "unit": UNIT,
           "ms_per_step": 1e3 * blk["median"],
           "ms_per_step_min_max": [1e3 * blk["min"], 1e3 * blk["max"]],
           "gpu_launches": launches // repeats, "clocks": clocks.summary()}
    tr.release_graphs()      # (captured graphs that hold NCCL kernels must not outlive the communicator)
    del tr
    if profile:
        tr_e, _ = make_trainer(wl, batch, dev, layer_seed=0, cuda_graph="eager")
        with serial_kernels():
            for i in range(3):
                tr_e.train_step(batches[i % nb])
            prof = kernel_profile(tr_e, batches, 6)
        _, table = rooflines(prof, name, wl, batch, peaks, peak_src)
        out["kernels"] = {n: {kk: vv for kk, vv in e.items() if kk not in ("per_step",)} for n, e in table.items()}
        del tr_e
    del batches, rows
    gc.collect()
    torch.cuda.empty_cache()
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1250, help="timed steps of the headline value and the e2e leg")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=25,
                    help="blocks the --steps timed steps are cut into; the median block's time per step "
                         "is reported")
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="tiny")
    ap.add_argument("--batch", type=int, default=None,
                    help="rows per GPU per step (default 75776 = 148 SMs x 128 rows x 4; dp workloads: "
                         "that global batch / N)")
    ap.add_argument("--precision", choices=["bf16", "fp32"], default="bf16")
    ap.add_argument("--resident-batches", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-workloads", action="store_true", help="skip the `workloads` block")
    ap.add_argument("--value-only", action="store_true",
                    help="only the HBM-resident timed leg (used under ncu; prints a reduced line)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", type=Path, default=None, metavar="DIR",
                    help="write the metrics and model state of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs is not None:
        ap.error("--dump-outputs writes the outputs of the B200 path: not with --impl reference")
    args.warmup = max(args.warmup, 3)
    wl = WORKLOADS[args.workload]
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    if args.batch is None:
        # K1 walks the batch in 128-row tiles on 148 persistent CTAs: 148 * 128 * 4 = 75776 rows is
        # exactly four waves (65536 would be 3.46 -> 4 waves with a 14 % idle tail)
        args.batch = wl["batch"] // world_env if wl["dp"] else wl["batch"]

    if args.impl == "reference":
        run_reference_arm(args, wl)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist_on = world > 1
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU fallback for the product path")
    numa = bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    if dist_on:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = f"cuda:{local_rank}"
    d, F, k = wl["d"], wl["d"] * wl["expansion"], wl["k"]

    peaks, peak_src = load_peaks()
    dp = wl["dp"] and dist_on
    bf16 = args.precision == "bf16"
    tr, cfg = make_trainer(wl, args.batch, dev, layer_seed=0 if dp else rank, use_amp=bf16, data_parallel=dp)
    nb = max(2, args.resident_batches)
    rows = synth(nb * args.batch, d, seed=1234 + rank)
    dev_batches = [rows[i * args.batch:(i + 1) * args.batch].to(dev) for i in range(nb)]
    repeats = max(1, args.repeats)

    # ---- value: inputs resident in HBM ----
    with ClockSampler(local_rank) as clocks:
        runner = step_runner(tr, dev_batches)
        blk, launches = time_blocks(runner, args.steps, args.warmup, repeats, dist_on)
    sec = blk["median"]                      # per step
    value = args.batch * world / sec
    if args.dump_outputs is not None:
        tr.consolidate_weights()             # data parallel: gathers every rank's weight rows (collective)
        if rank == 0:
            dump_outputs(args.dump_outputs, runner.last, tr.model)

    if args.value_only:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
                              "steps": args.steps, "warmup": args.warmup,
                              "ms_per_step": 1e3 * sec, "gpu_launches": launches,
                              "note": "value-only leg (not a bench line)"}))
        if dist_on:
            tr.release_graphs()
            del tr
            gc.collect()
            torch.distributed.destroy_process_group()
        return

    # ---- e2e: pinned host batches through SAETrainer.train_epoch (H2D + metrics D2H inside) ----
    host_batches = [rows[i * args.batch:(i + 1) * args.batch].pin_memory() for i in range(nb)]
    # each block is one train_epoch call (its first H2D copy is not overlapped, as in any epoch)
    blk_e, _ = time_blocks(epoch_runner(tr, host_batches), args.steps, args.warmup, repeats, dist_on)
    e2e = args.batch * world / blk_e["median"]
    h2d_bytes = args.batch * d * 4 + 64          # batch + control block
    resident = resident_loader_rate(tr, rows, args.batch, dev) if (rank == 0 and not dp) else None

    line = None
    side: dict = {}
    if rank == 0:
        # per-kernel CUDA-event timing needs eager launches: same kernels, graph replay switched off
        tr_eager, _ = make_trainer(wl, args.batch, dev, layer_seed=rank, use_amp=bf16,
                                   cuda_graph="eager")       # single-rank kernels (no collective)
        with serial_kernels():
            for i in range(3):
                tr_eager.train_step(dev_batches[i % nb])
            prof = kernel_profile(tr_eager, dev_batches, min(args.steps, 10))
        del tr_eager
        roof, table = rooflines(prof, args.workload, wl, args.batch, peaks, peak_src)
        # the launch-bound YAML batch, for the record
        cfg_batch = 128
        tr_small, _ = make_trainer(wl, cfg_batch, dev, layer_seed=rank, use_amp=bf16)
        small_rows = synth(16 * cfg_batch, d, seed=4321 + rank).to(dev)
        small = [small_rows[i * cfg_batch:(i + 1) * cfg_batch].contiguous() for i in range(16)]
        blk_s, _ = time_blocks(step_runner(tr_small, small), 500, 10, 5, False)
        del tr_small
        det_info = None
        if bf16:      # the bit-reproducible accumulation mode, for the record (SAETrainer(deterministic=True))
            tr_det, _ = make_trainer(wl, args.batch, dev, layer_seed=rank, deterministic=True)
            # 5 blocks as long as one headline block
            blk_d, _ = time_blocks(step_runner(tr_det, dev_batches), 5 * max(1, args.steps // repeats), 3, 5, False)
            det_info = {"ms_per_step": 1e3 * blk_d["median"],
                        "value": args.batch / blk_d["median"], "unit": UNIT,
                        "note": "ordered split-K / fixed-point cross-row sums instead of float atomics; "
                                "bit-identical from run to run (tests/test_gpu_fullsize.py)"}
            del tr_det
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sec, "higher_is_better": True,
            "scaling": "strong" if wl["dp"] else "weak", "vs_baseline": None,
            "dtype": "bf16" if bf16 else "f32", "data": "synthetic",
            "config": workload_config(args, wl, world),
            "timing": {"blocks": blk["blocks"], "step_ms_median": 1e3 * sec, "step_ms_min": 1e3 * blk["min"],
                       "step_ms_max": 1e3 * blk["max"],
                       "method": "`steps` steps back to back cut into `blocks` blocks by CUDA events, median "
                                 "block time per step; barrier + synchronize around the run, max over ranks"},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 32,
                    "ms_per_step": 1e3 * blk_e["median"],
                    "ms_per_step_min_max": [1e3 * blk_e["min"], 1e3 * blk_e["max"]],
                    "h2d_gbs_per_gpu": h2d_bytes / blk_e["median"] / 1e9,
                    "host_numa": numa},
            "gpu_launches": launches,
            "clocks": clocks.summary(),
            "roofline": roof,
            "rooflines": {n: {kk: vv for kk, vv in e.items() if kk != "per_step"} for n, e in table.items()},
            "kernel_shares": {n: e["share_of_step"] for n, e in table.items()},
            "kernel_avg_ms": {n: e["avg_ms"] for n, e in table.items()},
            "yaml_batch": {"batch_rows": cfg_batch, "value": cfg_batch / blk_s["median"], "unit": UNIT,
                           "ms_per_step": 1e3 * blk_s["median"]},
            "deterministic_mode": det_info,
            "resident_loader": resident,
        }
    tr.release_graphs()
    del tr, dev_batches, host_batches, rows
    gc.collect()
    torch.cuda.empty_cache()

    # ---- `workloads` block: BASELINE configs[2] / [3] ----
    if args.workload == "tiny" and not args.no_side_workloads:
        s_block = max(3, min(args.steps, 10))
        s_rep = max(3, min(repeats, 7))
        if not dist_on:
            for name, key in (("small-dp", "small"), ("large-dp", "large-v3")):
                side[key] = side_workload(name, WORKLOADS[name]["batch"], dev, rank, world, s_block, 3, s_rep,
                                          peaks, peak_src, dp=False, global_rows=None, profile=True)
        else:
            for name, key in (("small-dp", "small"), ("large-dp", "large-v3")):
                full = WORKLOADS[name]["batch"]
                weak = side_workload(name, full, dev, rank, world, s_block, 3, s_rep, peaks, peak_src,
                                     dp=True, global_rows=full * world, profile=False)
                strong = side_workload(name, full // world, dev, rank, world, s_block, 3, s_rep, peaks,
                                       peak_src, dp=True, global_rows=(full // world) * world, profile=False)
                side[key + "_dp_weak"] = dict(weak, scaling="weak (fixed rows per GPU), batch-sharded, NCCL gradient exchange")
                side[key + "_dp_strong"] = dict(strong, scaling="strong (fixed global batch), batch-sharded, NCCL gradient exchange")
    if line is not None:
        if side:
            line["workloads"] = side
        if args.workload == "tiny" and not args.no_side_workloads and bf16:
            line["variants"] = variants_block(dev)
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            ref = cpu_reference_rate(wl, 8192, args.cpu_seconds, threads)
            port = cpu_oracle_rate(wl, min(args.batch, 16384), max(3.0, args.cpu_seconds / 3), threads)
            if ref is not None:
                line["cpu_baseline"] = ref
                line["cpu_baseline_port"] = port
            else:
                line["cpu_baseline"] = port
    if line is not None:
        print(json.dumps(line), flush=True)
    if dist_on:
        torch.distributed.barrier()
        gc.collect()                 # captured graphs that hold NCCL kernels must be gone before the communicator
        torch.cuda.synchronize()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
