#!/usr/bin/env python
"""Headline benchmark: image-pairs/sec, LightGlue matcher TRAINING step (forward + loss + backward +
gradient all-reduce + Adam) on synthetic N=2048, d=256, 9-layer pairs (BASELINE.json configs[2],
"SuperPoint + LightGlue MegaDepth-shape synthetic pairs"), one process per GPU.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29511 bench.py --gpus 8 --steps 10 --warmup 3
    python bench.py --impl reference ...      # the reference algorithm on the host CPU cores (oracle port)

Prints ONE JSON line on rank 0 (contract: see the task statement / DESIGN.md section "Measurement").
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "image-pairs/sec training SuperPoint+LightGlue N=2048 at 1/2/4/8 B200"
UNIT = "image-pairs/s"
N_KPTS, D_DESC, N_LAYERS, N_HEADS = 2048, 256, 9, 4
# algorithmic attention FLOPs per pair, forward + backward, no recompute counted (SURVEY.md 8d):
# C = 2 N^2 D ; fwd 7C/layer, bwd 14C/layer
ATTN_FLOPS_PER_PAIR = 21 * (2 * N_KPTS * N_KPTS * D_DESC) * N_LAYERS


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "tflops_burst": p["bf16_tflops"], "tflops_sustained": p["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (one `nvidia-smi -lms` process
    started before and stopped after it)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                          str(self.index), "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
            time.sleep(0.15)  # let the first samples arrive before the timed region starts
        except Exception:
            self.proc = None
        self.t0 = time.time()
        return self

    def __exit__(self, *a):
        if self.proc is None:
            return
        time.sleep(0.06)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        self.rows = [[c.strip() for c in line.split(",")] for line in out.strip().splitlines() if line.strip()]

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        reasons = []
        for name, col in (("hw_slowdown", 2), ("hw_thermal_slowdown", 3), ("sw_thermal_slowdown", 4), ("sw_power_cap", 5)):
            if any(len(r) > col and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


def host_threads():
    """Threads the CPU leg may use: affinity mask and cgroup CPU quota (LGB200_CPU_THREADS overrides)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    if os.environ.get("LGB200_CPU_THREADS"):
        n = min(n, int(os.environ["LGB200_CPU_THREADS"]))
    return max(1, n)


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def pin(data):
    if isinstance(data, dict):
        return {k: pin(v) for k, v in data.items()}
    return data.pin_memory() if torch.is_tensor(data) else data


def nbytes(data):
    if isinstance(data, dict):
        return sum(nbytes(v) for v in data.values())
    return data.numel() * data.element_size() if torch.is_tensor(data) else 0


# ------------------------------------------------------------------------------------------------
class CpuArm:
    """The reference's own implementation of the path on the host CPU cores (BASELINE.md section 4): the UNMODIFIED
    reference matcher driven through its real TwoViewPipeline (oracle/reference_runner.py; installed under oracle/_ref
    by the build, `kind: "reference"`), or, when that copy did not travel, the oracle port (`kind: "port"`).
    One step = zero_grad + forward + loss + backward + Adam on `B` pairs of the N=2048 / 9-layer workload, fp32."""

    def __init__(self, B=1, checkpointed=False, threads=None):
        from gluefactory_b200 import synthetic
        from oracle import reference_runner as R

        self.B, self.checkpointed = B, checkpointed
        torch.set_num_threads(threads or host_threads())
        conf = dict(synthetic.DEFAULT_CONF)
        w = synthetic.make_weights(conf, seed=0)
        data = synthetic.make_pairs(B, N_KPTS, seed=1234)
        if R.available():
            self.kind = "reference"
            self.tr = R.ReferenceTrainer(R.build_pipeline(conf, w, "cpu", checkpointed=checkpointed), lr=1e-4)
            batch = R.pipeline_batch(data)
            self.step = lambda: self.tr.step(batch)
        else:
            from oracle import lightglue_oracle as O

            self.kind = "port"
            ww = {k: v.clone().requires_grad_(True) for k, v in w.items()}
            state = {}

            def step():
                _, st = O.train_step_cpu(ww, data, conf, adam_state=state.get("s"))
                state["s"] = st
            self.step = step

    def time_steps(self, steps, warmup):
        for _ in range(warmup):
            self.step()
        t0 = time.time()
        for _ in range(steps):
            self.step()
        return (time.time() - t0) / max(steps, 1)


def pick_threads(budget_s=40.0):
    """The oracle's / reference's N=2048 GEMMs are small: all cores is not always fastest.  Time ONE step at every
    candidate thread count (bounded) and keep the best; the sweep is reported so the choice is visible."""
    cand = sorted({host_threads(), min(host_threads(), 64), min(host_threads(), 32), min(host_threads(), 16)}, reverse=True)
    sweep, t_start = {}, time.time()
    for n in cand:
        arm = CpuArm(B=1, threads=n)
        arm.step()  # warm-up (allocator, thread pool)
        t0 = time.time()
        arm.step()
        sweep[n] = time.time() - t0
        if time.time() - t_start > budget_s:
            break
    best = min(sweep, key=sweep.get)
    return best, {str(k): round(1.0 / v, 4) for k, v in sweep.items()}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores, same metric / unit.
    A 'step' is a bounded sample of the workload (ONE pair of the same N=2048 / 9-layer configuration per step; the
    variants object adds the reference YAML's per-GPU batch of 4 and activation checkpointing)."""
    if rank != 0:
        return
    budget = float(os.environ.get("LGB200_REF_BUDGET_S", "240"))
    t_begin = time.time()
    threads, sweep = pick_threads()
    arm = CpuArm(B=1, checkpointed=False, threads=threads)
    t0 = time.time()
    arm.step()
    t_one = time.time() - t0
    left = lambda: budget - (time.time() - t_begin)  # noqa: E731
    warm = max(0, min(args.warmup - 1, int(0.2 * left() / max(t_one, 1e-3))))
    steps = max(1, min(args.steps, int(0.55 * left() / max(t_one, 1e-3)) - warm))
    dt = arm.time_steps(steps, warm)
    val = 1.0 / dt
    variants = []
    for B, ckpt in ((4, False), (1, True)):
        if left() < (B * t_one) * 3.5 or arm.kind != "reference" and ckpt:
            continue
        v = CpuArm(B=B, checkpointed=ckpt, threads=threads)
        vdt = v.time_steps(2, 1)
        variants.append({"pairs_per_step": B, "checkpointed": ckpt, "value": B / vdt, "steps": 2, "warmup": 1})
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "steps_requested": args.steps, "warmup": warm + 1, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"LightGlue train step N={N_KPTS} d={D_DESC} L={N_LAYERS} (configs[2]); one pair per step",
                   "pairs_per_step": 1, "checkpointed": False, "flash": False, "variants": variants},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": arm.kind,
                         "host_cpus": os.cpu_count(), "cpu_model": cpu_model(), "torch": torch.__version__,
                         "thread_sweep_pairs_per_s": sweep,
                         "sample": f"{steps} train steps of 1 pair (N={N_KPTS}, L={N_LAYERS}, fp32, "
                                   f"{'unmodified reference through TwoViewPipeline' if arm.kind == 'reference' else 'oracle port'})"
                                   f" after {warm + 1} warm-up"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_sample(seconds=25.0):
    """Bounded CPU sample for the default run's `cpu_baseline` object (rank 0, N=1 only)."""
    threads = min(host_threads(), int(os.environ.get("LGB200_CPU_BASELINE_THREADS", "32")))
    arm = CpuArm(B=1, threads=threads)
    t0 = time.time()
    arm.step()
    t_one = time.time() - t0
    steps = max(1, min(4, int(seconds / max(t_one, 1e-3)) - 1))
    dt = arm.time_steps(steps, 0)
    return {"value": 1.0 / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": arm.kind, "host_cpus": os.cpu_count(),
            "cpu_model": cpu_model(),
            "sample": f"{steps} train steps of 1 pair (N={N_KPTS}, L={N_LAYERS}, fp32, "
                      f"{'unmodified reference' if arm.kind == 'reference' else 'oracle port'}) after 1 warm-up; "
                      "`--impl reference` runs the full-thread sweep, batch-4 and checkpointed variants"}


def gpu_eager_baseline(dev, B=4, steps=5, warmup=3):
    """The same-box GPU competitor (BASELINE.md section 4, SURVEY section 0 fact 1): the reference ships no GPU kernels,
    so its PyTorch modules on this B200 (`.cuda()`; fp32 and `--mp bfloat16` autocast) are what the plugin replaces.
    Bounded: B pairs per step (the reference YAML's per-GPU batch), a few steps, rank 0 at N=1 only."""
    from gluefactory_b200 import synthetic
    from oracle import reference_runner as R

    if not R.available():
        return {"unavailable": "reference not installed under oracle/_ref"}
    conf = dict(synthetic.DEFAULT_CONF)
    w = synthetic.make_weights(conf, seed=0)
    batch = synthetic.to_device(R.pipeline_batch(synthetic.make_pairs(B, N_KPTS, seed=1234)), dev)
    out = {"pairs_per_step": B, "steps": steps, "warmup": warmup, "unit": UNIT,
           "what": "unmodified reference matcher through TwoViewPipeline on this GPU, PyTorch eager (train.py loop restated)"}
    for tag, mp_dtype, ckpt in (("fp32", None, False), ("bf16_autocast", torch.bfloat16, False),
                                ("bf16_autocast_checkpointed", torch.bfloat16, True)):
        try:
            tr = R.ReferenceTrainer(R.build_pipeline(conf, w, dev, checkpointed=ckpt), lr=1e-4, mp_dtype=mp_dtype)
            for _ in range(warmup):
                tr.step(batch)
            torch.cuda.synchronize(dev)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(steps):
                tr.step(batch)
            e.record()
            torch.cuda.synchronize(dev)
            out[tag] = B * steps / (s.elapsed_time(e) / 1e3)
            del tr
            torch.cuda.empty_cache()
        except Exception as ex:  # noqa: BLE001 -- a baseline must never take the bench down
            out[tag] = None
            out[tag + "_error"] = str(ex)[:200]
    return out


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=int(os.environ.get("LGB200_BENCH_BATCH", "32")), help="pairs per GPU per step")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--kpts", type=int, default=2048, help="keypoints per image: 2048 = BASELINE configs[2] (the headline), "
                    "1024 = configs[1] (recorded under profiles/, not the driver's line)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-timing", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from the host instead of replaying "
                    "one CUDA graph of the whole training step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step computed "
                    "(loss, per-pair loss terms, updated parameters) as DIR/<name>.npy, so that two builds can be compared")
    args = ap.parse_args()

    global N_KPTS, ATTN_FLOPS_PER_PAIR
    N_KPTS = args.kpts
    ATTN_FLOPS_PER_PAIR = 21 * (2 * N_KPTS * N_KPTS * D_DESC) * N_LAYERS
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"

    import torch.distributed as dist

    from gluefactory_b200 import _lib, synthetic
    from gluefactory_b200.matchers.lightglue import LightGlue
    from gluefactory_b200.trainer import MatcherTrainer

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    conf = dict(synthetic.DEFAULT_CONF, precision=args.precision)
    model = LightGlue(conf)
    model.load_state_dict(synthetic.make_weights(conf, seed=0), strict=False)
    model = model.to(dev)
    # labels are generated on the device inside every step (gt.cu, the reference's ground_truth component): a batch
    # is keypoints + descriptors + image sizes + the homography, nothing N x N crosses PCIe
    from gluefactory_b200.matchers.homography_matcher import HomographyMatcher

    trainer = MatcherTrainer(model, lr=1e-4, ground_truth=HomographyMatcher({"th_positive": 3.0, "th_negative": 3.0, "transposed_assignment": True}))

    B = args.batch
    pool = [pin(synthetic.make_pairs(B, N_KPTS, seed=1234 + 1000 * rank + i, with_gt=False)) for i in range(2)]
    pool_dev = [synthetic.to_device(p, dev) for p in pool]
    h2d = nbytes(pool[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            fn(i)
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    use_graph = not args.no_graph
    l0 = _lib.launch_count
    trainer.step(pool_dev[0])  # also the per-step kernel count (the graph replays exactly these launches)
    launches_per_step = _lib.launch_count - l0
    if use_graph:
        trainer.capture(pool_dev[0], dev, warmup=2)

    last = []  # (loss, losses) of the latest resident step

    def step_resident(i):
        if use_graph:
            last[:] = trainer.step_graphed(pool_dev[i % len(pool_dev)])  # device-to-device copy into the static inputs + replay
        else:
            loss, losses = trainer.step(pool_dev[i % len(pool_dev)])
            # detached: holding the loss terms must not keep the step's autograd graph alive into the next step
            last[:] = loss, {k: v.detach() if torch.is_tensor(v) else v for k, v in losses.items()}

    host_loss = []

    def step_e2e(i):
        if use_graph:
            # H2D of this step's inputs from pinned memory: queued one step ahead on a copy stream (prefetch=), so the
            # transfer of batch i+1 overlaps the compute of batch i; every step still moves its own h2d bytes
            loss, _ = trainer.step_graphed(pool[i % len(pool)], prefetch=pool[(i + 1) % len(pool)])
        else:
            loss, _ = trainer.step(pool[i % len(pool)], device=dev)
        host_loss.append(loss.item())                             # D2H read of the step's result

    for i in range(args.warmup):
        step_resident(i)
    with ClockSampler(local) as clk:
        ms = timed(step_resident, args.steps)
        launches = launches_per_step * args.steps
    clocks = clk.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last, model)
    # dominant kernel, timed live with CUDA events on the launching stream (second pass, so the
    # event records do not perturb the headline number)
    roof = None
    if not args.no_kernel_timing:
        roof = kernel_roofline(trainer, pool_dev, B, dev)
    for i in range(2):
        step_e2e(i)
    ms_e2e = timed(step_e2e, args.steps)

    pairs = B * world * args.steps
    value = pairs / (ms / 1e3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": f"LightGlue matcher train step, N=M={N_KPTS} keypoints, d={D_DESC}, L={N_LAYERS}, H={N_HEADS} "
                               f"(BASELINE.json configs[{2 if N_KPTS == 2048 else 1}]); device GT labels+forward+loss+backward+"
                               "all-reduce+Adam",
                   "pairs_per_gpu_per_step": B, "global_batch": B * world, "parallelism": f"dp{world}",
                   "launch": "cuda-graph replay of the whole step" if use_graph else "eager (host launches)",
                   "l2": "per-step working set (activations + N x N similarities, >1 GB) exceeds the 126 MB L2; inputs rotate",
                   "attention_roofline_frac": value / world * ATTN_FLOPS_PER_PAIR / (measured_peaks()["tflops_sustained"] * 1e12)},
        "clocks": clocks,
        "e2e": {"value": pairs / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
    }
    if roof is not None:
        line["roofline"] = roof
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        del trainer, pool_dev
        torch.cuda.empty_cache()
        line["gpu_eager_baseline"] = gpu_eager_baseline(dev)
        line["cpu_baseline"] = cpu_baseline_sample()
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tear down without destroy_process_group(): with NCCL work captured inside a live CUDA graph the
        # communicator teardown was observed to hang on this stack.  Drop the graph, sync, barrier, hard-exit.
        trainer._graph = None
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


def dump_outputs(out_dir, loss, losses, model):
    """What a caller of the timed training step receives from its last call: the mean loss, every per-pair loss term and
    the parameters the optimiser step updated in place (all of them: 47.4 MB in float32 at d=256, L=9).  The inputs are
    seeded, so the same arguments give the same files up to floating-point reordering."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss}
    arrays.update({f"losses.{k}": v for k, v in losses.items() if torch.is_tensor(v)})
    arrays.update({f"param.{k}": p for k, p in model.named_parameters()})
    for name, t in arrays.items():
        t = t.detach().cpu()
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy() if t.dtype == torch.float64 else t.float().numpy())


def kernel_roofline(trainer, pool_dev, B, dev):
    """Device time of the attention kernels, measured live with CUDA events around every launch of the C-ABI entry
    points inside two extra eager steps, against their ALGORITHMIC FLOPs (SURVEY 8d, no recompute counted):
    with C = 2 N^2 D per pair, one launch covers the 2B sequences of the batch and
        forward : self 4C (2 images x {QK^T, PV}), cross 3C (S shared by the two directions; executed as 4C)
        backward: self 8C, cross 6C.
    The top-level object is the dominant group (attention backward, self and cross launches averaged with their own
    FLOP counts); `kernels` lists forward / backward, self / cross separately."""
    from gluefactory_b200 import _lib

    names = {"lgb200_attn_fwd", "lgb200_attn_bwd"}
    _lib.timed_events.clear()
    _lib.timed_entry = names
    # kv_shift (> 0 for the cross-attention launches) is argument 9 of attn_fwd and 14 of attn_bwd (include/lgb200.h)
    _lib.timed_tagger = lambda name, a: "cross" if (a[9] if name == "lgb200_attn_fwd" else a[14]) else "self"
    for i in range(2):
        trainer.step(pool_dev[i % len(pool_dev)])
    torch.cuda.synchronize()
    _lib.timed_entry, _lib.timed_tagger = None, None
    groups = {}
    for s, e, tag in _lib.timed_events:
        groups.setdefault(tag, []).append(s.elapsed_time(e))
    _lib.timed_events.clear()
    if not groups:
        return None
    peaks = measured_peaks()
    C = 2 * N_KPTS * N_KPTS * D_DESC * B  # one all-heads contraction for every pair of the batch
    alg = {("lgb200_attn_fwd", "self"): 4 * C, ("lgb200_attn_fwd", "cross"): 3 * C,
           ("lgb200_attn_bwd", "self"): 8 * C, ("lgb200_attn_bwd", "cross"): 6 * C}
    traffic = {}
    tpath = os.path.join(ROOT, "profiles", "r02_roofline_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        # only quote a capture taken at this run's batch size and keypoint count
        if tj.get("sequences_per_launch") == 2 * B and tj.get("keypoints", 2048) == N_KPTS:
            traffic = tj.get("dram_bytes_per_launch", {})
    kernels = {}
    for (name, kind), ts in sorted(groups.items()):
        avg_ms = sum(ts) / len(ts)
        ach = alg[(name, kind)] / (avg_ms * 1e-3) / 1e12
        kernels[f"{name[7:]}_{kind}"] = {"avg_launch_ms": avg_ms, "launches_timed": len(ts), "achieved": ach,
                                         "frac": ach / peaks["tflops_sustained"], "algorithmic_gflop": alg[(name, kind)] / 1e9}
    bw = [(k, v) for k, v in kernels.items() if k.startswith("attn_bwd")]
    flops = sum(v["algorithmic_gflop"] * v["launches_timed"] for _, v in bw) * 1e9
    secs = sum(v["avg_launch_ms"] * v["launches_timed"] for _, v in bw) * 1e-3
    n = sum(v["launches_timed"] for _, v in bw)
    achieved = flops / secs / 1e12
    return {"kernel": "lgb200_attn_bwd (attn_bwd_prep_fused + attn_bwd_fused + dq_convert; self 8C and cross 6C launches)",
            "bound": "tensor", "achieved": achieved, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
            "frac": achieved / peaks["tflops_sustained"], "traffic": traffic.get("lgb200_attn_bwd"),
            "traffic_source": "profiles/r02_roofline_traffic.json (ncu --set full of this command at this batch size)" if traffic else None,
            "avg_launch_ms": secs / n * 1e3, "launches_timed": n, "kernels": kernels,
            "peak_source": peaks["source"] + ", sustained (kernel timed inside a long step)"}


if __name__ == "__main__":
    main()
