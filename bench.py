#!/usr/bin/env python
"""bench.py -- the UnFlow hot path on N B200s (one process per GPU).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the reference
    python bench.py ... --dump-outputs DIR                     # also write the last timed step's outputs

Workload ("step" = one pass of the hot path over one batch of synthetic input): the full
unsupervised FlowNetC training step of BASELINE.json configs[2]/[3] -- bidirectional FlowNetC
forward (correlation d=20), 5-level census / fb-occlusion / 2nd-order-smoothness loss, backward,
gradient all-reduce (N>1) and Adam update -- on 4 synthetic KITTI-shaped 384x1280 pairs PER GPU
(weak scaling: global batch 4*N; configs[3] is N=8 -> batch 32).  configs[1] (forward only) is a
subset of this step and is covered by the parity tests.

One JSON line on rank 0:
  value   frame-pairs/s, whole job, inputs already resident in HBM when the timed region starts
  e2e     the same metric through the public API (e2eflow ... Trainer.step) with the inputs in
          pinned HOST memory: H2D copy of both frames and D2H read of the loss inside every step
  roofline  correlation forward kernel: algorithmic bytes / CUDA-event time measured live inside
          the timed region, against the measured HBM peak (MEASURED_PEAKS.json); extra fields give
          the fp32-FMA fraction and the same figures for the other hand-written kernels
  cpu_baseline  (N=1) the CPU oracle (a restatement of the reference -- the reference itself has
          no CPU path for this graph, SURVEY.md R1) on a bounded sample, timed on the host cores
  clocks  nvidia-smi SM clock / throttle reasons sampled (every 100 ms) during the timed region
Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.
--steps K sets the steps of every timed region: the headline and e2e regions run exactly K, the
per-kernel eager pass (graph mode) and the fp32 pass at most K.
--dump-outputs DIR: after the headline region, rank 0 writes what its last step returned to the
caller as DIR/<name>.npy (float32): ``loss`` and, at the same DUMP_SAMPLE seeded flat positions, the
updated trained variables (``params``) and Adam moments (``adam_m``, ``adam_v``).  Inputs and
initial weights are seeded, so two builds run with the same arguments can be compared output for output.
L2: one step streams several GB of activations (>> 126 MB L2), so no explicit flush is needed.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from unflow_b200 import synthetic as synth  # noqa: E402

H, W, PER_GPU_BATCH = 384, 1280, 4
DUMP_SAMPLE = 1 << 21        # per array: 3 x 8 MB for FlowNetC's 39.2 M trained floats
METRIC = "frame-pairs/s at 384x1280 FlowNetC"


def load_peaks():
    peaks = {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "_source": "fallback (B200_PROFILING.md)"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peaks.update(json.load(fh))
            peaks["_source"] = "measured (MEASURED_PEAKS.json)"
    except Exception:
        pass
    return peaks


class ClockSampler:
    """nvidia-smi clocks / throttle reasons.  ONE nvidia-smi process per bench run, started before the warm-up
    and sampling every 100 ms; every line is stamped with the host time it arrived at, and a timed region
    (bracketed by synchronisations) picks the samples that fall inside it.  (A sampler started at the beginning
    of a 0.28 s region often delivered its first line after the region had ended: "samples": 0.)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []          # (arrival time, line)

    def start(self):
        if self.proc is not None:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def close(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            self.proc = None

    def window(self, t0, t1):
        """Statistics of the samples that arrived in [t0, t1]; if there are none (a very short region), of
        the samples within 0.3 s around it -- flagged "around_region" (they see the warm-up replays of the same
        step that precede the region and the legs that follow it)."""
        if self.proc is None and not self.lines:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)         # let the sample that covers the end of the region arrive
        pick = [ln for (t, ln) in self.lines if t0 <= t <= t1 + 0.1]
        widened = False
        if not pick:
            pick = [ln for (t, ln) in self.lines if t0 - 0.3 <= t <= t1 + 0.3]
            widened = True
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in pick:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        out = {"sm_mhz": statistics.median(sm) if sm else None,
               "sm_max_mhz": max(smax) if smax else None, "samples": len(sm),
               "reasons": sorted(reasons)}
        if widened:
            out["around_region"] = True
        return out


def make_batch(rank, pinned):
    im1, im2, _ = synth.image_pair(PER_GPU_BATCH, H, W, seed=1234 + rank)
    if pinned:
        im1, im2 = im1.pin_memory(), im2.pin_memory()
    return im1, im2


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def dump_outputs(out_dir, trainer, loss):
    """The outputs of the step that just ran (see the module docstring); host copies."""
    n = trainer.num_params
    g = torch.Generator().manual_seed(0)
    idx = torch.randperm(n, generator=g)[:min(n, DUMP_SAMPLE)].sort().values.to(trainer.device)
    arrays = {"loss": loss.detach().float().reshape(1)}
    for name, flat in (("params", trainer.flat_param), ("adam_m", trainer.adam_m), ("adam_v", trainer.adam_v)):
        arrays[name] = flat[idx]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy().astype(np.float32))


def run_ours(args):
    from unflow_b200 import _native
    from unflow_b200.e2eflow import ops
    from unflow_b200.e2eflow.core.train import Trainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d" % args.gpus)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        # keep stdout to the single JSON line: NCCL's own banner ("NCCL version ...") goes to a file
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/unflow_nccl.%h.%p.log")
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=300))
    _native.lib()  # fail loudly if libunflow.so is missing
    from unflow_b200.e2eflow.core import conv_ops
    conv_ops.set_mode(args.conv)
    torch.backends.cudnn.benchmark = bool(args.cudnn_benchmark)

    global PER_GPU_BATCH
    PER_GPU_BATCH = args.batch
    params = dict(synth.KITTI_PARAMS, learning_rate=1.0e-5, flownet=args.spec)
    trainer = Trainer(params, synth.KITTI_NORMALIZATION, dev, seed=1234)
    trainer.broadcast_variables(0)
    h_im1, h_im2 = make_batch(rank, pinned=True)
    d_im1, d_im2 = h_im1.to(dev), h_im2.to(dev)
    loss_host = torch.zeros((), dtype=torch.float32).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def resident_step():
        last["loss"] = trainer.step(d_im1, d_im2)
        return last["loss"]

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()          # runs for the whole bench; timed regions pick their samples by time

    def timed(fn, steps, hook=False):
        barrier()
        _native.reset_launch_count()
        if hook:
            ops.kernel_timer.enable()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        start.record()
        for _ in range(steps):
            fn()
        end.record()
        barrier()
        t1 = time.time()
        launches = _native.launch_count()
        ktimes = ops.kernel_timer.collect() if hook else {}
        clocks = sampler.window(t0, t1) if rank == 0 else None
        ms = torch.tensor([start.elapsed_time(end)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), launches, ktimes, clocks

    for _ in range(args.warmup):
        resident_step()
    # eager pass: per-kernel CUDA-event timings for the roofline objects (and the value itself when
    # graphs are off)
    eager_steps = args.steps if not args.graph else min(args.steps, 5)
    ms, launches, ktimes, clocks = timed(resident_step, eager_steps, hook=True)
    kbytes = dict(ops.kernel_timer.bytes)
    steps_timed = eager_steps
    steps_timed_eager = eager_steps
    if args.graph:
        trainer.capture(d_im1, d_im2)
        for _ in range(2):
            resident_step()
        ms, _, _, clocks = timed(resident_step, args.steps)
        launches = trainer._graph_launches * args.steps
        steps_timed = args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, trainer, last["loss"])

    def e2e_step():   # host batch -> (static) device buffers, step, loss back to the host
        if args.graph:
            loss = trainer.step(h_im1, h_im2)
        else:
            loss = trainer.step(h_im1.to(dev, non_blocking=True), h_im2.to(dev, non_blocking=True))
        loss_host.copy_(loss, non_blocking=True)
        return loss

    if args.prefetch and args.graph:
        # opt-in: the copy of step i+1's batch overlaps step i (still inside the timed region, still
        # one H2D of both frames and one D2H of the loss per step)
        def e2e_step():   # noqa: F811
            loss = trainer.step_prefetched()
            trainer.prefetch(h_im1, h_im2)
            loss_host.copy_(loss, non_blocking=True)
            return loss
        trainer.prefetch(h_im1, h_im2)
    for _ in range(min(args.warmup, 2)):
        e2e_step()
    ms_e2e, _, _, _ = timed(e2e_step, args.steps)
    torch.cuda.synchronize()
    final_loss = float(loss_host.item())
    fp32_exact = None
    if args.also_fp32 and args.conv != "fp32" and world == 1:
        conv_ops.set_mode("fp32")
        saved_graph, trainer._graph = trainer._graph, None     # eager: the captured graph is the 3xTF32 step
        for _ in range(3):
            resident_step()
        steps32 = max(1, args.steps // 2)
        ms32, _, _, _ = timed(resident_step, steps32)
        trainer._graph = saved_graph
        fp32_exact = {"ms_per_step": round(ms32 / steps32, 3),
                      "value": round(PER_GPU_BATCH * world / (ms32 / steps32 * 1e-3), 3),
                      "unit": "frame-pairs/s", "conv_precision": "fp32 (cuDNN, no tensor cores)"}
        conv_ops.set_mode(args.conv)

    sampler.close()
    params_in_sync = None
    if world > 1:
        # every rank must hold bit-identical variables after the timed steps (same all-reduced
        # gradient, same Adam update): min == max over ranks of an order-independent integer checksum
        chk = trainer.flat_param.view(torch.int32).to(torch.int64).sum().reshape(1)
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        params_in_sync = bool(int(lo.item()) == int(hi.item()))
    if rank != 0:
        _finish(world)
        return
    peaks = load_peaks()
    pairs = PER_GPU_BATCH * world * args.steps
    value = PER_GPU_BATCH * world * steps_timed / (ms * 1e-3)
    e2e = pairs / (ms_e2e * 1e-3)
    fma_peak = 148 * 128 * 2 * peaks["sm_max_mhz"] * 1e6 / 1e12

    def roof(name, nbytes=None, flops=None):
        t = ktimes.get(name)
        if not t:
            return None
        if nbytes is None:   # spans that declared their bytes: average over all launches
            nbytes = kbytes.get(name, 0) / len(t)
        avg = sum(t) / len(t) * 1e-3
        r = {"kernel": name, "bound": "hbm", "launches_timed": len(t), "avg_us": round(avg * 1e6, 2),
             "achieved": round(nbytes / avg / 1e9, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
             "frac": round(nbytes / avg / 1e9 / peaks["hbm_gbs"], 4), "peak_source": peaks["_source"],
             "algorithmic_bytes": nbytes, "traffic": TRAFFIC.get(name)}
        if flops:
            r["fp32_tflops"] = round(flops / avg / 1e12, 2)
            r["fma_frac"] = round(flops / avg / 1e12 / fma_peak, 4)
        return r

    Bc, C, hc, wc, D2 = PER_GPU_BATCH, 256, H // 8, W // 8, 441
    corr_bytes = 4 * Bc * hc * wc * (2 * C + D2)
    corr_flops = 2 * Bc * hc * wc * C * D2
    npx0 = PER_GPU_BATCH * (H // 4) * (W // 4)
    # tensor-core conv kernels: nominal flops (2 x multiply-adds of the fp32 convolution) are executed as
    # three TF32 MMA passes (hi*hi + hi*lo + lo*hi); the tensor roofline is the measured sustained bf16
    # GEMM rate / 2 (TF32 has half the bf16 MMA rate)
    tf32_peak = peaks.get("bf16_tflops_sustained", 1442.1) / 2.0

    def tensor_roof(name, label):
        t = ktimes.get(name)
        if not t:
            return None
        total_ms = sum(t)
        flops = kbytes.get(name, 0)                      # the spans declare nominal flops in the bytes slot
        nominal = flops / (total_ms * 1e-3) / 1e12
        return {"kernel": label, "bound": "tensor", "launches_timed": len(t),
                "avg_us": round(total_ms / len(t) * 1e3, 2), "achieved": round(3 * nominal, 1),
                "peak": round(tf32_peak, 1), "unit": "TFLOP/s", "frac": round(3 * nominal / tf32_peak, 4),
                "peak_source": peaks["_source"] + ": bf16_tflops_sustained / 2 (TF32)",
                "nominal_fp32_tflops": round(nominal, 1), "mma_passes_per_product": 3,
                "algorithmic_flops": int(flops // max(len(t), 1)), "traffic": TRAFFIC.get(name),
                "ms_per_step": round(total_ms / max(steps_timed_eager, 1), 3)}

    roofs = [tensor_roof("tc_conv", "tc_conv_kernel (tcgen05 3xTF32 conv / deconv forward + input gradient, all launches)"),
             tensor_roof("tc_wgrad", "tc_wgrad_kernel (tcgen05 3xTF32 weight gradient, all launches)"),
             # one-pass bidirectional correlation: inputs read once, both volumes written (+ the zero fill of the
             # reverse volume); flops = the ONE set of products both volumes share
             roof("correlation_fwd_bidir", 4 * Bc * hc * wc * (2 * C + 3 * D2), corr_flops),
             # gradient fold (read 2 volumes, write 1) + the two gradient launches on the folded volume
             roof("correlation_bwd_bidir", 4 * Bc * hc * wc * (3 * D2 + D2 + 4 * C), 2 * corr_flops),
             roof("correlation_fwd", corr_bytes, corr_flops),
             roof("correlation_bwd", 4 * Bc * hc * wc * (D2 + 4 * C), 2 * corr_flops),
             roof("level_loss_fwd_%dx%d" % (H // 4, W // 4), (44 + 16) * npx0),
             roof("level_loss_bwd_%dx%d" % (H // 4, W // 4), (60 + 16) * npx0),
             roof("conv_operand"), roof("narrow_conv_fwd"), roof("narrow_conv_wgrad"), roof("adam")]
    roofs = [r for r in roofs if r]
    line = {
        "metric": METRIC, "value": round(value, 3), "unit": "frame-pairs/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / steps_timed, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (seeded smooth images + smooth <=8px flow + noise; random-init weights)",
        "config": {"workload": ("BASELINE configs[2]/[3]: FlowNetC full unsupervised training step "
                                "(bidir forward, corr d=20, 5-level census/fb/2nd-order loss, backward, "
                                "grad all-reduce, Adam), 384x1280, batch 4 per GPU") if (args.spec == "C" and args.batch == 4)
                   else ("BASELINE configs[4] geometry: stacked %s unsupervised training step (forward of every "
                         "network + loss; backward / Adam of the last network, config.ini:55-58), 384x1280, batch %d per GPU"
                         % (args.spec, args.batch)),
                   "flownet": args.spec,
                   "global_batch": PER_GPU_BATCH * world, "parallelism": "dp%d" % world,
                   "l2": "inputs+activations per step >> 126 MB L2 (no flush needed)",
                   "conv_precision": ("fp32 (cuDNN, TF32 disabled)" if args.conv == "fp32" else
                                      "3xTF32 split on tensor cores, hand-written tcgen05 kernels with fp32 register "
                                      "accumulation (2e-6 vs float64 per layer, parity-tested)"),
                   "cudnn_benchmark": bool(args.cudnn_benchmark),
                   "cuda_graph": bool(args.graph)},
        "e2e": {"value": round(e2e, 3), "unit": "frame-pairs/s", "ms_per_step": round(ms_e2e / args.steps, 3),
                "h2d_bytes_per_step": 2 * h_im1.numel() * 4, "d2h_bytes_per_step": 4},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "final_loss": final_loss,
    }
    if fp32_exact:
        line["fp32_exact"] = fp32_exact
    if params_in_sync is not None:
        line["params_in_sync"] = params_in_sync
    if roofs:
        line["roofline"] = roofs[0]
        line["rooflines_other"] = roofs[1:]
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(steps=1, warmup=0)
    print(json.dumps(line), flush=True)
    _finish(world)


def _finish(world):
    """Leave without ncclCommDestroy: destroy_process_group() was observed to hang for minutes after
    the timed work was done (communicators that were used inside a captured CUDA graph), which would
    burn the GPU lease; all results are already printed and flushed."""
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


# measured once with `ncu --set full` (profiles/): dram__bytes_read.sum + dram__bytes_write.sum per launch
TRAFFIC = {}
try:
    with open(os.path.join(ROOT, "profiles", "dram_traffic.json")) as _fh:
        TRAFFIC = json.load(_fh)
except Exception:
    pass


# ---------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle (CPU restatement of the reference) on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_step_fn():
    from oracle import flownet as ofl, unsupervised as oun, ops as oops
    # all the host threads this process can really use (affinity / cgroup quota aware; capped:
    # the conv sizes of one image pair stop scaling beyond a few dozen threads)
    if os.environ.get("UNFLOW_CPU_THREADS"):
        oops.set_num_threads(int(os.environ["UNFLOW_CPU_THREADS"]))
    else:
        oops.calibrate_threads()
    tfv = ofl.init_variables('C', False, seed=1234)
    for k in tfv:
        tfv[k].requires_grad_(True)
    im1, im2, _ = synth.image_pair(1, H, W, seed=1234)

    def step():
        for v in tfv.values():
            v.grad = None
        loss = oun.unsupervised_loss(tfv, (im1, im2), synth.KITTI_PARAMS, synth.KITTI_NORMALIZATION,
                                     augment=False)
        loss.backward()
        return float(loss.detach())

    return step, oops.num_threads()


def cpu_baseline(steps=1, warmup=0):
    step, nthreads = cpu_step_fn()
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": round(1.0 / dt, 4), "unit": "frame-pairs/s", "cores": int(nthreads), "host_cpus": int(os.cpu_count() or 1),
            "kind": "port",
            "sample": "%d step(s) of 1 pair 384x1280: FlowNetC fwd + 5-level loss + backward "
                      "(no optimiser), CPU restatement of the reference in oracle/ (the reference "
                      "has no CPU kernels for this graph)" % steps,
            "seconds_per_pair": round(dt, 3)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    step, nthreads = cpu_step_fn()
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    total = time.perf_counter() - t0
    value = args.steps / total
    cb = {"value": round(value, 4), "unit": "frame-pairs/s", "cores": int(nthreads), "host_cpus": int(os.cpu_count() or 1), "kind": "port",
          "sample": "each step = 1 pair 384x1280 (FlowNetC fwd + 5-level loss + backward) on the host "
                    "cores; CPU restatement of the reference (oracle/), the reference itself has no "
                    "CPU path (SURVEY.md R1)"}
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 4), "unit": "frame-pairs/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(total / args.steps * 1e3, 2), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "BASELINE configs[2]/[3] step graph, bounded sample: 1 pair per step "
                                   "on the host CPU", "global_batch": 1, "parallelism": "cpu"},
            "cpu_baseline": cb,
            "e2e": {"value": round(value, 4), "unit": "frame-pairs/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def _watchdog():
    """A hung collective must not burn the GPU lease: dump every thread's Python stack and exit."""
    import faulthandler
    secs = int(os.environ.get("UNFLOW_BENCH_WATCHDOG", "900"))
    if secs > 0:
        faulthandler.dump_traceback_later(secs, exit=True)


def main():
    _watchdog()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy "
                         "(this repo's CUDA path only)")
    ap.add_argument("--prefetch", type=int, default=0,
                    help="1: overlap the host->device copy of the next batch with the running step in the "
                         "e2e loop (Trainer.prefetch / step_prefetched; opt-in, not yet measured)")
    ap.add_argument("--conv", default=os.environ.get("UNFLOW_CONV_PRECISION", "3xtf32"),
                    choices=["fp32", "3xtf32"],
                    help="arithmetic of the conv stacks: 3xtf32 = tensor cores at fp32-level accuracy "
                         "(parity-tested at the same 1e-4 flow tolerance), fp32 = plain cuDNN float32")
    ap.add_argument("--cudnn-benchmark", type=int, default=int(os.environ.get("UNFLOW_CUDNN_BENCHMARK", "1")),
                    help="1: let cuDNN autotune its algorithm per conv shape during warm-up")
    ap.add_argument("--graph", type=int, default=int(os.environ.get("UNFLOW_CUDA_GRAPH", "1")),
                    help="1: replay the whole training step as one CUDA graph (value and e2e); the "
                         "per-kernel roofline timings always come from an eager pass")
    ap.add_argument("--spec", default="C", help="network stack (reference `flownet` parameter): C (headline), CSS = BASELINE configs[4]")
    ap.add_argument("--batch", type=int, default=4, help="image pairs per GPU (4 = BASELINE configs[2]/[3]; configs[4] uses 2)")
    ap.add_argument("--also-fp32", type=int, nargs="?", const=1, default=1,
                    help="1 (default, N=1 only): additionally time the exact-fp32 conv mode (no tensor "
                         "cores) for a few steps and report it as fp32_exact next to the 3xTF32 headline")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_ours(args)


if __name__ == "__main__":
    main()
