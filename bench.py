#!/usr/bin/env python
"""bench.py -- image-pairs/sec of the DeMoN two-view inference path at 256x192 (BASELINE.json `metric`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config b64|b1|refine1024] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the full pipeline (bootstrap + 3 x iterative + refinement, examples/example.py:87-99)
over one batch of 64 synthetic pairs per GPU: BASELINE.json configs[2] at N=1, configs[3] (512 pairs over 8
GPUs) at N=8 -- weak scaling, pairs are independent, the only collective is ONE NCCL all-gather (one call) of the final
depth / motion tensors, inside the timed region and inside the CUDA graph of the step.
--config b1 = configs[1] (one pair per step: latency); --config refine1024 = configs[4] (RefinementNet at 1024x768,
batch 8; a step = one RefinementNet.eval).  The default is the headline workload; the other two are recorded under profiles/.

One JSON line on stdout (rank 0):
  value        pairs/s, inputs resident in HBM, whole job; `--inflight` (default 2) batches per GPU are in flight on their
               own streams and pipelines (every step is still one full batch through the whole path)
  e2e          the same metric end to end from pinned HOST buffers: N=1 through the C-ABI host entry
               (demon_pipeline_forward_host_async: H2D, pipeline, D2H); N>1 H2D of the rank's inputs, pipeline, the
               all-gather, D2H of the gathered result on rank 0 (of the own shard on the other ranks)
  roofline     the dominant kernel timed with CUDA events around its launches on the launching stream in a second,
               single-stream timed region; peak = a TF32 GEMM measured on this GPU in this run
  cpu_baseline the CPU oracle (torch-CPU fp32 + C geometry ops) on a bounded sample, host cores stated
  check        after the timed regions: demon_check_errors() (a timed-out tcgen05 pipeline wait would have produced
               garbage) and one sample of the LAST timed step against the CPU oracle (inverse-depth L1-rel)
`--impl reference` times that CPU path alone with the same --steps / --warmup, 8 pairs per step (TensorFlow 1.4 cannot
be installed here, DESIGN.md section 5).

`--dump-outputs DIR` writes what the timed path returned in the last step of the timed region behind `value` as
DIR/<name>.npy, one file per key of its result dict (the pipeline: predict_depth0, predict_rotation,
predict_translation of the whole global batch in batch order, written by rank 0).  Inputs and weights are seeded, so two
builds run with the same arguments can be compared output for output.  Above DUMP_LIMIT_BYTES in all, the same fixed,
seeded sample of batch entries is written for every output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

PER_GPU_BATCH = 64
ITERATIONS = 3
METRIC = "image_pairs_per_sec_256x192"
N_INPUT_SETS = 4     # rotating input batches: 4 x 75.5 MB > 126 MB L2 (plus a ~2.7 GB activation workspace per step)
REF_PAIRS_PER_STEP = 8
DUMP_LIMIT_BYTES = 60 * 10 ** 6     # --dump-outputs: at most 64 MB in all, .npy headers included
# conv1 / conv2 of netFlow2 and netDM2 depend only on the image pair: the pipeline runs them once per call instead of once
# per iteration (2 nets x 2 saved iterations x 221.7 MMAC).  Throughput and roofline figures keep counting the
# reference's algorithmic 30.353 GFLOP per pair; the executed work is stated next to it.
def hoisted_macs_per_pair():
    from demon_b200 import weights as W
    lm = W.layer_macs()
    return (ITERATIONS - 1) * sum(lm["%s/%s" % (net, l)] for net in ("netFlow2", "netDM2") for l in ("conv1y", "conv1x", "conv2y", "conv2x"))


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        try:
            p = json.load(open(path))
            burst = float(p.get("bf16_tflops", 1590.0))
            return {"hbm_gbs": float(p.get("hbm_gbs", 6650.0)), "bf16_tflops": burst,
                    "bf16_tflops_sustained": float(p.get("bf16_tflops_sustained", burst)), "source": "measured"}
        except (OSError, ValueError, TypeError):
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def measure_tf32_peak(dev, seconds=1.0):
    """Dense TF32 tensor-core throughput of THIS GPU right now: cuBLAS fp32 GEMM 8192^3 with TF32 math, back to back for
    ~1 s (sustained clocks), CUDA events.  Only the roofline denominator uses it; nothing on the timed path calls cuBLAS."""
    try:
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        c = torch.empty(n, n, device=dev)
        for _ in range(3):
            torch.matmul(a, b, out=c)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters, t_all, done = 20, 0.0, 0
        t_start = time.perf_counter()
        while time.perf_counter() - t_start < seconds:
            e0.record()
            for _ in range(iters):
                torch.matmul(a, b, out=c)
            e1.record()
            torch.cuda.synchronize()
            t_all += e0.elapsed_time(e1)
            done += iters
        torch.backends.cuda.matmul.allow_tf32 = old
        del a, b, c
        return 2.0 * n ** 3 * done / (t_all / 1e3) / 1e12
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """CPU threads this process may really use: scheduler affinity, capped by the cgroup CPU quota
    (os.cpu_count() reports the machine's cores, not the container's share)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return max(1, n)


def cores_note(threads):
    return ("%d threads used (fastest of a short calibration over {8, 16, 32}); the machine reports %d logical CPUs, this "
            "process may use %d (scheduler affinity / cgroup CPU quota)" % (threads, os.cpu_count() or 0, host_threads()))


def best_thread_count(run_one):
    """torch's CPU convolutions do not scale to every core count (oversubscription, tiny layers): try the full count
    and a few smaller ones on one small problem each and keep the fastest, so the baseline is the best the host can do."""
    full = host_threads()
    # more than ~32 threads only oversubscribes these small convolutions (measured: 128 threads are 100x slower than 8)
    cands = sorted({min(full, 32), min(full, 16), min(full, 8)}, reverse=True)
    best, best_t = full, None
    for c in cands:
        torch.set_num_threads(c)
        run_one()          # warm
        t0 = time.perf_counter()
        run_one()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def dump_outputs(out_dir, outputs):
    """Writes every array of `outputs` (name -> tensor or array, batch first) as out_dir/<name>.npy in float32 / float64;
    above DUMP_LIMIT_BYTES in all, a seeded sample of batch entries (the same for every array)."""
    arrays = {}
    for name, v in outputs.items():
        a = v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
        arrays[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        n = len(next(iter(arrays.values())))
        keep = np.sort(np.random.default_rng(0).choice(n, max(1, n * DUMP_LIMIT_BYTES // total), replace=False))
        arrays = {name: a[keep] for name, a in arrays.items()}
        print("bench.py: %d bytes of outputs: wrote a seeded sample of %d of %d batch entries" % (total, len(keep), n), file=sys.stderr)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def synthetic_inputs(batch, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(batch, 6, 192, 256, generator=g) - 0.5


def oracle_setup(pairs, seed=1234):
    from demon_b200 import weights as W
    from oracle import ops as oops
    from oracle.network import OracleNets
    net = OracleNets(W.synthetic_weights(0))
    ip = synthetic_inputs(pairs, seed).numpy()
    i22 = oops.median3x3_downsample(oops.median3x3_downsample(np.ascontiguousarray(ip[:, 3:6])))
    return net, ip, i22


def cpu_oracle_rate(pairs):
    """pairs/s of the CPU restatement of the reference path on `pairs` synthetic pairs (bounded sample).
    Returns (rate, seconds, threads used)."""
    net, ip, i22 = oracle_setup(pairs)
    threads = best_thread_count(lambda: net.bootstrap(ip[:1], i22[:1]))
    t0 = time.perf_counter()
    net.pipeline(ip, i22, iterations=ITERATIONS)
    dt = time.perf_counter() - t0
    return pairs / dt, dt, threads


def run_reference(args, rank):
    """Reference arm: the reference's own CPU implementation of the path on the host cores.  TensorFlow 1.4 cannot be
    installed offline, so the conv stack is the torch-CPU port and the geometry ops the C restatement (pinned bit for bit
    by the reference's op sources compiled as oracle/_ref): kind "port".  Same --steps / --warmup as the GPU arm; a step
    is a bounded sample of the step's workload."""
    if rank != 0:
        return
    steps, warmup = args.steps, max(0, args.warmup)
    if args.config == "refine1024":
        from demon_b200 import weights as W
        from oracle.network import OracleNets
        net = OracleNets(W.synthetic_weights(0))
        g = torch.Generator().manual_seed(1234)
        im = (torch.rand(1, 3, 768, 1024, generator=g) - 0.5).numpy()
        d2 = (torch.rand(1, 1, 192, 256, generator=g) * 0.5 + 0.25).numpy()
        threads = best_thread_count(lambda: net.refine(im, d2))
        sample, unit, run = 1, "images/s", (lambda: net.refine(im, d2))
        workload = "RefinementNet.eval at 1024x768 (BASELINE.json configs[4]), bounded sample of 1 image per step of the batch-8 workload, CPU"
    else:
        sample = 1 if args.config == "b1" else REF_PAIRS_PER_STEP
        net, ip, i22 = oracle_setup(sample)
        threads = best_thread_count(lambda: net.bootstrap(ip[:1], i22[:1]))
        unit, run = "pairs/s", (lambda: net.pipeline(ip, i22, iterations=ITERATIONS))
        workload = ("full pipeline (bootstrap + 3x iterative + refinement) at 256x192, %d pair(s) per step%s, CPU"
                    % (sample, "" if args.config == "b1" else " = a bounded sample of the batch-64 step"))
    for _ in range(warmup):
        run()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = run()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    value = sample * steps / dt
    line = {"impl": "reference", "metric": METRIC if args.config != "refine1024" else "images_per_sec_refine_1024x768", "value": value,
            "unit": unit, "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": workload},
            "cpu_baseline": {"value": value, "unit": unit, "cores": threads, "kind": "port",
                             "sample": "%d steps x %d, torch-CPU fp32 convolutions + C geometry ops (oracle/); %s" % (steps, sample, cores_note(threads))},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def l1_rel(a, r):
    return float(np.abs(a - r).sum() / np.abs(r).sum())


def layer_roofline(lib, net_ptr, lm, B, steps, ms_local, precision, tf32_peak, pk):
    """Per-layer CUDA-event times (demon_net_profile_*) folded per kernel family -> roofline of the dominant kernel."""
    FAMILIES = {0: "conv_simt_kernel (fp32 CUDA-core implicit GEMM)",
                1: "conv_tc_kernel (tcgen05 kind::tf32, operands in shared memory, %s)" % precision,
                2: "conv_tc_halo_kernel<halo> (tcgen05 kind::tf32, TMA halo tile, A operand in TMEM, %s)" % precision,
                3: "conv_tc_halo_kernel<per-tap> (tcgen05 kind::tf32, per-shift tiles, A operand in TMEM, %s)" % precision}
    fam = {k: [0.0, 0.0, 0] for k in FAMILIES}   # ms, MACs, launches
    top = []
    for i in range(lib.demon_net_num_layers(net_ptr)):
        name = lib.demon_net_layer_name(net_ptr, i).decode()
        t, calls, lpc, tc = ctypes.c_double(), ctypes.c_int64(), ctypes.c_int(), ctypes.c_int()
        lib.demon_net_layer_profile(net_ptr, i, ctypes.byref(t), ctypes.byref(calls), ctypes.byref(lpc), ctypes.byref(tc))
        if calls.value == 0:
            continue
        macs = lm[name] * B * calls.value
        f = fam[tc.value]
        f[0] += t.value; f[1] += macs; f[2] += calls.value * lpc.value
        top.append((t.value, name, macs, tc.value))
    top.sort(reverse=True)
    dom = max(fam, key=lambda k: fam[k][0])
    d_ms, d_macs, d_launches = fam[dom]
    achieved = 2.0 * d_macs / (d_ms / 1e3) / 1e12 if d_ms > 0 else 0.0
    mult = 3 if precision == "3xtf32" else 1
    if dom != 0:
        if tf32_peak:
            peak = tf32_peak
            peak_note = ("TF32 GEMM measured on this GPU in this run (cuBLAS fp32 8192^3 with TF32 math, sustained for ~1 s): %.1f TFLOP/s; "
                         "for reference %s bf16 sustained %.1f / 2 = %.1f" % (tf32_peak, pk["source"], pk["bf16_tflops_sustained"], pk["bf16_tflops_sustained"] / 2))
        else:
            peak = pk["bf16_tflops_sustained"] / 2.0
            peak_note = "DERIVED: %s bf16 sustained %.1f TF/s / 2 (kind::tf32 issues at half the bf16 rate); the TF32 GEMM measurement failed" % (pk["source"], pk["bf16_tflops_sustained"])
        peak_note += "; %s spends %d tensor MAC(s) per algorithmic MAC, so frac <= %.2f by construction" % (precision, mult, 1.0 / mult)
    else:
        peak = 2 * 128 * 148 * 1.965e9 / 1e12     # fp32 FFMA peak at clocks.max.sm
        peak_note = "fp32 FFMA peak 128 FMA/clk/SM x 148 SMs x 1965 MHz (no measured fp32 figure in MEASURED_PEAKS.json)"
    return {"bound": "tensor", "kernel": FAMILIES[dom], "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
            "frac": achieved / peak if peak else None, "traffic": None,
            "algorithmic_flops_per_launch": 2.0 * d_macs / max(1, d_launches), "avg_launch_ms": d_ms / max(1, d_launches),
            "launches_timed": d_launches, "kernel_share_of_step": d_ms / ms_local if ms_local else None, "peak_note": peak_note,
            "instrumented_ms_per_step": ms_local / steps,
            "kernels": [{"kernel": FAMILIES[k], "ms_per_step": fam[k][0] / steps, "share_of_step": fam[k][0] / ms_local,
                         "tflops": 2.0 * fam[k][1] / (fam[k][0] / 1e3) / 1e12 if fam[k][0] > 0 else 0, "launches_per_step": fam[k][2] // steps}
                        for k in sorted(fam, key=lambda k: -fam[k][0]) if fam[k][2]],
            "top_layers_ms_per_step": [{"layer": n, "ms": t / steps, "tflops": 2.0 * m / (t / 1e3) / 1e12 if t > 0 else 0, "kernel": k}
                                       for t, n, m, k in top[:8]]}, dom


def attach_traffic(roofline, dom):
    """DRAM traffic of the heaviest launch of the dominant kernel, from the committed `ncu --set full` capture."""
    for fname in ("r02_traffic.json", "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", fname)
        if not os.path.isfile(tpath):
            continue
        tj = json.load(open(tpath))
        key = {2: "refine0_upconv", 1: "refine3_upconv", 3: "refine3_upconv"}.get(dom)
        if key not in tj:
            key = {2: "refine0_upconv", 1: "refine2_upconv", 3: "refine2_upconv"}.get(dom)
        if key in tj:
            roofline["traffic"] = {"bytes": tj[key], "launch": key,
                                   "algorithmic_bytes": {"refine0_upconv": 2 * 64 * 96 * 128 * 128 * 4 + 4 * 4 * 128 * 32 * 4,
                                                         "refine2_upconv": 64 * 24 * 32 * 256 * 4 + 64 * 48 * 64 * 64 * 4,
                                                         # netFlow2/refine3/upconv: concat4 [64,12,16,576] in, [64,24,32,128] out, 4x4 kernel
                                                         "refine3_upconv": 64 * 12 * 16 * 576 * 4 + 64 * 24 * 32 * 128 * 4 + 16 * 128 * 576 * 4}.get(key),
                                   "source": "profiles/%s (one launch at batch 64, dram__bytes_read.sum + dram__bytes_write.sum of an ncu --set full capture)" % fname}
            return


def bench_refine(args, rank, local, world, dev, lib, precision):
    """BASELINE.json configs[4]: RefinementNet at 1024x768, batch 8, one GPU.  A step = one RefinementNet.eval."""
    from demon_b200 import _lib, weights as W
    from demon_b200.networks_original import Session, RefinementNet
    B, H, Wd = 8, 768, 1024
    sess = Session(precision=precision)
    sess.load_weights(W.synthetic_weights(0))
    rn = RefinementNet(sess, batch_size=B, image_size=(H, Wd))
    g = torch.Generator().manual_seed(1234 + rank)
    ims = [(torch.rand(B, 3, H, Wd, generator=g) - 0.5).to(dev) for _ in range(4)]      # 4 x 75.5 MB rotating inputs > L2
    d2s = [(torch.rand(B, 1, H // 4, Wd // 4, generator=g) * 0.5 + 0.25).to(dev) for _ in range(4)]
    net = sess.net(B, (H, Wd))
    for i in range(max(3, args.warmup)):
        out = rn.eval(ims[i % 4], d2s[i % 4])
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = lib.demon_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        out = rn.eval(ims[i % 4], d2s[i % 4])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    launches = int(lib.demon_launch_count() - l0)
    _lib.check(lib.demon_net_profile_begin(net.ptr))
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for i in range(args.steps):
        out = rn.eval(ims[i % 4], d2s[i % 4])
    e3.record()
    torch.cuda.synchronize()
    ms_local = e2.elapsed_time(e3)
    _lib.check(lib.demon_net_profile_end(net.ptr))
    clocks = sampler.stop()
    _lib.check_errors()
    tf32_peak = measure_tf32_peak(dev)
    roofline, dom = layer_roofline(lib, net.ptr, W.layer_macs((H, Wd)), B, args.steps, ms_local, precision, tf32_peak, peaks())
    # end to end: numpy in -> numpy out through RefinementNet.eval (pageable host arrays, H2D + D2H + sync inside)
    im_h, d2_h = ims[0].cpu().numpy(), d2s[0].cpu().numpy()
    rn.eval(im_h, d2_h)
    n_e2e = max(2, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        res = rn.eval(im_h, d2_h)
    dt = time.perf_counter() - t0
    # check: one image of the last result against the CPU oracle
    from oracle.network import OracleNets
    ref = OracleNets(W.synthetic_weights(0)).refine(im_h[:1], d2_h[:1])["predict_depth0"].numpy()
    flops_img = 2.0 * W.macs_per_pair()["refine_fn"](H, Wd)
    value = B * args.steps / (ms / 1e3)
    line = {"metric": "images_per_sec_refine_1024x768", "value": value, "unit": "images/s", "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if precision == "fp32" else ("tf32x3" if precision == "3xtf32" else "tf32"), "data": "synthetic",
            "config": {"workload": "BASELINE.json configs[4]: RefinementNet (depth_refine_block) at 1024x768, batch 8, 1 GPU", "precision": precision,
                       "flops_per_image": flops_img, "l2": "4 rotating input batches of 75.5 MB (> 126 MB L2) and a %.2f GB activation workspace"
                                                          % (lib.demon_net_workspace_bytes(net.ptr) / 1e9)},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "algorithmic_tflops": flops_img * value / 1e12,
            "e2e": {"value": B * n_e2e / dt, "unit": "images/s", "h2d_bytes_per_step": int(im_h.nbytes + d2_h.nbytes), "d2h_bytes_per_step": int(B * H * Wd * 4),
                    "api": "RefinementNet.eval(numpy, numpy) -> numpy: pageable host arrays, copies and synchronisation inside the call"},
            "check": {"tc_timeouts": 0, "l1_rel_vs_cpu_oracle_fp32": l1_rel(res["predict_depth0"][:1], ref), "sample": "image 0 of the last e2e step"}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="b64", choices=["b64", "b1", "refine1024"])
    ap.add_argument("--precision", default=None, choices=["fp32", "3xtf32", "tf32"])
    ap.add_argument("--batch", type=int, default=None, help="pairs per GPU (default: 64 = BASELINE.json configs[2]; 1 with --config b1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--inflight", type=int, default=None, help="batches in flight per GPU (pipelines on their own streams); default 2, 1 with --config b1")
    ap.add_argument("--no-step-graph", action="store_true", help="do not capture pipeline + all-gather in one CUDA graph per step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    from demon_b200 import _lib, parallel, weights as W
    from demon_b200.networks_original import Session, DemonPipeline, DEFAULT_PRECISION
    rank, local, world = parallel.init_from_env()
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = _lib.load()
    precision = args.precision or DEFAULT_PRECISION
    if args.config == "refine1024":
        if rank == 0:
            bench_refine(args, rank, local, world, dev, lib, precision)
        return
    B = args.batch if args.batch is not None else (1 if args.config == "b1" else PER_GPU_BATCH)
    NF = max(1, args.inflight if args.inflight is not None else (1 if args.config == "b1" else 2))

    sess = Session(precision=precision)
    sess.load_weights(W.synthetic_weights(0))
    pipes = [DemonPipeline(sess, batch_size=B, iterations=ITERATIONS, private_net=(k > 0)) for k in range(NF)]
    net = pipes[0].net
    inputs = [synthetic_inputs(B, 1234 + rank + 1000 * i).to(dev) for i in range(N_INPUT_SETS)]
    gathers = [parallel.OutputGather(B, world, device=dev) for _ in range(NF)]
    # the pipeline writes its results straight into the send buffer of the all-gather
    outs = []
    for g in gathers:
        d, r, t = g.local_buffers()
        outs.append({"predict_depth0": d, "predict_rotation": r, "predict_translation": t})
    streams = [torch.cuda.Stream(device=dev) for _ in range(NF)]

    def body(k):   # pipeline on the staged inputs + the ONE collective of the path
        pipes[k].forward_staged(outs[k])
        gathers[k]()

    # One CUDA graph per in-flight slot: the ~230 kernels of the pipeline AND the NCCL all-gather are captured together
    # (demon_pipeline_forward sees the capture and launches its kernels into it), so a step is one graph launch.
    graphs = [None] * NF
    graph_note = "off"
    if not args.no_step_graph:
        try:
            for k in range(NF):
                with torch.cuda.stream(streams[k]):
                    pipes[k].stage(inputs[0])
                    for _ in range(2):
                        body(k)          # warm: the first eager pass, NCCL's lazy initialisation
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=streams[k]):
                    body(k)
                graphs[k] = g
            graph_note = "one CUDA graph per step: pipeline kernels + all-gather"
        except Exception as e:   # keep measuring without the step graph (the C call then replays its own graph, the gather is a separate launch)
            graphs = [None] * NF
            graph_note = "capture failed (%s): pipeline graph inside the C call, gather launched separately" % str(e).splitlines()[0][:120]
            torch.cuda.synchronize()

    def step2(i):
        k = i % NF
        with torch.cuda.stream(streams[k]):
            pipes[k].stage(inputs[(i // NF) % N_INPUT_SETS])
            if graphs[k] is not None:
                graphs[k].replay()
            else:
                body(k)

    def step1(i):   # everything on slot 0, one batch at a time (the instrumented region)
        with torch.cuda.stream(streams[0]):
            pipes[0].stage(inputs[i % N_INPUT_SETS])
            body(0)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput -------------------------------------------------------------
    # Two timed regions: the first gives `value` (no instrumentation, NF batches in flight); the second runs the same
    # steps on one stream with CUDA events around every layer launch on the launching stream (demon_net_profile_*) and
    # feeds the roofline figures.
    for i in range(NF * max(args.warmup, 3)):
        step2(i)
    for i in range(args.warmup):
        step1(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = lib.demon_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(streams[0])
    for k in range(1, NF):
        streams[k].wait_event(ev0)
    for i in range(args.steps):
        step2(i)
    for k in range(1, NF):
        ev_b = torch.cuda.Event()
        ev_b.record(streams[k])
        streams[0].wait_event(ev_b)
    ev1.record(streams[0])
    barrier()
    ms_value = ev0.elapsed_time(ev1)
    launches = int(lib.demon_launch_count() - launches0)
    if graphs[0] is not None:   # kernels replayed from the step graphs are not seen by the library's launch counter
        launches += args.steps * lib.demon_net_pipeline_launches(net.ptr, ITERATIONS)
    last_k = (args.steps - 1) % NF
    last_in = inputs[((args.steps - 1) // NF) % N_INPUT_SETS]
    last_depth0 = gathers[last_k].depth_all[rank, 0, 0].cpu().numpy()       # sample 0 of this rank's shard, last timed step
    last_trans0 = gathers[last_k].translation_all[rank, 0].cpu().numpy()
    if args.dump_outputs and rank == 0:
        g = gathers[last_k]
        dump_outputs(args.dump_outputs, {"predict_depth0": g.depth_all.flatten(0, 1), "predict_rotation": g.rotation_all.flatten(0, 1),
                                         "predict_translation": g.translation_all.flatten(0, 1)})
    _lib.check_errors()
    # time of the gather alone (it is inside `value`): per-N record for the scaling discussion
    gather_ms = None
    if world > 1:
        eg0, eg1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        with torch.cuda.stream(streams[0]):
            eg0.record()
            for _ in range(10):
                gathers[0]()
            eg1.record()
        barrier()
        gather_ms = parallel.max_over_ranks(eg0.elapsed_time(eg1) / 10, dev)
    _lib.check(lib.demon_net_profile_begin(net.ptr))
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev2.record(streams[0])
    for i in range(args.steps):
        step1(i)
    ev3.record(streams[0])
    barrier()
    ms_local = ev2.elapsed_time(ev3)
    _lib.check(lib.demon_net_profile_end(net.ptr))
    clocks = sampler.stop() if rank == 0 else None
    _lib.check_errors()
    ms = parallel.max_over_ranks(ms_value, dev)
    value = world * B * args.steps / (ms / 1e3)

    tf32_peak = measure_tf32_peak(dev) if rank == 0 else None
    roofline, dom = layer_roofline(lib, net.ptr, W.layer_macs(), B, args.steps, ms_local, precision, tf32_peak, peaks())
    if B == PER_GPU_BATCH:
        attach_traffic(roofline, dom)

    # ---- end to end from pinned host buffers, copies inside the timed region -----------------------------------------
    NE = NF
    h_in = [synthetic_inputs(B, 4321 + rank + 1000 * i).pin_memory() for i in range(NE)]
    e2e_steps = max(4, min(args.steps, 20))
    if world == 1:
        # through the C-ABI host entry: H2D, pipeline, D2H of depth0 + motion; NE pipelines on NE streams so that one
        # batch's copies overlap the other's compute; the region ends when the last result is on the host
        h_depth = [torch.empty(B, 1, 192, 256).pin_memory() for _ in range(NE)]
        h_rot = [torch.empty(B, 3).pin_memory() for _ in range(NE)]
        h_tr = [torch.empty(B, 3).pin_memory() for _ in range(NE)]

        def e2e_step(i):
            k = i % NE
            streams[k].synchronize()            # the previous result of this slot is on the host (and may be consumed)
            pipes[k].forward_host_async(h_in[k], None, h_depth[k], h_rot[k], h_tr[k], streams[k])
        d2h = int((h_depth[0].numel() + 6 * B) * 4)
        api = ("demon_pipeline_forward_host_async (C ABI) via DemonPipeline.forward_host_async: pinned host buffers, %d pipeline(s) on "
               "own streams so that one batch's copies overlap the other's compute" % NE)
    else:
        # N > 1: pinned host -> device, pipeline, the all-gather, then the gathered result to the host of rank 0 (the own
        # shard on the other ranks): the multi-GPU end-to-end path includes the path's only collective
        rec = gathers[0].record
        h_out = [torch.empty(world * rec if rank == 0 else rec).pin_memory() for _ in range(NE)]

        def e2e_step(i):
            k = i % NE
            streams[k].synchronize()
            with torch.cuda.stream(streams[k]):
                pipes[k].stage(h_in[k])          # H2D (pinned, asynchronous)
                if graphs[k] is not None:
                    graphs[k].replay()
                else:
                    body(k)
                h_out[k].copy_(gathers[k].flat_all if rank == 0 else gathers[k].local, non_blocking=True)
        d2h = int((world * rec if rank == 0 else rec) * 4)
        api = ("DemonPipeline.stage (H2D from pinned host) + forward_staged + OutputGather (one NCCL all-gather) + D2H of the gathered "
               "depth/motion on rank 0 (%d bytes; the own shard, %d bytes, on the other ranks)" % (world * rec * 4, rec * 4))
    for i in range(3 * NE):
        e2e_step(i)
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    torch.cuda.synchronize()
    dt_local = time.perf_counter() - t0
    barrier()
    _lib.check_errors()
    dt = parallel.max_over_ranks(dt_local, dev)
    e2e = {"value": world * B * e2e_steps / dt, "unit": "pairs/s", "h2d_bytes_per_step": int(h_in[0].numel() * 4),
           "d2h_bytes_per_step": d2h, "steps": e2e_steps, "api": api}
    # the same end to end from uint8 images (what examples/example.py loads): /255 - 0.5, pair concat and image2_2 on the
    # device, a quarter of the host -> device bytes.  Extra information; `e2e` above stays on the fp32 inputs the CPU arm gets.
    e2e_u8 = None
    if world == 1:
        g8 = torch.Generator().manual_seed(99)
        h_u8 = [torch.randint(0, 256, (B, 2, 192, 256, 3), generator=g8, dtype=torch.uint8).pin_memory() for _ in range(NE)]

        def e2e_u8_step(i):
            k = i % NE
            streams[k].synchronize()
            pipes[k].forward_host_u8(h_u8[k], None, h_depth[k], h_rot[k], h_tr[k], streams[k], sync=False)
        for i in range(3 * NE):
            e2e_u8_step(i)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            e2e_u8_step(i)
        torch.cuda.synchronize()
        dt8 = time.perf_counter() - t0
        _lib.check_errors()
        e2e_u8 = {"value": B * e2e_steps / dt8, "unit": "pairs/s", "h2d_bytes_per_step": int(h_u8[0].numel()), "d2h_bytes_per_step": d2h,
                  "steps": e2e_steps, "api": "demon_pipeline_forward_host_u8_async (C ABI) via DemonPipeline.forward_host_u8(sync=False): uint8 "
                  "[B,2,192,256,3] images in pinned host memory, preprocessing on the device"}

    # ---- CPU side (rank 0): check of the last timed step against the oracle, and the CPU baseline at N=1 -------------
    cpu, check = None, None
    if rank == 0:
        from oracle import ops as oops
        from oracle.network import OracleNets
        onet = OracleNets(W.synthetic_weights(0))
        ip1 = last_in[:1].cpu().numpy()
        i22 = oops.median3x3_downsample(oops.median3x3_downsample(np.ascontiguousarray(ip1[:, 3:6])))
        torch.set_num_threads(min(host_threads(), 16))
        ref = onet.pipeline(ip1, i22, iterations=ITERATIONS)
        check = {"tc_timeouts": 0, "l1_rel_depth0_vs_cpu_oracle_fp32": l1_rel(last_depth0, ref["predict_depth0"].numpy()[0, 0]),
                 "max_abs_translation_diff": float(np.abs(last_trans0 - ref["predict_translation"].numpy()[0]).max()),
                 "sample": "pair 0 of rank 0's shard in the LAST step of the timed region behind `value` (read from the gathered buffer)",
                 "tolerance": 1e-4}
        assert check["l1_rel_depth0_vs_cpu_oracle_fp32"] < 1e-3, "the timed region produced wrong depth: %r" % check
        if world == 1 and not args.no_cpu_baseline:
            pairs = 8 if B >= 8 else 1
            rate, secs, threads = cpu_oracle_rate(pairs)
            cpu = {"value": rate, "unit": "pairs/s", "cores": threads, "kind": "port",
                   "sample": "%d pair(s) of the same synthetic workload, one pass (%.1f s), torch-CPU fp32 convolutions + C geometry ops; %s"
                             % (pairs, secs, cores_note(threads))}

    if rank == 0:
        alg_flops = 2.0 * W.macs_per_pair()["pipeline"]
        line = {"metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32" if precision == "fp32" else ("tf32x3" if precision == "3xtf32" else "tf32"), "data": "synthetic",
                "config": {"workload": "BASELINE.json configs[%d]: batch=%d synthetic 256x192 pair(s) per GPU, full pipeline "
                                       "(bootstrap + 3x iterative + refinement), %d GPU(s)" % ((1 if B == 1 else 2) if world == 1 else 3, B, world),
                           "global_batch": world * B, "precision": precision, "iterations": ITERATIONS,
                           "l2": "%d rotating input batches of %.1f MB%s and a %.2f GB activation workspace rewritten every step"
                                 % (N_INPUT_SETS, B * 6 * 192 * 256 * 4 / 1e6, " (> 126 MB L2)" if B >= 32 else "",
                                    lib.demon_net_workspace_bytes(net.ptr) / 1e9),
                           "parallelism": "dp%d, one NCCL all-gather (one call) of depth0+motion per step" % world if world > 1 else "single GPU",
                           "step_graph": graph_note,
                           "batches_in_flight": "%d per GPU (pipelines with own workspaces on their own CUDA streams, steps alternate); the " % NF +
                                                "instrumented region behind `roofline` runs the same steps on one stream",
                           "flops_per_pair": alg_flops,
                           "executed_flops_per_pair": alg_flops - 2.0 * hoisted_macs_per_pair(),
                           "flops_note": "value, algorithmic_tflops and roofline count the reference's algorithmic work; conv1/conv2 of the "
                                         "iterative nets are loop invariant and executed once per call (bit identical)"},
                "gpu_launches": launches, "clocks": clocks, "e2e": e2e, "e2e_u8": e2e_u8, "roofline": roofline, "cpu_baseline": cpu, "check": check,
                "gather_ms": gather_ms, "algorithmic_tflops": alg_flops * value / 1e12}
        print(json.dumps(line), flush=True)
    if world > 1:
        # Leave without tearing NCCL down: the step graphs hold captured NCCL kernels, and destroy_process_group() on a
        # communicator that instantiated CUDA graphs still reference has been seen to hang after the result line was printed
        # (2 GPUs, torch 2.11 / NCCL 2.28).  Everything is synchronised and flushed; the exit code is 0 on every rank.
        torch.distributed.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
