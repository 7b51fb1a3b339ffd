"""
bench.py - headline benchmark of the DCSCN hot path (BASELINE.json: "output Mpixels/sec DCSCN L12 x2").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Headline: a "step" is one forward pass of DCSCN L12 F196->48 x2 over one batch of 256 synthetic 48x48 Y tiles
(BASELINE.json configs[1]) per GPU; `value` is whole-job output Mpixels/s with inputs resident in HBM, `e2e` is
the same metric through the reference-facing host-buffer call (H2D of x and x2 from pinned memory and D2H of y
inside the timed region).  Weights: the reference's own L12 x2 checkpoint (tests/golden/models fixture).

The same JSON line carries sub-records for the other BASELINE.json configurations, each measured in the same run with
CUDA events (max over ranks) and each with a self-check:
  * `ensemble8` (configs[2]): the 8-transform self-ensemble of Set5 img_001 (256x256 LR) with the transforms spread
    over the N ranks and ONE NCCL all-reduce of the float64 partial sums; max |sharded - single-rank|.
  * `train`     (configs[3]): data-parallel train step of DCSCN L12 x4, 64 patches of 48x48 per rank, ONE flat
    all-reduce of [gradients | loss | mse]; patches/s, achieved TFLOP/s, and max |w_DP - w_single-rank| after one
    update of a small batch.
  * `ds`        (configs[4]): depthwise-separable c-DCSCN x4 inference with its HBM roofline.
  * `latency`   : batch-1 whole-image Set5 evaluation (the reference's evaluate.py shape), seconds per image.

`--impl reference` times the CPU oracle (the reference's graph restated on torch-CPU fp32; TensorFlow is not
installable in this image, see DESIGN.md) on all host cores of the box on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "dcscn-super-resolution_b200"))

MODEL = "dcscn_L12_F196to48_NIN_A64_PS_R1F32"
MODEL_X4 = "dcscn_L12_F196to48_Sc4_NIN_A64_PS_R1F32"
MODEL_DS = "dcscn_L7_F32to8_G1.20_Sc4_NIN_A24_B8_PS_DS_R1F32"
BATCH, TILE, SCALE = 256, 48, 2
CPU_TILES = 32   # tiles per CPU-oracle call, in the reference arm AND in the in-line cpu_baseline
# SURVEY.md section 8(d): algorithmic work, no padding / recompute
FLOP_PER_LR_PX_TOTAL = 3508584.0           # L12 x2 forward
MAC_PER_LR_PX_TC = 1754292 - 9 * 196 - 4 * 864  # tensor-core layers: all but CNN1 (cin=1) and R-CNN1 (cout=1, 4 HR px per LR px)
FLOP_PER_LR_PX_X4 = 6183528.0              # L12 x4 forward; a train step is counted as 3x (forward + dgrad + wgrad)
DS_BYTES_PER_LR_PX = (331 + 570) * 4.0     # DS c-DCSCN x4, layer-by-layer HBM floor (SURVEY.md 8d)


def load_weights(model=MODEL):
    from helper import tf_bundle
    r = tf_bundle.BundleReader(os.path.join(ROOT, "tests", "golden", "models", model + ".ckpt"))
    return {k: r.get_tensor(k) for k in r.keys()}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1405.3), d.get("bf16_tflops", 1652.1), d.get("hbm_gbs", 6560.6), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], None, set(), []
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax = float(r[1])
                power.append(float(r[2]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


def ncu_traffic():
    """DRAM bytes (read + write) of the tcgen05 conv launches of one step, from the newest committed `ncu --set full`
    capture (profiles/r*_traffic.json); (None, None) if there is none.  NOT measured by this run: bench.py cannot run
    under a profiler and report a timing at once."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
    for f in reversed(files):
        try:
            t = json.load(open(f))
            return int(t["dram_bytes_read"] + t["dram_bytes_write"]), "committed capture %s: %s" % (os.path.basename(f), t["source"])
        except (OSError, KeyError, ValueError):
            continue
    return None, None


# --------------------------------------------------------------------------------------------- CPU oracle ----
def _usable_cpus():
    """Cores this process may really use: scheduler affinity capped by the cgroup CPU quota (a container that sees 128
    CPUs but owns 16 of them runs 16x slower with 128 threads than with 16)."""
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n)


def _pin_cpu_threads(probe=None):
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm must use the whole box whatever launched it.  The thread count is
    the fastest of a few candidates (usable cores, half, quarter, torch's own default) on a short probe run - more
    threads than the box really gives is much slower, not faster."""
    import torch
    n = _usable_cpus()
    cands = sorted({n, max(1, n // 2), max(1, n // 4), min(n, max(1, torch.get_num_threads()))}, reverse=True)
    if probe is None or len(cands) == 1:
        torch.set_num_threads(cands[0])
        return torch.get_num_threads()
    best, best_t = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        probe()                                   # warm the pool at this size
        t0 = time.perf_counter()
        probe()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return torch.get_num_threads()


def cpu_oracle_passes(passes, warm, tiles=CPU_TILES):
    """`passes` timed forwards of the CPU oracle (torch-CPU fp32) over `tiles` 48x48 tiles of the bench workload;
    returns (per-pass seconds list, threads)."""
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import dcscn_oracle as O
    orc = O.Oracle(O.OracleConfig(), load_weights(), torch.float32)
    g = np.random.RandomState(0)
    x = (g.rand(tiles, TILE, TILE, 1) * 255).astype(np.float32)
    x2 = (g.rand(tiles, SCALE * TILE, SCALE * TILE, 1) * 255).astype(np.float32)
    threads = _pin_cpu_threads(probe=lambda: orc.forward(x[:4], x2[:4]))
    for _ in range(max(1, warm)):
        orc.forward(x, x2)   # warm-up (thread pool, oneDNN primitive cache)
    secs = []
    for _ in range(passes):
        t0 = time.perf_counter()
        orc.forward(x, x2)
        secs.append(time.perf_counter() - t0)
    return secs, threads


def _median(v):
    s = sorted(v)
    return s[len(s) // 2] if len(s) % 2 else 0.5 * (s[len(s) // 2 - 1] + s[len(s) // 2])


def run_reference(args, rank, world):
    if rank != 0:
        return
    steps, warm = max(3, args.steps), args.warmup
    secs, threads = cpu_oracle_passes(steps, warm)
    med = _median(secs)
    val = CPU_TILES * (SCALE * TILE) ** 2 / med / 1e6
    sample = ("%d of the 256 48x48 tiles per step, %d timed steps, value from the MEDIAN step; torch-CPU fp32 oracle port "
              "(TensorFlow not installable)" % (CPU_TILES, steps))
    line = {
        "impl": "reference", "metric": "output Mpixels/sec DCSCN L12 x2", "value": val, "unit": "Mpixels/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": med * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "DCSCN L12 F196->48 x2 inference, 48x48 Y tiles, CPU sample of %d tiles/step" % CPU_TILES,
                   "cpu_threads": threads, "launched_by": "torchrun" if world > 1 else "python"},
        "cpu_baseline": {"value": val, "unit": "Mpixels/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ helpers ----
class Job:
    """One rank of the bench job: device, optional NCCL group, max-over-ranks reductions."""

    def __init__(self, rank, world, local_rank):
        import torch
        self.torch = torch
        self.rank, self.world, self.local = rank, world, local_rank
        torch.cuda.set_device(local_rank)
        self.dist = None
        if world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.dist is None:
            return float(v)
        t = self.torch.tensor([float(v)], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps, warm):
        """W warm-up calls, barrier + sync, K calls between two CUDA events, barrier + sync; max ms over ranks."""
        torch = self.torch
        for i in range(warm):
            fn(i)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warm + i)
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1))

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def umma_isolated(device):
    """kind::f16 tcgen05.mma throughput with operands resident in shared memory (dcscn_umma_probe, csrc/umma_probe.cuh),
    measured in this run: the pipe's peak at N = 256 and the cost of one K = 16 slice of the three-product scheme for the
    widths of the thin layers (a UMMA cannot go faster than its operands leave shared memory: ~40 cycles at N <= 80)."""
    import ctypes
    from helper import engine as E
    lib = E.load_library()

    def one(n, mode, iters=3000):
        ms, cyc = ctypes.c_float(), ctypes.c_double()
        if lib.dcscn_umma_probe(device, 2, n, mode, iters, ctypes.byref(ms), ctypes.byref(cyc)):
            return None
        prods = 3 if mode == 0 else 1
        macs = 74 * iters * 4 * prods * 256 * n * 16
        return {"tflops_issued": round(2 * macs / (ms.value * 1e-3) / 1e12, 1), "cycles_per_k16_slice": round(cyc.value / (iters * 4), 1)}
    try:
        out = {"what": "tcgen05.mma kind::f16 cta_group::2 M=256, both operands in shared memory, 74 CTA pairs, no loads / epilogue",
               "n256_three_products": one(256, 0)}
        for n in (48, 80, 112, 160):
            out["n%d_three_products" % n] = one(n, 0)
        return out
    except Exception as e:  # noqa: BLE001
        return {"error": "%s: %s" % (type(e).__name__, e)}


def headline(job, args):
    import numpy as np
    import torch
    from helper import engine as E
    rank, world = job.rank, job.world
    prec = {"f16x3": E.PRECISION_F16X3, "f16x1": E.PRECISION_F16X1}[args.precision]
    eng = E.Engine(E.make_config(device_id=job.local, precision=prec))
    eng.set_params(load_weights())

    gen = torch.Generator().manual_seed(0 + rank)
    x_host = (torch.rand(BATCH, TILE, TILE, 1, generator=gen) * 255).pin_memory()
    x2_host = (torch.rand(BATCH, SCALE * TILE, SCALE * TILE, 1, generator=gen) * 255).pin_memory()
    y_host = torch.empty(BATCH, SCALE * TILE, SCALE * TILE, 1).pin_memory()
    x, x2 = x_host.cuda(), x2_host.cuda()
    y = torch.empty_like(x2)
    warm = max(args.warmup, 3)

    for _ in range(warm):
        eng.forward(x, x2, y)
    job.barrier()
    sampler = ClockSampler(job.local)
    if rank == 0:
        sampler.start()
    launches0 = eng.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        eng.forward(x, x2, y)
    ev1.record()
    job.barrier()
    ms = job.max_over_ranks(ev0.elapsed_time(ev1))
    launches = eng.launch_count - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # y of the last timed step, before the strict pass below overwrites it with another promotion setting
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "y.npy"), y.cpu().numpy())
    out_px_step = BATCH * (SCALE * TILE) ** 2
    value = world * out_px_step * args.steps / (ms / 1e3) / 1e6

    # ---- end to end through the host-buffer API (pinned host memory in, pinned host memory out) ----
    for _ in range(2):
        eng.forward_host(x_host, x2_host, y_host)
    job.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.forward_host(x_host, x2_host, y_host)
    torch.cuda.synchronize()
    e2e_s = job.max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * out_px_step * args.steps / e2e_s / 1e6

    # ---- per-launch device times (separate pass; CUDA events on the launching stream; median of >= 5 reps) ----
    eng.set_option("timing", 1)
    per = {}
    for _ in range(max(5, min(args.steps, 9))):
        eng.forward(x, x2, y)
        for name, t in eng.timings():
            per.setdefault(name, []).append(t)
    eng.set_option("timing", 0)
    torch.cuda.synchronize()
    per = {k: _median(v) for k, v in per.items()}

    # ---- strict setting: every (chunk, dx) unit promoted to the fp32 RN sum (seg_chunks = 1): the setting that holds
    # 1e-3 absolute against the fp64 forward on these uniform-noise tiles (tests/test_gpu_forward.py) ----
    eng.set_option("seg_chunks", 1)
    n_strict = max(5, min(args.steps, 20))
    ms_strict = job.timed(lambda i: eng.forward(x, x2, y), n_strict, 3) / n_strict
    eng.close()
    strict = {"setting": "seg_chunks=1 (fp32 promotion after every (64-channel chunk, dx) unit of K = 192)",
              "ms_per_step": ms_strict, "value": world * out_px_step / (ms_strict / 1e3) / 1e6, "unit": "Mpixels/s",
              "noise_tile_error": "<= 1e-3 absolute vs the fp64 forward (default periods: ~1.35e-3; fp32 CPU forward: ~2.4e-3)"}
    return dict(ms=ms, value=value, e2e_value=e2e_value, launches=launches, clocks=clocks, per=per, warm=warm, strict=strict,
                h2d=int(x_host.numel() * 4 + x2_host.numel() * 4), d2h=int(y_host.numel() * 4))


def sub_ensemble(job, args):
    """BASELINE configs[2]: 8-transform self-ensemble of Set5 img_001 (LR 256x256), transforms spread over the ranks."""
    import numpy as np
    import torch
    from helper import engine as E
    from helper import loader, utilty as util
    img = util.set_image_alignment(util.load_image(os.path.join(ROOT, "tests", "golden", "data", "set5", "img_001.png"),
                                                   print_console=False), SCALE)
    lr = loader.build_input_image(img, channels=1, scale=SCALE, alignment=SCALE, convert_ycbcr=True)
    bic = util.resize_image_by_pil(lr, SCALE)
    h, w = lr.shape[:2]
    eng = E.Engine(E.make_config(device_id=job.local))
    eng.set_params(load_weights())
    xd = torch.from_numpy(np.ascontiguousarray(lr, dtype=np.float32).reshape(h, w)).cuda()
    x2d = torch.from_numpy(np.ascontiguousarray(bic, dtype=np.float32).reshape(SCALE * h, SCALE * w)).cuda()
    out = torch.empty(SCALE * h, SCALE * w, dtype=torch.float64, device="cuda")
    steps = max(5, min(args.steps, 20))
    ms = job.timed(lambda i: eng.forward_ensemble_sharded(xd, x2d, 8, out=out), steps, 3)
    single = eng.forward_ensemble(xd, x2d, 8)          # every rank: all 8 transforms alone
    diff = job.max_over_ranks(float((out - single).abs().max().item()))
    eng.close()
    out_px = (SCALE * h) * (SCALE * w)
    return {
        "workload": "self_ensemble=8 of Set5 img_001 (LR %dx%d -> %dx%d), transforms r, r+N, ... on rank r, one float64 "
                    "NCCL all-reduce of the partial sums (reference loop: DCSCN.py:560-573)" % (h, w, SCALE * h, SCALE * w),
        "ms_per_image": ms / steps, "images_per_s": 1e3 * steps / ms,
        "value": out_px * steps / (ms / 1e3) / 1e6, "unit": "output Mpixels/s (one image, all 8 passes)",
        "forward_mpix_per_s": 8 * out_px * steps / (ms / 1e3) / 1e6,
        "collective": "all_reduce(sum) of %d float64 (%.2f MB) per image" % (out_px, out_px * 8 / 1e6) if job.world > 1 else "none (1 rank)",
        "max_abs_sharded_minus_single_rank": diff,
    }


def sub_train(job, args):
    """BASELINE configs[3]: L12 x4 train step, 64 patches of 48x48 per rank, data parallel."""
    import numpy as np
    import torch
    from helper import engine as E
    rank, world = job.rank, job.world
    per_gpu = 64
    w4 = load_weights(MODEL_X4)
    eng = E.Engine(E.make_config(scale=4, device_id=job.local, dropout_keep=0.8))
    eng.set_params(w4)
    gen = torch.Generator().manual_seed(2 + rank)
    x = (torch.rand(per_gpu, 48, 48, 1, generator=gen) * 255).cuda()
    x2 = (torch.rand(per_gpu, 192, 192, 1, generator=gen) * 255).cuda()
    y = (torch.rand(per_gpu, 192, 192, 1, generator=gen) * 255).cuda()
    steps = max(5, min(args.steps, 20))
    l0 = eng.launch_count
    # tiny lr: every kernel of the step runs (forward, backward, all-reduce, clip, Adam, weight refresh) while the weights
    # stay next to the checkpoint's (uniform-noise targets at lr 2e-3 would blow a converged model up within the run)
    ms = job.timed(lambda i: eng.train_step_data_parallel(x, x2, y, lr=1e-6, seed=i * world + rank), steps, 3)
    launches = (eng.launch_count - l0) / (steps + 3)
    eng.close()
    sustained = measured_peaks()[0]
    flop_step = 3.0 * FLOP_PER_LR_PX_X4 * per_gpu * 48 * 48          # per rank
    tfs = flop_step / (ms / steps / 1e3) / 1e12                       # per GPU

    # ---- equivalence: one data-parallel update == one single-rank update on the whole small batch (dropout off) ----
    nb, hw = 8, 24
    eq = None
    if nb % world == 0:
        g = np.random.RandomState(7)
        xs = (g.rand(nb, hw, hw, 1) * 255).astype(np.float32)
        x2s = (g.rand(nb, 4 * hw, 4 * hw, 1) * 255).astype(np.float32)
        ys = np.clip(x2s + g.randn(nb, 4 * hw, 4 * hw, 1).astype(np.float32) * 8, 0, 255).astype(np.float32)
        e2 = E.Engine(E.make_config(scale=4, device_id=job.local, dropout_keep=1.0))
        e2.set_params(w4)
        e2.train_step_host(xs, x2s, ys, lr=0.002, seed=1, apply_update=True)        # single rank, whole batch
        names = ["CNN2/conv_W", "A1/conv_W", "Up-PS2/Up-PS2_CNN/conv_W", "R-CNN1/conv_W", "CNN12/conv_B", "B2/prelu/B2_prelu"]
        w_single = {n: e2.get_param(n) for n in names}
        e2.set_params(w4)
        e2.reset_optimizer()
        sh = slice(rank, None, world)
        e2.train_step_data_parallel(np.ascontiguousarray(xs[sh]), np.ascontiguousarray(x2s[sh]),
                                    np.ascontiguousarray(ys[sh]), lr=0.002, seed=1)
        d = max(float(np.abs(e2.get_param(n) - w_single[n]).max()) for n in names)
        step_size = max(float(np.abs(w_single[n] - w4[n]).max()) for n in names)
        e2.close()
        eq = {"max_abs_w_dp_minus_w_single": job.max_over_ranks(d), "max_abs_update": step_size, "lr": 0.002,
              "batch": "%d patches of %dx%d, dropout off, Adam step 1, %d variables compared" % (nb, hw, hw, len(names))}
    return {
        "workload": "DCSCN L12 F196->48 x4 train step, %d 48x48 patches per rank (global batch %d), dropout keep 0.8, "
                    "MSE + L2, global-norm clip, Adam (reference: DCSCN.py:334-425)" % (per_gpu, per_gpu * world),
        "ms_per_step": ms / steps, "value": per_gpu * world * steps / (ms / 1e3), "unit": "patches/s",
        "collective": ("one all_reduce(sum) of [gradients | loss | mse] = %d fp32 (%.2f MB) per step, then mean + clip + Adam "
                       "on every rank" % (2087102 + 2, (2087102 + 2) * 4 / 1e6)) if world > 1 else "none (1 rank)",
        "tflops_per_gpu": tfs, "frac_of_bf16_sustained": tfs / sustained,
        "flop_model": "3 x forward (6,183,528 FLOP per LR pixel, SURVEY.md 8d) per patch pixel",
        "gpu_launches_per_step": launches, "timed_with": "lr = 1e-6 on the checkpoint weights (every kernel of the step runs; uniform-noise targets at lr 2e-3 would blow a converged model up within the run)",
        "dp_equals_single_rank": eq,
    }


def sub_ds(job, args):
    """BASELINE configs[4]: depthwise-separable c-DCSCN L7 x4 inference, 256 tiles."""
    import torch
    from helper import engine as E
    eng = E.Engine(E.make_config(scale=4, layers=7, filters=32, min_filters=8, filters_decay_gamma=1.2, nin_filters=24,
                                 nin_filters2=8, reconstruct_layers=0, pixel_shuffler_filters=1, depthwise_separable=True,
                                 device_id=job.local))
    eng.set_params(load_weights(MODEL_DS))
    gen = torch.Generator().manual_seed(3 + job.rank)
    x = (torch.rand(256, 48, 48, 1, generator=gen) * 255).cuda()
    x2 = (torch.rand(256, 192, 192, 1, generator=gen) * 255).cuda()
    yb = torch.empty_like(x2)
    steps = max(5, min(args.steps, 30))
    ms = job.timed(lambda i: eng.forward(x, x2, yb), steps, 3)
    eng.close()
    hbm = measured_peaks()[2]
    bytes_step = DS_BYTES_PER_LR_PX * 256 * 48 * 48
    gbs = bytes_step / (ms / steps / 1e3) / 1e9
    return {
        "workload": "depthwise-separable c-DCSCN L7 x4 inference, batch=256 synthetic 48x48 tiles per rank",
        "ms_per_step": ms / steps, "value": job.world * 256 * 192 * 192 * steps / (ms / 1e3) / 1e6, "unit": "output Mpixels/s",
        "dtype": "f32 (CUDA cores)",
        "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                     "algorithmic_bytes_per_step": bytes_step,
                     "bytes_model": "layer-by-layer floor (331 floats written + 570 read) x 4 B per LR pixel, SURVEY.md 8d"},
    }


def sub_latency(job, args):
    """Batch-1 whole-image evaluation of Set5 (the shape of the reference's evaluate.py:93-107): wall-clock seconds
    per image around load -> Y -> bicubic -> do() -> PSNR, self_ensemble 8 and 1; rank 0 only."""
    if job.rank != 0:
        return None
    import glob
    import numpy as np
    from helper import engine as E
    from helper import loader, utilty as util
    files = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "data", "set5", "*.png")))
    eng = E.Engine(E.make_config(device_id=job.local))
    eng.set_params(load_weights())
    res = {}
    for ens in (8, 1):
        for timed_pass in (False, True):          # first pass builds the per-shape launch plans
            t_total, t_gpu, psnrs = 0.0, 0.0, []
            for f in files:
                t0 = time.perf_counter()
                true_image = util.set_image_alignment(util.load_image(f, print_console=False), SCALE)
                lr = loader.build_input_image(true_image, channels=1, scale=SCALE, alignment=SCALE, convert_ycbcr=True)
                bic = util.resize_image_by_pil(lr, SCALE)
                t1 = time.perf_counter()
                if ens > 1:
                    out = eng.forward_ensemble_host(lr, bic, ens)
                else:
                    h, w = lr.shape[:2]
                    out = eng.forward_host(np.ascontiguousarray(lr, np.float32).reshape(1, h, w, 1),
                                           np.ascontiguousarray(bic, np.float32).reshape(1, SCALE * h, SCALE * w, 1))[0]
                t2 = time.perf_counter()
                psnr, _ = util.compute_psnr_and_ssim(util.convert_rgb_to_y(true_image), out, border_size=SCALE)
                t_total += time.perf_counter() - t0
                t_gpu += t2 - t1
                psnrs.append(psnr)
        res["ens%d" % ens] = {"s_per_image": t_total / len(files), "s_per_image_engine_call": t_gpu / len(files),
                              "psnr_set5": float(np.mean(psnrs))}
    eng.close()
    res["workload"] = "Set5 (5 images, LR 114..256 px), L12 x2, batch 1, host pre/post (PIL, numpy) inside the timed region"
    return res


def run_ours(args, rank, world, local_rank):
    job = Job(rank, world, local_rank)
    hd = headline(job, args)
    subs = {}
    if args.sub:
        for name, fn in (("ensemble8", sub_ensemble), ("train", sub_train), ("ds", sub_ds), ("latency", sub_latency)):
            try:
                subs[name] = fn(job, args)
            except Exception as e:  # noqa: BLE001  a failing sub-record must not take the headline down
                subs[name] = {"error": "%s: %s" % (type(e).__name__, e)}
                if world > 1:
                    raise            # ranks would desynchronise: fail loudly under torchrun
    if rank == 0:
        ms, per = hd["ms"], hd["per"]
        sustained, burst, hbm, how = measured_peaks()
        lr_px = BATCH * TILE * TILE
        tc_names = [n for n in per if n not in ("CNN1", "R-CNN1")]
        tc_ms = sum(per[n] for n in tc_names)
        tc_flops = 2.0 * MAC_PER_LR_PX_TC * lr_px
        achieved = tc_flops / (tc_ms / 1e3) / 1e12
        passes = 3 if args.precision == "f16x3" else 1
        traffic, traffic_src = ncu_traffic()
        isolated = umma_isolated(job.local)
        roofline = {
            "bound": "tensor",
            "kernel": "conv_tc_halo2_kernel (3x3 layers) / conv_tc_pair_kernel (A1+B1): the %d tcgen05 conv launches of one step" % len(tc_names),
            "achieved": achieved, "peak": sustained, "unit": "TFLOP/s", "frac": achieved / sustained,
            "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (%s); kind::f16 UMMAs issue at the bf16 rate - the pipe "
                           "measured in isolation in this run is `kind_f16_isolated`" % how,
            "kind_f16_isolated": isolated,
            "algorithmic_flop_per_launch_set": tc_flops, "launch_set_ms": tc_ms,
            "launch_ms_method": "CUDA events around every launch on the launching stream, median of >= 5 steps",
            "mma_passes": passes, "frac_of_issued_mma": achieved * passes / sustained,
            "traffic": traffic, "traffic_unit": "DRAM bytes (read + write) of the same launches of one step",
            "traffic_source": traffic_src,
            "launch_ms": {k: round(v, 4) for k, v in per.items()},
        }
        secs, cores = cpu_oracle_passes(max(3, int(args.cpu_seconds / 0.7)), 1)
        cpu_val = CPU_TILES * (SCALE * TILE) ** 2 / _median(secs) / 1e6
        line = {
            "metric": "output Mpixels/sec DCSCN L12 x2", "value": hd["value"], "unit": "Mpixels/s", "n_gpus": world,
            "steps": args.steps, "warmup": hd["warm"], "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16x3 (fp16 hi/lo split operands, fp32 accumulate; fp32-equivalent)" if passes == 3 else "f16",
            "data": "synthetic",
            "config": {"workload": "DCSCN L12 F196->48 x2 inference, batch=256 synthetic 48x48 Y-tiles per GPU "
                                   "(BASELINE.json configs[1]), weights = reference L12 x2 checkpoint",
                       "global_batch": BATCH * world, "parallelism": "dp%d (independent tiles, no collective)" % world,
                       "l2": "per-step working set (activation planes) 4.3 GB >> 126 MB L2; no explicit flush"},
            "clocks": hd["clocks"],
            "e2e": {"value": hd["e2e_value"], "unit": "Mpixels/s", "h2d_bytes_per_step": hd["h2d"], "d2h_bytes_per_step": hd["d2h"]},
            "gpu_launches": int(hd["launches"]),
            "roofline": roofline,
            "cpu_baseline": {"value": cpu_val, "unit": "Mpixels/s", "cores": cores, "kind": "port",
                             "sample": "%d passes over %d 48x48 tiles of the same workload (median pass %.2f s), torch-CPU fp32 oracle"
                                       % (len(secs), CPU_TILES, _median(secs))},
            "algorithmic_tflops": FLOP_PER_LR_PX_TOTAL * lr_px * world / (ms / args.steps / 1e3) / 1e12,
        }
        line["strict"] = hd["strict"]
        line.update(subs)
        print(json.dumps(line))
    job.close()


def run_secondary(args, rank, world, local_rank):
    """`--workload train|ds|ensemble`: one sub-record alone, as its own JSON line (for profiling runs)."""
    job = Job(rank, world, local_rank)
    fn = {"train": sub_train, "ds": sub_ds, "ensemble": sub_ensemble, "latency": sub_latency}[args.workload]
    rec = fn(job, args)
    if rank == 0:
        rec = dict(rec)
        rec.update({"n_gpus": world, "higher_is_better": True, "data": "synthetic", "scaling": "weak"})
        print(json.dumps(rec))
    job.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="f16x3", choices=["f16x3", "f16x1"])
    ap.add_argument("--cpu-seconds", type=float, default=10.0, dest="cpu_seconds")
    ap.add_argument("--no-sub", action="store_false", dest="sub", help="headline only (skip ensemble8 / train / ds / latency)")
    ap.add_argument("--workload", default="infer", choices=["infer", "train", "ds", "ensemble", "latency"],
                    help="infer = headline line with all sub-records; the others print one sub-record alone")
    ap.add_argument("--dump-outputs", default=None, dest="dump_outputs", metavar="DIR",
                    help="write the headline's output of its last timed step (rank 0) as DIR/y.npy, float32 "
                         "[256, 96, 96, 1]; the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "infer"):
        ap.error("--dump-outputs writes the headline's output: it needs --impl ours --workload infer")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # convenience: re-launch ourselves under torchrun, one process per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.workload != "infer":
        run_secondary(args, rank, world, local_rank)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
