"""bench.py — headline benchmark of the DiffBIR hot path (see BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload 512|tiled2048]
                    [--dump-outputs DIR]

A "step" is one full restoration of one synthetic image per GPU through SwinIRPipeline: SwinIR
stage 1 -> VAE encode + CLIP -> 50-step spaced sampler (cfg 4.0, ControlNet + UNet, batched
cond/uncond) -> VAE decode -> colour fix -> uint8.  Random-init SD-2.1 / SwinIR weights
(no network for checkpoints), synthetic image-like input.

  value : MPix/s with the uint8 input already resident in HBM (CUDA-event time, max over ranks)
  e2e   : the same through the public API Pipeline.run(host uint8) -> host uint8 (H2D + D2H inside)
  roofline : tcgen05 GEMM/conv kernel family — algorithmic FLOPs of every launch of one
             ControlNet+UNet forward / CUDA-event time of those launches, vs the measured bf16 peak
  cpu_baseline : the fp32 oracle port of the reference on the host cores, bounded sample
                 (1 of 50 sampler steps; SwinIR, VAE encode/decode once), extrapolated.

  tiled2048 : EVERY line (N = 1, 2, 4, 8) also restores ONE 2048x2048 image with tiled sampling
             (tile 512 / stride 256 -> 49 latent tiles, configs[3]): the tiles are sharded round-robin over
             the ranks, one NCCL all-gather of the per-tile eps per step, every rank blends + updates
             the full latent. Its MPix/s across N is the STRONG-scaling curve of the path that has a
             collective; `value` stays the 512^2 replica throughput (weak scaling, no collective).
  v21_1024_b4 : EVERY line also restores ONE batch of 4 1024^2 images with the v2.1 settings (configs[4]); at N > 1
             the 8 (image, CFG branch) forwards of a step are sharded over the ranks (all-gather of eps per step)
  phases_ms : CUDA-event time of each pipeline stage of the 512^2 image
  --dump-outputs DIR : after the timed 512^2 steps, each rank writes the uint8 image its last timed step
             returned as DIR/restored_rank<R>.npy (float32, exact). Inputs, weights and seeds are fixed, so two
             builds run with the same arguments can be compared output for output. The GEMM planner picks split-K
             plans by timing, so two runs can differ by one level on a few percent of the pixels;
             DBIR_DETERMINISTIC=1 pins batch-invariant plans and makes the bits reproducible.
  gpu_torch_baseline : the reference algorithm (oracle port) as stock PyTorch kernels on the same
             GPU, fp16 autocast, bounded sample -- informational (SURVEY 8d "GPU baseline")

Multi-GPU (torchrun, one rank per GPU): the 512x512 workload has no tiles, so ranks are
independent replicas (weak scaling, no collective); --workload tiled2048 makes the tiled run the
headline `value` instead (strong scaling).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "MPix/s end-to-end 50-step restore @512px"
SAMPLER_STEPS = 50


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    """(sustained bf16 TFLOP/s, burst bf16 TFLOP/s, HBM GB/s, source)"""
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return (d.get("bf16_tflops_sustained", 1400.0), d.get("bf16_tflops", 1590.0), d.get("hbm_gbs", 6650.0),
                "measured (MEASURED_PEAKS.json)")
    return 1400.0, 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


def host_threads() -> int:
    """Host threads the CPU arms use: every core this process may run on, whatever OMP_NUM_THREADS says
    (torchrun exports OMP_NUM_THREADS=1 to its workers)."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


_CAL = {}


def calibrated_threads():
    """Thread count for the CPU arms: the fastest of {all, 1/2, 1/4 of the host threads, 32} on a short fp32
    conv + matmul probe. Every schedulable thread is not always the fastest choice (SMT siblings, cgroup
    CPU quotas below the affinity mask: a 128-thread box ran the oracle 5x slower than a 64-thread one),
    and the baseline should be the reference's best, not its worst."""
    if _CAL:
        return _CAL["best"], _CAL["probe_ms"]
    import torch
    import torch.nn.functional as F
    n = host_threads()
    cands = sorted({c for c in (n, n // 2, n // 4, 32, 16) if 1 <= c <= n}, reverse=True)
    x = torch.randn(2, 320, 64, 64)
    w = torch.randn(320, 320, 3, 3)
    a = torch.randn(8192, 320)
    b = torch.randn(320, 1280)
    res = {}
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            F.conv2d(x, w, padding=1); a @ b
            t0 = time.perf_counter()
            for _ in range(3):
                F.conv2d(x, w, padding=1)
                a @ b
            res[c] = (time.perf_counter() - t0) / 3 * 1e3
    best = min(res, key=res.get)
    torch.set_num_threads(best)
    _CAL.update(best=best, probe_ms={str(k): round(v, 2) for k, v in res.items()})
    return best, _CAL["probe_ms"]


# ------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle port of the reference on the host cores
# ------------------------------------------------------------------------------------------
def cpu_reference_times(n_steps: int = 1, warm: int = 0, size: int = 512):
    """Times the reference algorithm (oracle port, fp32, all host threads) on a bounded sample of
    the 512x512 workload: SwinIR forward, VAE encode, `n_steps` sampler steps (2 forwards each, as
    spaced_sampler.py:156-157), VAE decode.  Returns component seconds."""
    import torch
    from diffbir_b200 import arch
    from diffbir_b200.utils.synth import make_state_dict, synthetic_lq
    from oracle import cldm as ocl
    from oracle import swinir as osw
    torch.set_num_threads(calibrated_threads()[0])
    torch.manual_seed(231)
    L = size // 8
    t = {}
    with torch.no_grad():
        ssd = make_state_dict(arch.swinir_shapes(arch.SWINIR_CFG), 1238)
        x = torch.tensor(synthetic_lq(size, size)).float().div(255).permute(0, 3, 1, 2).contiguous()
        t0 = time.perf_counter(); clean = osw.swinir_forward(ssd, x); t["swinir"] = time.perf_counter() - t0
        del ssd
        vsd = make_state_dict(arch.vae_shapes(arch.VAE_CFG), 1235)
        t0 = time.perf_counter(); c_img = ocl.vae_encode_mode(vsd, clean * 2 - 1); t["vae_encode"] = time.perf_counter() - t0
        t0 = time.perf_counter(); ocl.vae_decode(vsd, c_img / 0.18215); t["vae_decode"] = time.perf_counter() - t0
        del vsd
        usd = make_state_dict(arch.unet_shapes(arch.UNET_CFG), 1234, arch.is_zero_init)
        csd = make_state_dict(arch.unet_shapes(arch.CONTROLNET_CFG, True), 1237, arch.is_zero_init)
        xt = torch.randn(1, 4, L, L)
        ctx = torch.randn(1, 77, 1024)
        tt = torch.full((1,), 999)
        steps = []
        for i in range(warm + n_steps):
            t0 = time.perf_counter()
            ec = ocl.cldm_forward(usd, csd, xt, tt, ctx, c_img, [1.0] * 13)
            eu = ocl.cldm_forward(usd, csd, xt, tt, ctx, c_img, [1.0] * 13)
            xt = xt - 0.01 * (eu + 4.0 * (ec - eu))
            dt = time.perf_counter() - t0
            if i >= warm:
                steps.append(dt)
        t["sampler_step"] = steps
    return t, torch.get_num_threads()


def cpu_image_seconds(t, step_s):
    # the reference encodes the condition image twice (pipeline.py:117-128)
    return t["swinir"] + 2 * t["vae_encode"] + SAMPLER_STEPS * step_s + t["vae_decode"]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t, cores = cpu_reference_times(n_steps=args.steps, warm=args.warmup)
    step_s = statistics.median(t["sampler_step"])
    total = cpu_image_seconds(t, step_s)
    mpix = 512 * 512 / 1e6 / total
    sample = (f"oracle port of the reference (fp32, {cores} threads): SwinIR 512^2 {t['swinir']:.2f}s, VAE encode "
              f"{t['vae_encode']:.2f}s (x2), decode {t['vae_decode']:.2f}s measured once; {len(t['sampler_step'])} of 50 sampler "
              f"steps measured (median {step_s:.2f}s, 2 forwards each), image time extrapolated to 50 steps")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": mpix, "unit": "MPix/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": total * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BSR pipeline 512x512, 50-step spaced sampler, cfg 4.0, random-init SD2.1 UNet+ControlNet (configs[1])"},
        "cpu_baseline": {"value": mpix, "unit": "MPix/s", "cores": cores, "kind": "port", "sample": sample,
                         "component_seconds": {"swinir": t["swinir"], "vae_encode": t["vae_encode"],
                                               "vae_decode": t["vae_decode"], "sampler_step_median": step_s,
                                               "sampler_steps": t["sampler_step"]},
                         "thread_probe_ms": calibrated_threads()[1], "host_threads": host_threads(),
                         "note": ("CPU arm, independent of the GPU count: thread count = the fastest of a short probe over "
                                  "{all, 1/2, 1/4 of the host threads, 32, 16} (torchrun's OMP_NUM_THREADS=1 is overridden); "
                                  "ratios against it are only meaningful at N=1")},
        "e2e": {"value": mpix, "unit": "MPix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def kernel_census(pipe, torch, lib, nb=2, batch_invariant=None, per_shape=True):
    """Records the tensor-core launches of one ControlNet+UNet forward (batch 2 = cond/uncond of a
    512^2 image), then replays each kernel family back-to-back inside a CUDA graph and times the
    replay with CUDA events on the launching stream (steady state, same buffers as the real forward).
    Returns per-family totals and the per-shape table (per-shape numbers from per-launch events)."""
    eng = pipe.cldm.engine
    dev = eng.dev
    # nb = 2: the plans of the 512^2 loop; the tiled run pins the batch-invariant ones (batch_invariant=True)
    eng.batch_invariant = eng.deterministic if batch_invariant is None else batch_invariant
    x = torch.randn(nb, 4, 64, 64, device=dev)
    ci = torch.randn(nb, 4, 64, 64, device=dev) * 0.5
    eng.set_context(torch.randn(nb, 77, 1024, device=dev))
    eng.set_timesteps([500], nb)
    eng.load_step(0)
    two = eng.two_streams
    eng.two_streams = False                  # record on one stream
    eng.forward(x, ci, [1.0] * 13)
    torch.cuda.synchronize()
    lib.record_begin()
    eng.forward(x, ci, [1.0] * 13)
    calls = lib.record_end()
    eng.two_streams = two
    fam, shapes = {}, {}
    names = {"gemm": "gemm+conv (gemm_tc_kernel)", "conv": "gemm+conv (gemm_tc_kernel)",
             "attention": "attention (attn_fwd_kernel)"}

    def replay_ms(sel, reps=5):
        for c in sel:
            c[3]()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for c in sel:
                c[3]()
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    for fname in set(names.values()):
        sel = [c for c in calls if names[c[0]] == fname]
        if sel:
            fam[fname] = [sum(c[2] for c in sel), replay_ms(sel), len(sel)]
    by_shape = {}
    for c in calls:
        by_shape.setdefault((c[0],) + tuple(c[1]), []).append(c)
    if per_shape:
        for k, sel in by_shape.items():      # per-shape: the launches of that shape back-to-back in a graph
            shapes[k] = [sum(c[2] for c in sel), replay_ms(sel, 3), len(sel)]
    return fam, shapes


def gpu_torch_baseline(torch, dev, n_steps: int = 3):
    """Informational: the reference algorithm (oracle port = the reference's own op sequence) executed by
    stock PyTorch kernels (cuDNN / cuBLAS / SDPA-free matmul attention) on this GPU under fp16 autocast,
    on a bounded sample of the 512^2 workload; 50-step image time extrapolated. Not the product path."""
    from diffbir_b200 import arch
    from diffbir_b200.utils.synth import make_state_dict, synthetic_lq
    from oracle import cldm as ocl
    from oracle import swinir as osw

    def todev(sd):
        return {k: v.to(dev) for k, v in sd.items()}

    def timed(fn, reps=1):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            r = fn()
        e1.record()
        torch.cuda.synchronize()
        return r, e0.elapsed_time(e1) / reps

    t = {}
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        ssd = todev(make_state_dict(arch.swinir_shapes(arch.SWINIR_CFG), 1238))
        x = torch.tensor(synthetic_lq(512, 512)).float().div(255).permute(0, 3, 1, 2).contiguous().to(dev)
        osw.swinir_forward(ssd, x)
        clean, t["swinir"] = timed(lambda: osw.swinir_forward(ssd, x))
        del ssd
        vsd = todev(make_state_dict(arch.vae_shapes(arch.VAE_CFG), 1235))
        ocl.vae_encode_mode(vsd, clean.float() * 2 - 1)
        c_img, t["vae_encode"] = timed(lambda: ocl.vae_encode_mode(vsd, clean.float() * 2 - 1))
        ocl.vae_decode(vsd, c_img / 0.18215)
        _, t["vae_decode"] = timed(lambda: ocl.vae_decode(vsd, c_img / 0.18215))
        del vsd
        usd = todev(make_state_dict(arch.unet_shapes(arch.UNET_CFG), 1234, arch.is_zero_init))
        csd = todev(make_state_dict(arch.unet_shapes(arch.CONTROLNET_CFG, True), 1237, arch.is_zero_init))
        xt = torch.randn(1, 4, 64, 64, device=dev)
        ctx = torch.randn(1, 77, 1024, device=dev)
        tt = torch.full((1,), 999, device=dev)

        def step():
            ec = ocl.cldm_forward(usd, csd, xt, tt, ctx, c_img.float(), [1.0] * 13)
            eu = ocl.cldm_forward(usd, csd, xt, tt, ctx, c_img.float(), [1.0] * 13)
            return eu + 4.0 * (ec - eu)
        step()
        _, t["sampler_step"] = timed(step, n_steps)
    total_ms = t["swinir"] + 2 * t["vae_encode"] + SAMPLER_STEPS * t["sampler_step"] + t["vae_decode"]
    del usd, csd
    torch.cuda.empty_cache()
    return {"value": 512 * 512 / 1e6 / (total_ms / 1e3), "unit": "MPix/s", "ms_per_image": total_ms,
            "component_ms": t, "kind": "oracle port of the reference on stock PyTorch CUDA kernels, fp16 autocast, eager",
            "sample": f"SwinIR, VAE encode (x2 as the reference), decode once; {n_steps} sampler steps (2 forwards each) "
                      "timed and extrapolated to 50"}


class Watchdog:
    """A stalled phase must not cost the run its measured headline: past the deadline (DBIR_BENCH_DEADLINE_S, default
    1500 s; a normal run takes 3-4 minutes) rank 0 prints the line with whatever has been measured so far plus
    `"incomplete": <phase that never finished>` and every rank leaves the process."""

    def __init__(self, rank: int):
        self.rank, self.line, self.phase = rank, None, "start-up"
        self.lock, self.done = threading.Lock(), False
        self.deadline = float(os.environ.get("DBIR_BENCH_DEADLINE_S", "1500"))
        threading.Thread(target=self._watch, daemon=True).start()

    def _watch(self):
        time.sleep(self.deadline)
        with self.lock:
            if self.done:
                return
            self.done = True
            log(f"[rank {self.rank}] bench deadline ({self.deadline:.0f} s) passed in phase '{self.phase}'")
            if self.rank == 0 and self.line is not None:
                print(json.dumps(dict(self.line, incomplete=self.phase)), flush=True)
            os._exit(0 if self.line is not None else 3)

    def finish(self, line):
        with self.lock:
            if self.done:
                return
            self.done = True
            print(json.dumps(line), flush=True)


def run_leg(name: str, limit_s: int):
    """`python bench.py --leg <name>` in a child process; its last stdout line is the leg's JSON object."""
    try:
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--leg", name], capture_output=True, text=True,
                           timeout=limit_s)
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        if r.returncode == 0 and lines:
            return json.loads(lines[-1])
        return {"unavailable": f"leg exited with {r.returncode}: {(r.stderr or '')[-160:]}"}
    except subprocess.TimeoutExpired:
        return {"unavailable": f"not finished within its {limit_s} s limit"}
    except Exception as ex:
        return {"unavailable": repr(ex)[:200]}


def leg_main(name: str):
    if name == "gpu_torch":
        import torch
        torch.cuda.set_device(0)
        print(json.dumps(gpu_torch_baseline(torch, "cuda:0")))
    elif name == "cpu":
        t, cores = cpu_reference_times(n_steps=1)
        step_s = t["sampler_step"][0]
        total = cpu_image_seconds(t, step_s)
        print(json.dumps({"value": 512 * 512 / 1e6 / total, "unit": "MPix/s", "cores": cores, "kind": "port",
                          "thread_probe_ms": calibrated_threads()[1], "host_threads": host_threads(),
                          "sample": (f"oracle port, fp32: SwinIR {t['swinir']:.2f}s + VAE encode 2x{t['vae_encode']:.2f}s + "
                                     f"1 of 50 sampler steps ({step_s:.2f}s, 2 forwards) x50 + VAE decode {t['vae_decode']:.2f}s "
                                     f"= {total:.1f}s per 512^2 image (extrapolated)")}))
    else:
        raise SystemExit(f"unknown leg {name}")


def run_ours(args):
    import numpy as np
    import torch
    from diffbir_b200 import lib
    from diffbir_b200.sampler import sampler as sampler_mod
    from diffbir_b200.utils.synth import RUN_DEFAULTS, build_synthetic_pipeline, synthetic_lq

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    lib.load()
    dog = Watchdog(rank)
    headline_tiled = args.workload == "tiled2048"
    t_build = time.time()
    pipe = build_synthetic_pipeline(dev, seed=1234)
    log(f"[rank {rank}] pipeline built in {time.time() - t_build:.1f}s")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(vals):
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    # ------------------------------------------------------------------ 512^2 replicas
    kw = dict(RUN_DEFAULTS)
    lq = synthetic_lq(512, 512, seed=rank)            # replicas restore different images
    lq_pinned = torch.from_numpy(lq).pin_memory()
    lq_dev = lq_pinned.to(dev)

    def one(device_resident: bool):
        torch.manual_seed(231)
        if device_resident:
            return pipe.run_device(lq_dev, **kw)
        return pipe.run(lq_pinned, **kw)

    log(f"[rank {rank}] 512^2: warm-up")
    for _ in range(max(args.warmup, 3)):              # W >= 3 (timing rules)
        one(True)
    out = one(False)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    n0 = lib.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.nvtx.range_push("dbir_timed")      # ncu --nvtx --nvtx-include "dbir_timed/" profiles exactly this region
    e0.record()
    for _ in range(args.steps):
        restored = one(True)
    e1.record()
    torch.cuda.nvtx.range_pop()
    barrier()
    dev_ms = e0.elapsed_time(e1)
    launches = lib.launches() - n0
    if args.dump_outputs:
        dump_dir = Path(args.dump_outputs)
        dump_dir.mkdir(parents=True, exist_ok=True)
        np.save(dump_dir / f"restored_rank{rank}.npy", restored.cpu().numpy().astype(np.float32))
    # end-to-end through the public API (pinned host uint8 in, host uint8 out)
    barrier()
    w0 = time.perf_counter()
    for _ in range(args.steps):
        out = one(False)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - w0) * 1e3
    barrier()
    clk = clocks.stop() if rank == 0 else None
    # phase breakdown of one more image (CUDA events at the stage boundaries)
    pipe.marks = []
    one(True)
    torch.cuda.synchronize()
    phases = pipe.phases_ms()
    pipe.marks = None
    dev_ms, e2e_ms = reduce_max([dev_ms, e2e_ms])
    mpix_512 = world * args.steps * 512 * 512 / 1e6
    value_512, e2e_512 = mpix_512 / (dev_ms / 1e3), mpix_512 / (e2e_ms / 1e3)

    log(f"[rank {rank}] 512^2 timed: {dev_ms / args.steps:.1f} ms per image")
    wl_512 = "BSR pipeline 512x512, 50-step spaced sampler, cfg 4.0, random-init SD2.1 UNet+ControlNet (configs[1])"
    line = {
        "metric": METRIC, "value": value_512, "unit": "MPix/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 operands / f32 accumulate" if lib.operand_dtype() == torch.float16 else "bf16 operands / f32 accumulate",
        "data": "synthetic",
        "config": {
            "workload": wl_512, "images_per_gpu_per_step": 1, "sampler_steps": SAMPLER_STEPS,
            "parallelism": "independent replicas, no collective (the sharded path with a collective is the tiled2048 block)",
            "l2": "no flush needed: each forward streams 2.6 GB of weights >> 126 MB L2",
        },
        "e2e": {"value": e2e_512, "unit": "MPix/s", "h2d_bytes_per_step": int(lq.nbytes), "d2h_bytes_per_step": int(out.nbytes),
                "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": int(launches),
        "clocks": clk,
        "phases_ms": phases,
        "batch4_512": None, "tiled2048": None, "v21_1024_b4": None, "roofline": None, "cpu_baseline": None,
        "gpu_torch_baseline": None,
    }
    dog.line, dog.phase = line, "batch4_512"
    # ------------------------------------------------------------------ 512^2, four images per call (throughput mode)
    b4 = None
    if not args.no_batch4:
        lq4 = torch.from_numpy(synthetic_lq(512, 512, batch=4, seed=100 + rank)).to(dev)
        torch.manual_seed(231)
        pipe.run_device(lq4, **dict(kw, steps=3))                # warm-up: plans and graphs of the batch-8 forward
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.manual_seed(231)
        c0.record()
        pipe.run_device(lq4, **kw)
        c1.record()
        barrier()
        (b4_ms,) = reduce_max([c0.elapsed_time(c1)])
        b4 = {"value": world * 4 * 512 * 512 / 1e6 / (b4_ms / 1e3), "unit": "MPix/s", "images_per_gpu_per_call": 4,
              "ms_per_call": b4_ms, "scaling": "weak",
              "note": "same workload as `value` with 4 images per Pipeline.run call (8 forwards per graph replay): the "
                      "throughput mode of a folder run; the headline `value` keeps one image per call (latency mode)"}

    log(f"[rank {rank}] batch-4 block done")
    line["batch4_512"], dog.phase = b4, "tiled2048"
    # ------------------------------------------------------------------ tiled 2048^2 (sharded, all-gather per step)
    tiled = None
    if not args.no_tiled:
        tkw = dict(RUN_DEFAULTS, cldm_tiled=True, cldm_tile_size=512, cldm_tile_stride=256)
        lq_t = synthetic_lq(2048, 2048, seed=0)       # ONE image, the same on all ranks
        lq_t_pinned = torch.from_numpy(lq_t).pin_memory()
        lq_t_dev = lq_t_pinned.to(dev)
        torch.manual_seed(231)
        pipe.run_device(lq_t_dev, **dict(tkw, steps=3))          # warm-up: plans, graph capture, NCCL channels
        barrier()
        sampler_mod.Sampler.time_collective = True
        pipe.marks = []
        t_ms, t_e2e_ms = [], []
        for _ in range(args.tiled_images):
            barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.manual_seed(231)
            a0.record()
            pipe.run_device(lq_t_dev, **tkw)
            a1.record()
            barrier()
            t_ms.append(a0.elapsed_time(a1))
        tphases = pipe.phases_ms()
        smp = pipe.last_sampler
        ag = [a.elapsed_time(b) for a, b in smp.last_stats.get("allgather_events", [])]
        stats = dict(smp.last_stats)
        pipe.marks = None
        sampler_mod.Sampler.time_collective = False
        for _ in range(args.tiled_images):
            barrier()
            w0 = time.perf_counter()
            torch.manual_seed(231)
            out_t = pipe.run(lq_t_pinned, **tkw)
            torch.cuda.synchronize()
            t_e2e_ms.append((time.perf_counter() - w0) * 1e3)
        barrier()
        t_total, t_e2e_total, ag_mean, loop_ms, serial_ms = reduce_max(
            [sum(t_ms), sum(t_e2e_ms), (sum(ag) / len(ag)) if ag else 0.0, tphases.get("sampler_loop", 0.0),
             sum(v for k, v in tphases.items() if k != "sampler_loop")])
        counts = torch.zeros(world, device=dev, dtype=torch.float64)
        counts[rank] = stats.get("units_this_rank", 0)
        if world > 1:
            dist.all_reduce(counts)
        mp = args.tiled_images * 2048 * 2048 / 1e6
        tiled = {"value": mp / (t_total / 1e3), "unit": "MPix/s", "scaling": "strong", "images": args.tiled_images,
                 "ms_per_image": t_total / args.tiled_images,
                 "e2e": {"value": mp / (t_e2e_total / 1e3), "unit": "MPix/s", "h2d_bytes_per_step": int(lq_t.nbytes),
                         "d2h_bytes_per_step": int(out_t.nbytes)},
                 "tiles": int(stats.get("tiles", 0)), "tile_forwards_per_rank": [int(c) for c in counts.tolist()],
                 "tile_forwards_per_step_max_rank": int(max(counts.tolist())),
                 "allgather_ms_per_step": ag_mean, "allgather_bytes_per_rank_per_step":
                     int(((2 * stats.get("tiles", 0) + world - 1) // world) * 4 * 64 * 64 * 4) if world > 1 else 0,
                 "sampler_loop_ms": loop_ms, "replicated_serial_ms": serial_ms,
                 "phases_ms_rank0": tphases,
                 "workload": "Tiled BSR 2048x2048, tile 512 stride 256: the 98 (latent tile, CFG branch) forwards of a step sharded "
                             "round-robin over the ranks, one NCCL all-gather of per-tile eps per step (configs[3]); SwinIR / VAE / "
                             "CLIP replicated"}

    log(f"[rank {rank}] tiled-2048 block done")
    line["tiled2048"], dog.phase = tiled, "v21_1024_b4"
    # ------------------------------------------------------------------ v2.1 1024^2 batch 4 (configs[4])
    v21 = None
    if not args.no_v21:
        from diffbir_b200.model import Diffusion
        B5 = 4
        vkw = dict(RUN_DEFAULTS, pos_prompt="a photo of a mountain lake at sunrise, highly detailed, sharp focus")
        lq5 = synthetic_lq(1024, 1024, batch=B5, seed=5)           # the same 4 images on every rank
        lq5_pinned = torch.from_numpy(lq5).pin_memory()
        lq5_dev = lq5_pinned.to(dev)
        eps_diffusion, pipe.diffusion = pipe.diffusion, Diffusion(linear_start=0.00085, linear_end=0.0120, timesteps=1000,
                                                                  parameterization="v", zero_snr=True)
        pipe.shard_batch = world > 1
        torch.manual_seed(231)
        pipe.run_device(lq5_dev, **dict(vkw, steps=3))             # warm-up: plans, graphs, NCCL
        barrier()
        sampler_mod.Sampler.time_collective = True
        pipe.marks = []
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.manual_seed(231)
        b0.record()
        pipe.run_device(lq5_dev, **vkw)
        b1.record()
        barrier()
        v_ms = b0.elapsed_time(b1)
        vphases = pipe.phases_ms()
        vstats = dict(pipe.last_sampler.last_stats)
        vag = [a.elapsed_time(b) for a, b in vstats.get("allgather_events", [])]
        pipe.marks = None
        sampler_mod.Sampler.time_collective = False
        barrier()
        w0 = time.perf_counter()
        torch.manual_seed(231)
        out5 = pipe.run(lq5_pinned, **vkw)
        torch.cuda.synchronize()
        v_e2e_ms = (time.perf_counter() - w0) * 1e3
        barrier()
        pipe.shard_batch = False
        pipe.diffusion = eps_diffusion
        v_ms, v_e2e_ms, v_loop, v_ag = reduce_max([v_ms, v_e2e_ms, vphases.get("sampler_loop", 0.0),
                                                   (sum(vag) / len(vag)) if vag else 0.0])
        mp5 = B5 * 1024 * 1024 / 1e6
        v21 = {"value": mp5 / (v_ms / 1e3), "unit": "MPix/s", "scaling": "strong", "ms_per_batch": v_ms,
               "e2e": {"value": mp5 / (v_e2e_ms / 1e3), "unit": "MPix/s", "h2d_bytes_per_step": int(lq5.nbytes),
                       "d2h_bytes_per_step": int(out5.nbytes)},
               "forwards_per_step_rank0": int(vstats.get("forwards_per_step", 0)), "forwards_per_step_total": 2 * B5,
               "allgather_ms_per_step": v_ag, "sampler_loop_ms": v_loop, "phases_ms_rank0": vphases,
               "workload": "v2.1 (v-parameterization, zero terminal SNR) caption-conditioned BSR 1024x1024, 50-step spaced, cfg 4.0, "
                           "batch 4: the 8 (image, CFG branch) forwards of a step sharded round-robin over the ranks, one NCCL "
                           "all-gather of eps per step (configs[4]); SwinIR / VAE / CLIP replicated; fp16 operands (the bf16 "
                           "build is DBIR_OPERANDS=bf16)"}

    log(f"[rank {rank}] v2.1 block done")
    line["v21_1024_b4"], dog.phase = v21, "roofline census"
    if rank != 0:
        dog.done = True
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel family (live CUDA events) --------------------------
    peak_tf, peak_burst, _, peak_src = measured_peaks()
    fam, shapes = kernel_census(pipe, torch, lib)
    gname = "gemm+conv (gemm_tc_kernel)"
    gf, gms, gn = fam[gname]
    achieved = gf / (gms * 1e-3) / 1e12
    forward_ms = sum(v[1] for v in fam.values())
    traffic = None
    for cand in ("r02_ncu_full_summary.json", "r01_ncu_full_summary.json"):
        tpath = ROOT / "profiles" / cand
        if tpath.exists():       # dram bytes (read + write) per launch from the committed `ncu --set full` capture
            rows = [r for r in json.loads(tpath.read_text()) if "gemm_tc_kernel" in r["kernel"]]
            if rows:
                traffic = {"dram_bytes_per_launch_mean": sum(r["dram_bytes"] for r in rows) / len(rows),
                           "l2_to_sm_bytes_per_launch_mean": sum(r["l2_to_sm_bytes"] for r in rows) / len(rows),
                           "launches": len(rows), "source": f"profiles/{cand}"}
                break
    att = fam.get("attention (attn_fwd_kernel)", [0, 1, 0])
    roof = {"bound": "tensor", "kernel": gname, "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
            "frac": achieved / peak_tf, "frac_of_burst_peak": achieved / peak_burst, "peak_burst": peak_burst,
            "peak_note": "frac = achieved / sustained cuBLAS bf16 peak (the family is timed inside a long step); "
                         "frac_of_burst_peak uses the isolated-kernel figure",
            "traffic": traffic, "peak_source": peak_src,
            "launches_per_forward": gn, "algorithmic_gflop_per_forward": gf / 1e9,
            "kernel_ms_per_forward": gms,
            "attention": {"achieved": att[0] / (att[1] * 1e-3) / 1e12, "frac": att[0] / (att[1] * 1e-3) / 1e12 / peak_tf,
                          "ms_per_forward": att[1]},
            "tensor_kernel_ms_per_forward": forward_ms}
    if not args.no_tiled:
        # the same family in the regime of the sharded tiled run: 14 tile-forwards per replay = the per-rank batch
        # of 49 tiles x 2 CFG branches on 8 GPUs, batch-invariant plans (no split-K)
        tfam, _ = kernel_census(pipe, torch, lib, nb=14, batch_invariant=True, per_shape=False)
        tg, ta = tfam[gname], tfam.get("attention (attn_fwd_kernel)", [0, 1, 0])
        roof["tiled_regime"] = {
            "forwards_per_replay": 14, "gemm_tflops": tg[0] / (tg[1] * 1e-3) / 1e12, "gemm_frac": tg[0] / (tg[1] * 1e-3) / 1e12 / peak_tf,
            "gemm_ms": tg[1], "attention_tflops": ta[0] / (ta[1] * 1e-3) / 1e12, "attention_frac": ta[0] / (ta[1] * 1e-3) / 1e12 / peak_tf,
            "attention_ms": ta[1], "note": "same kernel families at the per-rank batch of the 8-GPU tiled-2048 run (batch-invariant plans)"}
    census = Path(tempfile.mkdtemp(prefix="dbir_bench_")) / "kernel_census.csv"      # the source tree may be read-only
    with open(census, "w") as f:
        f.write("kind,shape,launches,gflop,ms,tflops\n")
        for k, (fl, ms, n) in sorted(shapes.items(), key=lambda kv: -kv[1][1]):
            f.write(f"{k[0]},{'x'.join(map(str, k[1:]))},{n},{fl / 1e9:.2f},{ms:.4f},{fl / (ms * 1e-3) / 1e12 if ms > 0 else 0:.1f}\n")
    log(f"[rank 0] kernel census done: {census}")
    line["roofline"], dog.phase = roof, "baselines"
    # ---- baselines on the same box, N = 1 only ------------------------------------------------
    cpu = gpu_base = None
    if world == 1 and not args.no_cpu_baseline:
        # The two informational baselines run as child processes with a time limit each: a stall in one of them
        # (a cold cuDNN page-in took 6 minutes on one box) must not cost the line its measured numbers.
        del pipe
        torch.cuda.empty_cache()
        gpu_base = run_leg("gpu_torch", 240)
        log(f"[rank 0] GPU torch baseline: {str(gpu_base)[:200]}")
        cpu = run_leg("cpu", 300)
        log(f"[rank 0] CPU baseline: {str(cpu)[:200]}")
    line["cpu_baseline"], line["gpu_torch_baseline"] = cpu, gpu_base
    if headline_tiled and tiled is not None:
        line.update(metric="MPix/s end-to-end 50-step restore, tiled 2048px", value=tiled["value"],
                    ms_per_step=tiled["ms_per_image"], scaling="strong", e2e=tiled["e2e"],
                    steps=args.tiled_images)
        line["config"]["workload"] = tiled["workload"]
        line["config"]["parallelism"] = "tiles sharded round-robin + all-gather"
        line["replicas512"] = {"value": value_512, "e2e": e2e_512, "ms_per_step": dev_ms / args.steps}
    dog.finish(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="512", choices=["512", "tiled2048"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU and GPU-torch baseline legs")
    ap.add_argument("--no-tiled", action="store_true", help="skip the tiled-2048 block")
    ap.add_argument("--no-v21", action="store_true", help="skip the v2.1 1024^2 batch-4 block")
    ap.add_argument("--no-batch4", action="store_true", help="skip the 4-images-per-call 512^2 block")
    ap.add_argument("--tiled-images", type=int, default=1)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step returned to DIR/<name>.npy (float32)")
    ap.add_argument("--leg", default="", help=argparse.SUPPRESS)      # internal: one baseline leg in a child process
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.leg:
        leg_main(args.leg)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
