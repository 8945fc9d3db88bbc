#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json): Stable Diffusion v1-4 UNet, W4A8
(sm_abit 16, split shortcut), 50-step PLMS with classifier-free guidance, 8 images per GPU.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torch.distributed.run)
    python bench.py --impl reference ...                     (CPU arm: the oracle port of the reference path)
    python bench.py ... --dump-outputs DIR                   (also write the last timed step's outputs as DIR/*.npy)

A "step" is ONE denoising step of the batch: one UNet evaluation at batch 16 (8 images x [uncond, cond])
through the CUDA engine + the fused sampler update.  50 PLMS steps cost 51 UNet evaluations
(ldm/models/diffusion/plms.py:222-227), so images/s = 8 * N / (51 * step time).

Prints ONE JSON line (rank 0).  Weights are seeded synthetic (no checkpoints offline), activation
quantizers come from tests/golden/calib_sd_v1.json (reference 'max' quick-init on one seeded batch).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "q-diffusion_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

# BASELINE.json configs (SURVEY section 0 / 8d).  `evals` = UNet evaluations per image batch; `gop` = algorithmic integer
# GOP of one UNet evaluation of one image (2 x MACs of the conv/linear layers + attention QK^T and PV, SURVEY Appendix B).
WORKLOADS = {
    "sd_v1": dict(images_per_gpu=8, cfg=7.5, sampler="plms", evals=51, gop=803.3, sched=(0.00085, 0.0120),
                  desc="SD v1-4 UNet (860M) W4A8 asymmetric, sm_abit 16, split shortcut; PLMS-50 + CFG 7.5; "
                       "8 images/GPU -> UNet batch 16, 64x64x4 latents, 77x768 context"),
    "cifar10": dict(images_per_gpu=256, cfg=0.0, sampler="generalized", evals=100, gop=12.44, sched=None,
                    desc="CIFAR-10 DDIM UNet (35.7M) W4A8 symmetric, split shortcut; 100 DDIM steps (quad schedule, eta 0); "
                         "256 images/GPU, 32x32x3"),
    "lsun_bedroom": dict(images_per_gpu=64, cfg=0.0, sampler="ddim", eta=1.0, evals=200, gop=202.4, sched=(0.0015, 0.0195),
                         desc="LSUN-bedroom LDM-4 UNet (274M) W4A8 symmetric; 200 DDIM steps, eta 1; 64 images/GPU, 64x64x3 latents"),
    "lsun_church": dict(images_per_gpu=32, cfg=0.0, sampler="ddim", eta=0.0, evals=500, gop=41.85, sched=(0.0015, 0.0155),
                        desc="LSUN-church LDM-8 UNet (295M) W8A8 asymmetric; -c 400 => 500 DDIM steps (util.py:47-55); "
                             "32 images/GPU, 32x32x4 latents"),
}
WORKLOAD = "sd_v1"            # default headline; --workload selects another BASELINE config
IMAGES_PER_GPU = 8
UNET_EVALS_PER_IMAGE_BATCH = 51          # 50 PLMS steps (first step calls the UNet twice)
GOP_PER_IMAGE_EVAL = 803.3               # SURVEY 8(d): 401.64 GMAC per UNet evaluation of one image
CFG_SCALE = 7.5


def select_workload(name):
    global WORKLOAD, IMAGES_PER_GPU, UNET_EVALS_PER_IMAGE_BATCH, GOP_PER_IMAGE_EVAL, CFG_SCALE
    w = WORKLOADS[name]
    WORKLOAD, IMAGES_PER_GPU, UNET_EVALS_PER_IMAGE_BATCH = name, w["images_per_gpu"], w["evals"]
    GOP_PER_IMAGE_EVAL, CFG_SCALE = w["gop"], w["cfg"]
    return w


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(bf16_burst=p["bf16_tflops"], bf16_sustained=p["bf16_tflops_sustained"], hbm=p["hbm_gbs"],
                    source="MEASURED_PEAKS.json")
    return dict(bf16_burst=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region (B200_PROFILING.md recipe), sampled through NVML
    (same counters as the nvidia-smi query, but fast enough to get several samples inside a sub-second region)."""

    def __init__(self, index):
        self.rows, self.stop, self.index = [], False, index
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                     "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                     "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            while not self.stop:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((sm, mx, [n for n, bit in names.items() if r & bit]))
                time.sleep(0.02)
        except Exception as e:   # NVML unavailable: fall back to nvidia-smi polling
            q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            while not self.stop:
                try:
                    out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                         capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                    self.rows.append((int(out[0]), int(out[1]), [n for i, n in enumerate(names) if out[2 + i].strip().lower().startswith("active")]))
                except Exception:
                    pass
                time.sleep(0.05)

    def __enter__(self):
        self.th.start()
        time.sleep(0.05)
        return self

    def __exit__(self, *a):
        self.stop = True
        self.th.join(timeout=6)

    def summary(self):
        sm = sorted(r[0] for r in self.rows)
        reasons = sorted({n for r in self.rows for n in r[2]})
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max((r[1] for r in self.rows), default=None),
                    reasons=reasons, samples=len(self.rows))


def host_threads(cap=32):
    """CPU threads this process may really use: affinity mask and cgroup quota, not os.cpu_count() (the GPU boxes
    report 128+ logical CPUs to a container that owns far fewer; 128 torch threads there ran the oracle 10-50x slower)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                quota = int(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                period = int(f.read())
            if quota > 0:
                n = min(n, max(1, quota // period))
        except (OSError, ValueError):
            pass
    return max(1, min(n, cap))


def unet_evals_per_image():
    """UNet evaluations one image costs: `evals` sampler calls, doubled by classifier-free guidance."""
    return UNET_EVALS_PER_IMAGE_BATCH * (2 if CFG_SCALE else 1)


def cpu_eval_seconds(ckpt, batch=1, seed=99):
    """One UNet evaluation of the current workload at `batch` on the host cores through the oracle port of the reference's
    fake-quant fp32 path (the reference itself cannot travel to the GPU box: SURVEY 8c)."""
    from oracle import synth_cfg
    from qdiff_b200 import synth
    x, t, ctx = synth.calib_inputs(WORKLOAD, batch=batch, seed=seed)
    with torch.no_grad():
        t0 = time.time()
        synth_cfg.oracle_forward(WORKLOAD, ckpt, x, t, ctx)
        return time.time() - t0


def cpu_baseline(ckpt=None, budget_s=25.0):
    """The reference's CPU path on a BOUNDED sample (about `budget_s` seconds): UNet evaluations at batch 1, as many as fit;
    images/s = 1 / (evaluations per image x seconds per evaluation)."""
    import contextlib
    from qdiff_b200 import synth
    if ckpt is None:
        with contextlib.redirect_stdout(sys.stderr):
            _, ckpt = synth.full_ckpt(WORKLOAD)
    ckpt = {k: (v.float() if k.endswith(".alpha") else v.cpu()) for k, v in ckpt.items()}
    times, t_start = [], time.time()
    while not times or (time.time() - t_start + min(times) < budget_s and len(times) < 8):
        times.append(cpu_eval_seconds(ckpt, 1, seed=99 + len(times)))
    t_eval = min(times)
    n = unet_evals_per_image()
    return dict(value=1.0 / (n * t_eval), unit="images/s", cores=torch.get_num_threads(), kind="port",
                sample=f"{len(times)} UNet evaluation(s) at batch 1 ({t_eval:.2f} s best) of the {n} one image needs; oracle "
                       "port of the reference fake-quant fp32 path (the reference itself is not on the GPU box)",
                unet_eval_s=t_eval)


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path (oracle port) on the host cores, same
    metric / config as the GPU arm.  One step = a bounded sample of one denoising step: ONE UNet evaluation at batch 2
    (one image x [uncond, cond]) for guided workloads, batch 1 otherwise, scaled to the step's UNet batch; the scaling is
    stated in the line.  --true-batch times one evaluation at the GPU arm's full UNet batch instead (minutes for SD)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(host_threads())
    import contextlib
    from qdiff_b200 import synth
    w = select_workload(args.workload)
    with contextlib.redirect_stdout(sys.stderr):
        _, ckpt = synth.full_ckpt(WORKLOAD)
    ckpt = {k: (v.float() if k.endswith(".alpha") else v.cpu()) for k, v in ckpt.items()}
    unet_batch = IMAGES_PER_GPU * (2 if CFG_SCALE else 1)
    sample_batch = unet_batch if args.true_batch else (2 if CFG_SCALE else 1)
    times, t_start = [], time.time()
    for i in range(args.warmup + args.steps):
        dt = cpu_eval_seconds(ckpt, sample_batch, seed=7 + i)
        if i >= args.warmup:
            times.append(dt)
        if time.time() - t_start > 150 and times:
            break
    t_eval = sum(times) / len(times)
    ms_per_step = t_eval * (unet_batch / sample_batch) * 1e3
    value = IMAGES_PER_GPU / (UNET_EVALS_PER_IMAGE_BATCH * ms_per_step * 1e-3)
    sample = (f"{len(times)} x 1 UNet evaluation at batch {sample_batch} ({t_eval:.2f} s mean)" +
              ("" if sample_batch == unet_batch else f", scaled x{unet_batch // sample_batch} to the batch-{unet_batch} step"))
    cb = dict(value=value, unit="images/s", cores=torch.get_num_threads(), kind="port", sample=sample, unet_eval_s=t_eval)
    print(json.dumps({
        "impl": "reference", "metric": "images_per_sec", "value": value, "unit": "images/s", "n_gpus": args.gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "fp32 fake-quant (reference simulation)", "data": "synthetic",
        "config": {"workload": w["desc"],
                   "step": f"1 denoising step = 1 UNet evaluation at batch {unet_batch} (CPU arm: {sample})",
                   "host_threads": torch.get_num_threads()},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def gemm_roofline(prog, pk):
    """Replay the recorded per-step program op by op; CUDA events around every INT8 GEMM launch (default stream =
    the stream the engine launches on).  achieved = sum(2*M*N*K) / sum(duration)."""
    from qdiff_b200 import _lib
    first = prog.n_static
    gemm_ids = {i for i in range(first, prog.nops) if prog.op_kinds[i] == _lib.QD_OP_GEMM}
    prog.run_range(0, prog.nops)  # warm
    torch.cuda.synchronize()
    evs = []
    for i in range(first, prog.nops):
        if i in gemm_ids:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            prog.run_range(i, i + 1)
            e1.record()
            evs.append((i, e0, e1))
        else:
            prog.run_range(i, i + 1)
    torch.cuda.synchronize()
    tot_ms = sum(e0.elapsed_time(e1) for _, e0, e1 in evs)
    tot_ops = sum(prog.op_flops[i] for i, _, _ in evs)
    achieved = tot_ops / (tot_ms * 1e-3) / 1e12
    peak = 2.0 * pk["bf16_sustained"]
    # DRAM bytes per GEMM launch (dram__bytes_read.sum + dram__bytes_write.sum, mean over one step's launches): from the
    # ncu pass over this same command committed under profiles/ (tools/launch_summary.py --traffic), else null
    traffic, tsrc = None, None
    tf = os.path.join(ROOT, "profiles", f"r02_roofline_traffic_{WORKLOAD}.json")
    if os.path.exists(tf):
        with open(tf) as f:
            tj = json.load(f)
        traffic, tsrc = tj.get("gemm_dram_bytes_per_launch"), tj.get("source")
    return dict(bound="tensor", achieved=achieved, peak=peak, unit="TOP/s", frac=achieved / peak, traffic=traffic,
                traffic_source=tsrc,
                kernel="gemm_i8_kernel (tcgen05.mma kind::i8)", launches=len(evs), gemm_ms_per_step=tot_ms,
                algorithmic_ops_per_step=tot_ops,
                peak_source=f"2 x bf16_tflops_sustained ({pk['source']}); INT8 dense = 2x bf16 on sm_100a",
                note="events bracket each launch individually (serialised, includes launch gaps)")


def write_dumps(out_dir, arrays, limit=64 << 20):
    """DIR/<name>.npy per array; the workloads' outputs are a few MB, far below `limit` (64 MB in all)."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > limit:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {limit}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="sd_v1", choices=sorted(WORKLOADS),
                    help="BASELINE.json config: sd_v1 (cfg 4, the headline), cifar10 (cfg 2), lsun_bedroom (cfg 3), lsun_church (cfg 5)")
    ap.add_argument("--true-batch", action="store_true", help="reference arm: time the full UNet batch instead of a scaled sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels individually (for ncu launch lists)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0's shard) as DIR/<name>.npy, float32: x_prev "
                         "(the sampler's x_{t-1}), eps (the UNet output; [uncond; cond] when guided) and, for PLMS, e_t "
                         "(the guided eps the sampler keeps); every input is seeded, so equal arguments give equal inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the CUDA path's outputs (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference_arm(args)
    w = select_workload(args.workload)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: qdiff_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if dist is not None:
        dist.barrier()
    from qdiff_b200 import _lib, samplers, synth
    L = _lib.lib()

    import contextlib
    with contextlib.redirect_stdout(sys.stderr):   # the reference-compatible loaders print; stdout carries ONE JSON line
        qnn, ckpt = synth.build_qnn(WORKLOAD, cuda_graph=not args.no_graph)
    spec = synth.SPECS[WORKLOAD]
    B = IMAGES_PER_GPU
    guided = bool(CFG_SCALE)
    cfg_dedup = guided and os.environ.get("QDIFF_CFG_DEDUP", "1") != "0"
    UB = B * (2 if guided else 1)                # UNet batch of one step
    # every rank draws the FULL batch from the same seed and keeps its shard (N-rank == 1-rank results)
    from qdiff_b200 import dist as qdist
    lat_shape = (world * B,) + tuple(spec["in_shape"])
    extra = [(world * B,) + tuple(spec["ctx"])] if spec["ctx"] else []
    shards = qdist.shard_like_single_process(lat_shape, 42, rank, world, extra_shapes=extra)
    x_host = shards[0].pin_memory()
    c_host = None
    if spec["ctx"]:
        uc = torch.randn(1, *spec["ctx"], generator=torch.Generator().manual_seed(43)).expand(B, *spec["ctx"])
        c_host = (torch.cat([uc, shards[1]]) if guided else shards[1]).contiguous().pin_memory()   # [uncond; cond] as plms.py:187
    # ---- per-step constants of the workload's sampler (steady state of the loop)
    if w["sampler"] == "generalized":            # CIFAR script: quadratic schedule, 100 steps (sample_diffusion_ddim.py:294-301)
        import numpy as np
        seq = [int(v) for v in list(np.linspace(0, np.sqrt(1000 * 0.8), UNET_EVALS_PER_IMAGE_BATCH) ** 2)]
        betas = torch.from_numpy(np.linspace(0.0001, 0.02, 1000, dtype=np.float64)).float()
        acp = (1 - torch.cat([torch.zeros(1), betas])).cumprod(dim=0)
        ts = list(reversed(seq))
        nxt_t = list(reversed([-1] + seq[:-1]))
        alpha = [(float(acp[i + 1]), float(acp[j + 1])) for i, j in zip(ts, nxt_t)]
        sigma = [0.0] * len(ts)
        coef, olds_n = (1.0, 0, 0, 0), 0
    else:
        sched = samplers.Schedule("linear", 1000, *w["sched"])
        sampler = (samplers.PLMSSampler if w["sampler"] == "plms" else samplers.DDIMSampler)(qnn, sched)
        # custom steps as the scripts pass them: PLMS 50; DDIM -c 200 (bedroom) / -c 400, which the uniform discretisation
        # turns into 1000 // (1000 // 400) = 500 steps (util.py:47-55, SURVEY Appendix D Q6)
        sampler.make_schedule(50 if w["sampler"] == "plms" else {200: 200, 500: 400}[UNET_EVALS_PER_IMAGE_BATCH],
                              ddim_eta=w.get("eta", 0.0))
        ts = list(reversed(sampler.ddim_timesteps.tolist()))
        n = len(ts)
        alpha = [(float(sampler.ddim_alphas[n - 1 - i]), float(sampler.ddim_alphas_prev[n - 1 - i])) for i in range(n)]
        sigma = [float(sampler.ddim_sigmas[n - 1 - i]) for i in range(n)]
        coef, olds_n = (samplers.PLMSSampler._AB[3], 3) if w["sampler"] == "plms" else ((1.0, 0, 0, 0), 0)
    if w["sampler"] != "generalized" and len(ts) != (50 if w["sampler"] == "plms" else UNET_EVALS_PER_IMAGE_BATCH):
        raise SystemExit(f"schedule has {len(ts)} steps, expected {UNET_EVALS_PER_IMAGE_BATCH}")

    x = x_host.to(dev)
    ctx = c_host.to(dev) if c_host is not None else None
    nxt = torch.empty_like(x)
    e_t = torch.empty_like(x)
    gen = torch.Generator(device=dev).manual_seed(44)     # PLMS history and the eta > 0 noise: same draws on every run
    old = [torch.randn(x.shape, device=dev, generator=gen) for _ in range(3)]

    def step(i, x_in, nxt, ctx_dev):
        """One denoising step in the loop's steady state (PLMS: multistep order 4, 47 of the 50 steps): one UNet evaluation
        at the step's UNet batch through QuantModel.__call__ + the fused sampler update (+ the step's noise when eta > 0)."""
        k = i % len(ts)
        if guided and cfg_dedup:       # the engine's guided entry point: [x; x] is never materialised, the shared prefix runs once
            eps = qnn.forward_cfg(x_in, torch.full((B,), int(ts[k]), device=dev, dtype=torch.long), ctx_dev)
        else:
            t = torch.full((UB,), int(ts[k]), device=dev, dtype=torch.long)
            eps = qnn(torch.cat([x_in, x_in]) if guided else x_in, t, ctx_dev)
        a_t, a_prev = alpha[k]
        noise = torch.randn(x_in.shape, device=dev, generator=gen) if sigma[k] != 0.0 else None
        samplers._step(x_in, eps, nxt, a_t=a_t, a_prev=a_prev, sigma=sigma[k], cfg_scale=CFG_SCALE, coef=coef,
                       olds=tuple(old[:olds_n]) + (None,) * (3 - olds_n), eps_out=e_t if olds_n else None, noise=noise)
        return eps

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i, x, nxt, ctx)
    barrier()
    launches0 = L.qd_launch_count()
    with ClockSampler(local) as clocks:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.profiler.start()    # no-op unless run under `ncu --profile-from-start off` (profiles/: launch list)
        e0.record()
        for i in range(args.steps):
            eps = step(args.warmup + i, x, nxt, ctx)
        e1.record()
        barrier()
        torch.cuda.profiler.stop()
    ms = e0.elapsed_time(e1)
    # the e2e pass below reuses these buffers: copy the last timed step's outputs now
    dumps = None
    if args.dump_outputs:
        dumps = dict(x_prev=nxt, eps=eps, **(dict(e_t=e_t) if olds_n else {}))
        dumps = {k: v.float().cpu().numpy() for k, v in dumps.items()}
    launches = L.qd_launch_count() - launches0
    prog = qnn.program(x, ctx, cfg_dedup=True) if cfg_dedup else qnn.program(torch.cat([x, x]) if guided else x, ctx)
    # with a CUDA graph the kernels replay without passing through the C ABI: count them from the program
    if qnn.use_cuda_graph:
        launches = args.steps * (prog.kernel_launches + 1)

    # ---- e2e: the same step through the public API with HOST buffers.  Per step: H2D of the latents from pinned memory
    # and D2H of x_{t-1}; the prompt embeddings are a per-TRAJECTORY input (the sampler is handed them once per image
    # batch), so they are uploaded at the first step of every trajectory (every `evals` steps), inside the timed region.
    out_host = torch.empty_like(x_host)
    ctx_e2e = torch.empty_like(ctx) if ctx is not None else None
    h2d_ctx_events = [0]

    def e2e_step(i):
        xd = x_host.to(dev, non_blocking=True)
        if ctx_e2e is not None and i % UNET_EVALS_PER_IMAGE_BATCH == 0:
            ctx_e2e.copy_(c_host, non_blocking=True)       # new trajectory: new prompt embeddings (the engine re-projects K/V)
            h2d_ctx_events[0] += 1
        step(i, xd, nxt, ctx_e2e)
        out_host.copy_(nxt, non_blocking=True)
    for i in range(3):
        e2e_step(i)                                        # warm-up (i = 0 uploads the context)
    barrier()
    h2d_ctx_events[0] = 0
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(args.steps):
        e2e_step(i)                                        # i = 0 starts a trajectory: the context upload is timed
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)

    times = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        qdist.gather_latents(nxt, world)   # the path's only collective: final latent gather (SURVEY 8e)
    ms, ms_e2e = float(times[0]), float(times[1])
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    ms_step = ms / args.steps
    value = world * B / (UNET_EVALS_PER_IMAGE_BATCH * ms_step * 1e-3)
    e2e_value = world * B / (UNET_EVALS_PER_IMAGE_BATCH * (ms_e2e / args.steps) * 1e-3)
    pk = peaks()
    step_tops = UB * GOP_PER_IMAGE_EVAL / 1e3 / (ms_step * 1e-3)
    ctx_bytes = c_host.numel() * 4 if c_host is not None else 0
    line = {
        "metric": "images_per_sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int8 (W4/W8 codes x A8 codes, int32 accumulate; fp32 norms/softmax)",
        "data": "synthetic",
        "config": {"workload": w["desc"],
                   "step": f"1 denoising step = 1 UNet evaluation at batch {UB} + fused sampler update",
                   "unet_step_ms": ms_step, "unet_evals_per_image_batch": UNET_EVALS_PER_IMAGE_BATCH,
                   "l2": "working set per step (int8 weights + GBs of activations) is far larger than the 126 MB L2",
                   "cfg_prefix_dedup": bool(cfg_dedup),
                   "cfg_note": ("the guided batch [x; x] shares its UNet prefix up to the first cross-attention; the engine runs that "
                                "prefix once (bit-identical eps); whole_step_int8_tops counts the FULL batch-16 evaluation, "
                                "roofline.achieved only the executed GEMMs") if cfg_dedup else None,
                   "cuda_graph": bool(qnn.use_cuda_graph), "engine_ops_per_step": prog.nops - prog.n_static,
                   "context_ops_per_trajectory": prog.n_static,
                   "weights": "packed INT4 (two codes per byte)" if os.environ.get("QDIFF_W4_PACKED", "0") == "1" else "one code per byte (s8)",
                   "whole_step_int8_tops": step_tops, "parallelism": f"dp{world} (batch sharded, no collective in the loop)"},
        "e2e": {"value": e2e_value, "unit": "images/s",
                "h2d_bytes_per_step": x_host.numel() * 4 + (ctx_bytes * h2d_ctx_events[0]) // max(args.steps, 1),
                "d2h_bytes_per_step": out_host.numel() * 4, "ms_per_step": ms_e2e / args.steps,
                "note": f"latents up / x_prev down every step; prompt embeddings ({ctx_bytes} B) uploaded once per trajectory "
                        f"({h2d_ctx_events[0]} upload(s) inside the timed region)" if ctx_bytes else "latents up / x_prev down every step"},
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
    }
    if not args.no_roofline:
        line["roofline"] = gemm_roofline(prog, pk)
        line["roofline"]["whole_step_frac"] = step_tops / line["roofline"]["peak"]
    if world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(host_threads())
        cb = cpu_baseline(ckpt)
        line["cpu_baseline"] = cb
    if dumps is not None:
        write_dumps(args.dump_outputs, dumps)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
