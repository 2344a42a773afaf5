#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): images/sec @ SDXL 1024^2 50-step & latents/sec @ Flux 1024^2 28-step, 1/2/4/8 B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload all|sdxl|flux|vae|encoders] [--dump-outputs DIR]

ONE JSON line (rank 0).  Top level = BASELINE config 1: SDXL UNet 1024^2 bf16, batch 1 per GPU (CFG -> 2 samples per
forward), 50 Euler steps + VAE decode to a (1,3,1024,1024) tensor; a "step" is one whole image.
  value    : images/s, embeddings already resident in HBM when the timed region starts (seeded latent draw included)
  e2e      : the same through the public pipeline call with HOST (pinned) embeddings: H2D of the embeddings and D2H of the
             finished image inside the timed region
  roofline : the dominant kernel (conv_gemm_kernel: every Linear and Conv) timed launch by launch with CUDA events on the
             launching stream in a separate eager forward; achieved = algorithmic FLOPs / summed duration; peak = measured
             sustained bf16 GEMM (MEASURED_PEAKS.json).  `attention` = the same for the attention launches.
  cpu_baseline : the reference's own CPU path on a bounded sample (see cpu_reference)
  reference_cuda_eager : the UNMODIFIED reference UNet's CUDA-eager forward on the same B200 (cuBLASLt / cuDNN / SDPA): the
             "existing sm_100 kernel" bar at model level (only when baseline/_ref is on the box)
With --workload all (default) the line also carries
  flux     : BASELINE config 2 - latents/s, FluxTransformer2DModel Flux.1-dev shape, 28 FlowMatch steps (value, e2e, roofline of
             its GEMM and head_dim-128 attention launches, clocks)
  vae      : BASELINE config 4 - AutoencoderKL.decode 128^2 latent -> 1024^2, batch sweep 1 / 8 / 64
  config3  : (N > 1 only) BASELINE config 3 - SDXL batch 4 per GPU (global 32 at N = 8) through parallel.sdxl_data_parallel:
             one seeded full-batch latent draw sliced per rank, one all-gather of the decoded images, D2H once on rank 0
--impl reference times the UNMODIFIED reference (baseline/_ref) through its own StableDiffusionXLPipeline on the host cores.
Multi-GPU: one process per GPU (torchrun), each rank samples its own image (weak scaling), one all-gather of the decoded
images per step, max-over-ranks device timing.
Every timed loop runs exactly --steps steps.  --dump-outputs DIR writes what the last timed step of each section returned to
its caller as DIR/<name>.npy (float32; see Outputs): the inputs are seeded, so two builds run with the same arguments can be
compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries ONE JSON line: NCCL's version banner (NCCL_DEBUG=VERSION in this image's environment) goes there too
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"
import torch  # noqa: E402

UNET_FLOP_PER_SAMPLE = 6.7612e12      # BASELINE.md section 3 (FlopCounterMode on the reference, meta device)
VAE_FLOP_PER_IMAGE = 10.470e12
FLUX_FLOP_PER_FORWARD = 74.385e12
SDXL_SCHED = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", timestep_spacing="leading", steps_offset=1)
FLUX_SCHED = dict(shift=3.0, use_dynamic_shifting=True, base_shift=0.5, max_shift=1.15, base_image_seq_len=256, max_image_seq_len=4096)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], tflops=d.get("bf16_tflops_sustained", d["bf16_tflops"]), burst=d["bf16_tflops"], source="measured")
    return dict(hbm_gbs=6650.0, tflops=1400.0, burst=1590.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:  # noqa: BLE001
                pass

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                continue
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx or None, reasons=sorted(reasons), samples=len(sm))


def synthetic_embeds(batch, dtype, pin):
    g = torch.Generator().manual_seed(1)
    mk = lambda *s: torch.randn(*s, generator=g).to(dtype)  # noqa: E731
    t = dict(prompt_embeds=mk(batch, 77, 2048), negative_prompt_embeds=mk(batch, 77, 2048), pooled_prompt_embeds=mk(batch, 1280),
             negative_pooled_prompt_embeds=mk(batch, 1280))
    if pin:
        t = {k: v.pin_memory() for k, v in t.items()}
    return t


# ----------------------------------------------------------------------------------------------- reference arm (host cores)
def one_numa_node_physical_cores():
    """One logical CPU per physical core of NUMA node 0 (all of this process's CPUs when sysfs is silent): oversubscribing
    both NUMA nodes / hyperthreads made the round-1 CPU arm vary 10x between boxes."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except AttributeError:
        return list(range(os.cpu_count() or 1))

    def parse(s):
        out = []
        for part in s.strip().split(","):
            if "-" in part:
                a, b = part.split("-")
                out += list(range(int(a), int(b) + 1))
            elif part:
                out.append(int(part))
        return out

    try:
        with open("/sys/devices/system/node/node0/cpulist") as f:
            node0 = [c for c in parse(f.read()) if c in allowed]
    except OSError:
        node0 = allowed
    node0 = node0 or allowed
    seen, cores = set(), []
    for c in node0:
        try:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                sib = tuple(parse(f.read()))
        except OSError:
            sib = (c,)
        if sib not in seen:
            seen.add(sib)
            cores.append(c)
    return cores or allowed


def cpu_has_fast_bf16():
    try:
        with open("/proc/cpuinfo") as f:
            flags = f.read()
        return "amx_bf16" in flags or "avx512_bf16" in flags
    except OSError:
        return False


def cpu_reference(args, full=True):
    """The reference's CPU implementation of the path on a BOUNDED sample, on the physical cores of one NUMA node.

    With baseline/_ref on the box (kind "reference"): the UNMODIFIED `diffusers.StableDiffusionXLPipeline.__call__`
    (pipeline_stable_diffusion_xl.py:823) around the reference's own UNet2DConditionModel (SDXL-base config, 2.567 B random
    parameters) / EulerDiscreteScheduler / AutoencoderKL, batch 1 with CFG (two samples per UNet forward), n denoising steps
    with output_type="latent", plus (full=True) one `vae.decode` of the 128^2 latent; images/s = 1 / (50 * t_step + t_vae).
    Without it (kind "port"): the oracle's restatement of the same forward (oracle/unet.py) on the same inputs.
    dtype: bf16 when the host has AMX-bf16 / AVX512-bf16 (the reference's own choice for this workload, BASELINE.md section 2),
    fp32 otherwise - stated in `sample` and in the returned dict."""
    from baseline import ref_env
    from diffusers_b200 import specs
    cores = one_numa_node_physical_cores()
    prev_aff = None
    try:
        prev_aff = os.sched_getaffinity(0)
        os.sched_setaffinity(0, cores)
    except (AttributeError, OSError):
        pass
    prev_threads = torch.get_num_threads()
    torch.set_num_threads(len(cores))
    dt = torch.bfloat16 if cpu_has_fast_bf16() else torch.float32
    dname = "bf16" if dt == torch.bfloat16 else "fp32"
    t0 = time.time()
    cfg = dict(specs.SDXL_UNET_CONFIG)
    sd = specs.random_state_dict(specs.unet2d_condition_params(cfg), seed=0, dtype=dt)
    emb = synthetic_embeds(1, dt, pin=False)
    n_steps = max(1, min(args.steps, 3)) if full else 2
    n_warm = 1
    times = []
    with torch.no_grad():
        if ref_env.available():
            kind = "reference"
            diffusers = ref_env.import_reference()
            import inspect
            allowed = set(inspect.signature(diffusers.UNet2DConditionModel.__init__).parameters)
            with torch.device("meta"):
                unet = diffusers.UNet2DConditionModel(**{k: v for k, v in cfg.items() if k in allowed})
            unet.load_state_dict(sd, assign=True)
            unet.eval()
            vae = diffusers.AutoencoderKL(**{k: v for k, v in specs.SDXL_VAE_CONFIG.items() if k in inspect.signature(diffusers.AutoencoderKL.__init__).parameters})
            vae = vae.to(dt).eval()
            pipe = diffusers.StableDiffusionXLPipeline(vae=vae, text_encoder=None, text_encoder_2=None, tokenizer=None, tokenizer_2=None, unet=unet,
                                                       scheduler=diffusers.EulerDiscreteScheduler(**SDXL_SCHED))
            pipe.set_progress_bar_config(disable=True)

            def steps(n, seed):
                return pipe(**emb, height=1024, width=1024, num_inference_steps=n, guidance_scale=args.guidance_scale,
                            generator=torch.Generator().manual_seed(seed), output_type="latent").images

            steps(n_warm, 0)
            for i in range(2):  # two independent timed runs: the spread is reported
                a = time.perf_counter()
                lat = steps(n_steps, 1 + i)
                times.append((time.perf_counter() - a) / n_steps)
                if sum(times) * n_steps > 60:
                    break
            t_vae = None
            if full:
                a = time.perf_counter()
                vae.decode(lat / vae.config.scaling_factor, return_dict=False)
                t_vae = time.perf_counter() - a
        else:
            kind = "port"
            from oracle import unet as ounet
            g = torch.Generator().manual_seed(0)
            x = torch.randn(2, 4, 128, 128, generator=g).to(dt)
            ehs = torch.cat([emb["negative_prompt_embeds"], emb["prompt_embeds"]])
            added = dict(text_embeds=torch.cat([emb["negative_pooled_prompt_embeds"], emb["pooled_prompt_embeds"]]),
                         time_ids=torch.tensor([[1024., 1024, 0, 0, 1024, 1024]] * 2).to(dt))
            fwd = lambda: ounet.unet2d_condition_forward(sd, cfg, x, torch.tensor(981.0), ehs, added)  # noqa: E731
            fwd()
            for i in range(2):
                a = time.perf_counter()
                for _ in range(n_steps):
                    fwd()
                times.append((time.perf_counter() - a) / n_steps)
                if sum(times) * n_steps > 60:
                    break
            t_vae = None
    t_step = sum(times) / len(times)
    if t_vae is None:
        t_vae = t_step * VAE_FLOP_PER_IMAGE / (2 * UNET_FLOP_PER_SAMPLE)  # same FLOP rate assumed for the decode
        vae_note = "t_vae scaled from t_step by FLOPs"
    else:
        vae_note = f"t_vae measured once: {t_vae:.2f} s"
    ips = 1.0 / (args.denoise_steps * t_step + t_vae)
    spread = (max(times) - min(times)) / t_step if len(times) > 1 else 0.0
    what = ("unmodified diffusers.StableDiffusionXLPipeline (reference UNet2DConditionModel SDXL-base config + EulerDiscreteScheduler)"
            if kind == "reference" else "oracle port of UNet2DConditionModel.forward")
    sample = (f"{what}, batch 1 with CFG (2 samples per forward), {dname}, {len(cores)} threads pinned to the physical cores of NUMA node 0: "
              f"{len(times)} runs of {n_steps} denoising step(s) after {n_warm} warm-up = {', '.join(f'{t:.2f}' for t in times)} s per step "
              f"(spread {100 * spread:.0f}%); {vae_note}; images/s = 1 / ({args.denoise_steps} * t_step + t_vae)")
    try:
        if prev_aff is not None:
            os.sched_setaffinity(0, prev_aff)
    except OSError:
        pass
    torch.set_num_threads(prev_threads)
    return dict(value=ips, unit="images/s", cores=len(cores), kind=kind, sample=sample, dtype=dname, t_step_s=round(t_step, 3),
                t_step_runs_s=[round(t, 3) for t in times], run_spread=round(spread, 3), setup_s=round(time.time() - t0, 1))


def cpu_reference_subprocess(args):
    """cpu_baseline of the B200 arm: the same bounded sample as `--impl reference`, in a FRESH process.  In this process the
    OpenMP pool already exists (created unpinned while the GPU arm ran), so pinning now would not move its threads: the
    first build of this measured 4.8 s per step here against 3.06 s for the standalone reference arm on the same box."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--cpu-sample", "--steps", "2", "--warmup", "1",
           "--denoise-steps", str(args.denoise_steps), "--guidance-scale", str(args.guidance_scale)]
    try:
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
        for ln in reversed(p.stdout.splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return dict(value=None, unit="images/s", cores=0, kind="failed", sample=(p.stderr or p.stdout)[-300:])
    except Exception as e:  # noqa: BLE001
        return dict(value=None, unit="images/s", cores=0, kind="failed", sample=f"{type(e).__name__}: {e}"[:300])


def sdxl_workload(args):
    """config.workload of the headline benchmark: both arms (B200 and reference) report the same string."""
    return f"sdxl_unet_1024_{args.denoise_steps}step_cfg{args.guidance_scale}_b{args.batch}_per_gpu+vae_decode"


def run_reference(args, rank, world):
    if rank != 0:
        return
    cb = cpu_reference(args, full=True)
    line = dict(metric="images/sec @ SDXL 1024^2 50-step", value=cb["value"], unit="images/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1000.0 / cb["value"], higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype=cb["dtype"], data="synthetic (random-init weights, N(0,1) text embeddings, seeded latents)", impl="reference",
                config=dict(workload=sdxl_workload(args), global_batch=args.batch, parallelism=f"host cores ({cb['cores']} threads, one NUMA node)",
                            note="bounded sample of the workload (a few denoising steps + one decode), extrapolated to 50 steps: see cpu_baseline.sample"),
                cpu_baseline={k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "dtype", "t_step_runs_s", "run_spread")},
                e2e=dict(value=cb["value"], unit="images/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    emit(line)


# ----------------------------------------------------------------------------------------------- B200 arm: rooflines
def profiled(fn):
    """Runs fn() once with CUDA events around every conv_gemm / attention launch; returns (launch list, total ms)."""
    from diffusers_b200 import ops
    torch.cuda.synchronize()
    ops._PROFILE = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    try:
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
    finally:
        prof, ops._PROFILE = ops._PROFILE, None
    return [(a.elapsed_time(b), fl, kern, shape) for a, b, fl, kern, shape in prof], e0.elapsed_time(e1)


def kernel_roofline(prof, total_ms, kern, pk, extra=None):
    rows = [p for p in prof if p[2] == kern]
    if not rows:
        return None
    ms = sum(p[0] for p in rows)
    flops = sum(p[1] for p in rows)
    ach = flops / (ms * 1e-3) / 1e12
    by_shape = {}
    for t, fl, _, shape in rows:
        d = by_shape.setdefault(shape, [0, 0.0, 0.0])
        d[0] += 1
        d[1] += t
        d[2] += fl
    top = sorted(by_shape.items(), key=lambda kv: -kv[1][1])[:4]
    out = dict(bound="tensor", achieved=round(ach, 1), peak=pk["tflops"], unit="TFLOP/s", frac=round(ach / pk["tflops"], 4), traffic=None,
               kernel=kern, launches_per_forward=len(rows), algorithmic_flop_per_forward=flops, avg_launch_us=round(1000 * ms / len(rows), 2),
               kernel_ms_per_forward=round(ms, 3), forward_ms_eager=round(total_ms, 3), share_of_forward=round(ms / total_ms, 3),
               top_shapes=[dict(shape=list(s), launches=c, us_per_launch=round(1000 * t / c, 1), tflops=round(fl / t / 1e9, 1)) for s, (c, t, fl) in top],
               peak_source=pk["source"] + " (bf16_tflops_sustained: kernel timed inside a long step)")
    if extra:
        out.update(extra)
    return out


def conv_gemm_traffic():
    """DRAM traffic of conv_gemm's most frequent launch (linear 2048x1280x1280 + bias + residual, 192 per forward) from the
    committed `ncu --set full` capture; its algorithmic bytes are x 5.24 MB + W 3.28 MB + residual 5.24 MB read (the 5.24 MB
    output stays in L2) = 13.77 MB."""
    for name in ("r2_conv_gemm_traffic.json", "r1_conv_gemm_traffic.json"):
        tp = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tp):
            with open(tp) as f:
                cap = json.load(f)["launches"][0]
            return dict(traffic=cap["dram_bytes_read"] + cap["dram_bytes_write"],
                        traffic_note=f"bytes per launch of '{cap['launch']}' (ncu --set full capture, profiles/{name}); algorithmic 13.77e6")
    return dict(traffic=None)


def sdxl_unet_inputs(B2, dev, dt):
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(B2, 4, 128, 128, generator=g, device=dev).to(dt)
    ehs = torch.randn(B2, 77, 2048, generator=g, device=dev).to(dt)
    added = dict(text_embeds=torch.randn(B2, 1280, generator=g, device=dev).to(dt),
                 time_ids=torch.tensor([[1024., 1024, 0, 0, 1024, 1024]] * B2, device=dev).to(dt))
    return x, torch.tensor(981.0, device=dev), ehs, added


def sdxl_rooflines(unet, B2, pk):
    """Eager pass of one UNet forward with CUDA events around every conv_gemm / attention launch."""
    x, t, ehs, added = sdxl_unet_inputs(B2, unet.device, unet.dtype)
    was = unet.use_cuda_graph
    unet.enable_cuda_graph(False)
    fwd = lambda: unet(x, t, ehs, added_cond_kwargs=added, return_dict=False)  # noqa: E731
    for _ in range(2):
        fwd()
    prof, total = profiled(fwd)
    unet.use_cuda_graph = was
    return kernel_roofline(prof, total, "conv_gemm", pk, conv_gemm_traffic()), kernel_roofline(prof, total, "attention", pk)


def hbm_kernel_rooflines(dev, dt, pk):
    """The HBM-bound kernels of the path (SURVEY.md 8d) at their dominant SDXL shapes: 16 launches inside one CUDA graph
    over 8 rotating buffers (168 MB > L2, so the reads really come from HBM), algorithmic bytes = one read + one write of
    the activation, against the measured copy bandwidth."""
    from diffusers_b200 import ops
    g = torch.Generator(device=dev).manual_seed(0)
    out = []

    def timed(fn, n=16):
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for i in range(n):
                fn(i)
        gr.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        gr.replay()
        e1.record()
        torch.cuda.synchronize()
        return 1000.0 * e0.elapsed_time(e1) / n

    xs = [torch.randn(2 * 16384, 320, generator=g, device=dev).to(dt) for _ in range(8)]
    ys = [torch.empty_like(x) for x in xs]
    gam, bet = torch.randn(320, generator=g, device=dev).to(dt), torch.randn(320, generator=g, device=dev).to(dt)
    us = timed(lambda i: ops.group_norm(xs[i % 8], batch=2, hw=16384, groups=32, eps=1e-5, gamma=gam, beta=bet, silu=True, out=ys[i % 8]))
    nbytes = 2 * xs[0].numel() * 2
    out.append(dict(kernel="group_norm (+SiLU)", shape="2x16384x320", algorithmic_bytes=nbytes, us=round(us, 2),
                    achieved_gbs=round(nbytes / us / 1e3, 1), frac=round(nbytes / us / 1e3 / pk["hbm_gbs"], 4)))
    xl = [torch.randn(2048, 1280, generator=g, device=dev).to(dt) for _ in range(32)]
    yl = [torch.empty_like(x) for x in xl]
    lg, lb = torch.randn(1280, generator=g, device=dev).to(dt), torch.randn(1280, generator=g, device=dev).to(dt)
    us = timed(lambda i: ops.layer_norm(xl[i % 32], eps=1e-5, gamma=lg, beta=lb, out=yl[i % 32]), n=32)
    nbytes = 2 * xl[0].numel() * 2
    out.append(dict(kernel="layer_norm", shape="2048x1280", algorithmic_bytes=nbytes, us=round(us, 2), achieved_gbs=round(nbytes / us / 1e3, 1),
                    frac=round(nbytes / us / 1e3 / pk["hbm_gbs"], 4), note="10 MB per launch: launch-latency bound"))
    return out


def reference_cuda_eager(unet_cfg, dev, dt):
    """The unmodified reference UNet2DConditionModel in CUDA eager on this GPU (same config, random weights): ms per CFG forward."""
    from baseline import ref_env
    from diffusers_b200 import specs
    if not ref_env.available():
        return None
    import inspect
    diffusers = ref_env.import_reference()
    allowed = set(inspect.signature(diffusers.UNet2DConditionModel.__init__).parameters)
    with torch.device("meta"):
        m = diffusers.UNet2DConditionModel(**{k: v for k, v in unet_cfg.items() if k in allowed})
    sd = specs.random_state_dict(specs.unet2d_condition_params(unet_cfg), seed=0, dtype=dt, device=dev)
    m.load_state_dict(sd, assign=True)
    m.eval()
    x, t, ehs, added = sdxl_unet_inputs(2, dev, dt)
    with torch.no_grad():
        for _ in range(3):
            m(x, t, ehs, added_cond_kwargs=added, return_dict=False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            m(x, t, ehs, added_cond_kwargs=added, return_dict=False)
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    del m, sd
    torch.cuda.empty_cache()
    return dict(unet_forward_ms=round(ms, 2), tflops=round(2 * UNET_FLOP_PER_SAMPLE / ms / 1e9, 1),
                note="diffusers UNet2DConditionModel.forward, bf16 CUDA eager (cuBLASLt / cuDNN / SDPA), CFG batch 2, 5 timed forwards")


# ----------------------------------------------------------------------------------------------- B200 arm: workloads
class Outputs:
    """--dump-outputs: what the last timed step of each section returned, copied to the host as float32 right after its timed
    loop.  An array of more than `cap` elements is replaced by a fixed sample of its flattened values (indices drawn by
    torch.randint from seed 0, sorted): the SDXL images get 2^22 elements, every other array 2^20, so that the whole dump
    (at most 12 arrays) stays under 64 MB."""
    FLAGSHIP_CAP, CAP = 1 << 22, 1 << 20

    def __init__(self, directory):
        self.dir, self.arrays = directory, {}

    def keep(self, name, t, cap=CAP):
        if self.dir is None:
            return
        t = t.detach()
        if t.numel() > cap:
            idx = torch.randint(t.numel(), (cap,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        self.arrays[name] = t.float().cpu().numpy()

    def write(self):
        if self.dir is None:
            return
        import numpy as np
        os.makedirs(self.dir, exist_ok=True)
        assert sum(a.nbytes for a in self.arrays.values()) <= 64 << 20
        for name, a in self.arrays.items():
            np.save(os.path.join(self.dir, name + ".npy"), a)


OUTPUTS = Outputs(None)  # main() sets the directory on rank 0

class Ctx:
    def __init__(self, args, rank, world, local_rank):
        self.args, self.rank, self.world, self.local_rank = args, rank, world, local_rank
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        self.dt = torch.bfloat16
        self.pk = peaks()
        self.gpu_dead = False
        self.flux_state = None
        self.last = None  # what body() returned in the last step of the last timed loop

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(self, n, body):
        """barrier + sync, n x body(i) between CUDA events, barrier + sync; max over ranks.  Returns (ms, launches)."""
        from diffusers_b200 import ops
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = ops.launches()
        e0.record()
        for i in range(n):
            self.last = body(i)
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, ops.launches() - n0


def to_host(t):
    out = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    out.copy_(t, non_blocking=True)
    return out


def sdxl_section(cx):
    from diffusers_b200 import parallel, specs
    from diffusers_b200.autoencoder_kl import AutoencoderKL
    from diffusers_b200.pipelines import StableDiffusionXLPipeline
    from diffusers_b200.schedulers import EulerDiscreteScheduler
    from diffusers_b200.unet_2d_condition import UNet2DConditionModel
    args, dev, dt, world, pk = cx.args, cx.dev, cx.dt, cx.world, cx.pk
    unet = UNet2DConditionModel.random_init(seed=0, dtype=dt, device=dev)
    vae = AutoencoderKL.random_init(seed=0, dtype=dt, device=dev)
    pipe = StableDiffusionXLPipeline(vae, unet, EulerDiscreteScheduler(**SDXL_SCHED))
    B = args.batch
    host = synthetic_embeds(B, dt, pin=True)
    resident = {k: v.to(dev) for k, v in host.items()}
    call = dict(height=1024, width=1024, num_inference_steps=args.denoise_steps, guidance_scale=args.guidance_scale, output_type="pt")
    gather = world > 1 and B * world > 1

    def one_image(emb, seed, host_out):
        img = pipe(generator=torch.Generator(device=dev).manual_seed(seed), **emb, **call).images
        if gather:
            img = parallel.all_gather_batch(img, B * world)
        if host_out and (cx.rank == 0 or not gather):
            return to_host(img)
        return img

    for i in range(args.warmup):
        one_image(resident, i, False)
    with ClockSampler(cx.local_rank) as cs:
        ms, launches = cx.timed(args.steps, lambda i: one_image(resident, 1000 + i, False))
    OUTPUTS.keep("sdxl_images", cx.last, Outputs.FLAGSHIP_CAP)
    cx.last = None
    clocks = cs.summary()
    h2d = lambda: {k: v.to(dev, non_blocking=True) for k, v in host.items()}  # noqa: E731
    one_image(h2d(), 0, True)
    ms_e2e, _ = cx.timed(args.steps, lambda i: one_image(h2d(), 2000 + i, True))
    h2d_bytes = sum(v.numel() * v.element_size() for v in host.values())
    d2h_bytes = B * (world if gather else 1) * 3 * 1024 * 1024 * 2
    n_img = args.steps * B * world
    value = n_img / (ms * 1e-3)
    flops_per_img = 2 * args.denoise_steps * UNET_FLOP_PER_SAMPLE + VAE_FLOP_PER_IMAGE
    line = dict(metric="images/sec @ SDXL 1024^2 50-step", value=round(value, 4), unit="images/s", n_gpus=world, steps=args.steps,
                warmup=args.warmup, ms_per_step=round(ms / args.steps, 2), higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="bf16", data="synthetic (random-init weights, N(0,1) text embeddings, seeded latents)",
                config=dict(workload=sdxl_workload(args), global_batch=B * world, parallelism=f"dp{world}", cfg_batched=True,
                            l2="per-step working set >> L2: 5.1 GB of weights stream from HBM every UNet forward",
                            model="UNet2DConditionModel SDXL-base config (2.567 B params) + AutoencoderKL SDXL decoder"),
                e2e=dict(value=round(n_img / (ms_e2e * 1e-3), 4), unit="images/s", h2d_bytes_per_step=h2d_bytes, d2h_bytes_per_step=d2h_bytes,
                         note="pinned host embeddings in, decoded image(s) back to pinned host memory" + (" on rank 0 after the all-gather" if gather else "")),
                gpu_launches=launches, clocks=clocks,
                model_flops=dict(tflop_per_image=round(flops_per_img / 1e12, 1),
                                 achieved_tflops_per_gpu=round(value / world * flops_per_img / 1e12, 1),
                                 frac_of_peak=round(value / world * flops_per_img / 1e12 / pk["tflops"], 4)))
    if cx.rank == 0:
        roof, attn = sdxl_rooflines(unet, 2 * B, pk)
        line["roofline"] = roof
        line["attention"] = attn
        try:
            line["hbm_kernels"] = hbm_kernel_rooflines(dev, dt, pk)
        except Exception as e:  # noqa: BLE001  (a side measurement must never cost the headline line)
            line["hbm_kernels"] = f"failed: {e}"
    # BASELINE config 3: batch 4 per GPU through the seeded-slice data-parallel entry point (global 32 at N = 8)
    if world > 1 and not args.no_config3:
        line["config3"] = config3_section(cx, pipe)
    if cx.rank == 0 and world == 1 and not args.no_reference_cuda:
        try:
            line["reference_cuda_eager"] = reference_cuda_eager(dict(specs.SDXL_UNET_CONFIG), dev, dt)
        except Exception as e:  # noqa: BLE001
            line["reference_cuda_eager"] = f"failed: {type(e).__name__}: {str(e)[:160]}"
    del pipe, unet, vae
    torch.cuda.empty_cache()
    return line


def config3_section(cx, pipe):
    from diffusers_b200 import parallel
    args, dev, dt, world = cx.args, cx.dev, cx.dt, cx.world
    Bg = 4 * world
    host = synthetic_embeds(Bg, dt, pin=True)  # every rank holds the full-batch embeddings; the entry point slices them
    kw = dict(height=1024, width=1024, num_inference_steps=args.denoise_steps, guidance_scale=args.guidance_scale)

    def batch(seed):
        emb = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        imgs = parallel.sdxl_data_parallel(pipe, emb["prompt_embeds"], emb["negative_prompt_embeds"], emb["pooled_prompt_embeds"],
                                           emb["negative_pooled_prompt_embeds"], seed=seed, **kw)
        return to_host(imgs) if cx.rank == 0 else imgs

    batch(0)
    n = args.steps
    with ClockSampler(cx.local_rank) as cs:
        ms, launches = cx.timed(n, lambda i: batch(10 + i))
    OUTPUTS.keep("config3_images", cx.last)
    cx.last = None
    return dict(workload=f"sdxl_1024_{args.denoise_steps}step_cfg{args.guidance_scale}_global_batch{Bg}_b4_per_gpu(B_eff 8)",
                value=round(n * Bg / (ms * 1e-3), 4), unit="images/s", ms_per_batch=round(ms / n, 1), batches_timed=n, e2e=True,
                h2d_bytes_per_step=sum(v.numel() * v.element_size() for v in host.values()), d2h_bytes_per_step=Bg * 3 * 1024 * 1024 * 2,
                collective="one all_gather_into_tensor of the decoded images per batch", gpu_launches=launches, clocks=cs.summary(),
                note="one seeded full-batch latent draw sliced per rank (parallel.sdxl_data_parallel); host embeddings in, all images to rank 0's host")


def flux_section(cx):
    """BASELINE configs[2]: latents/sec, FluxTransformer2DModel (Flux.1-dev shape), 1024^2 (4096 image + 512 text tokens),
    28 FlowMatch steps, guidance 3.5, output_type='latent'.  N > 1: one latent per GPU per step (replicas, weak scaling)."""
    from diffusers_b200.pipelines import FluxPipeline
    from diffusers_b200.schedulers import FlowMatchEulerDiscreteScheduler
    from diffusers_b200.transformer_flux import FluxTransformer2DModel
    args, dev, dt, world, pk = cx.args, cx.dev, cx.dt, cx.world, cx.pk
    t0 = time.time()
    tr = FluxTransformer2DModel.random_init(seed=0, dtype=dt, device=dev)
    torch.cuda.synchronize()
    init_s = time.time() - t0

    class _V:
        config = type("C", (), dict(block_out_channels=(128, 256, 512, 512)))()

    pipe = FluxPipeline(FlowMatchEulerDiscreteScheduler(**FLUX_SCHED), _V(), tr)
    g = torch.Generator().manual_seed(1)
    host = dict(prompt_embeds=torch.randn(1, 512, 4096, generator=g).to(dt).pin_memory(),
                pooled_prompt_embeds=torch.randn(1, 768, generator=g).to(dt).pin_memory())
    nsteps = 28 if args.denoise_steps == 50 else args.denoise_steps
    call = dict(height=1024, width=1024, num_inference_steps=nsteps, guidance_scale=3.5, output_type="latent")
    n = args.steps

    def one(emb, seed, host_out):
        lat = pipe(generator=torch.Generator(device=dev).manual_seed(seed), **emb, **call).images
        return to_host(lat) if host_out else lat

    res = {k: v.to(dev) for k, v in host.items()}
    for i in range(max(1, min(args.warmup, 2))):
        one(res, i, False)
    with ClockSampler(cx.local_rank) as cs:
        ms, launches = cx.timed(n, lambda i: one(res, 100 + i, False))
    OUTPUTS.keep("flux_latents", cx.last)
    cx.last = None
    ms2, _ = cx.timed(n, lambda i: one({k: v.to(dev, non_blocking=True) for k, v in host.items()}, 200 + i, True))
    value = n * world / (ms * 1e-3)
    fl = nsteps * FLUX_FLOP_PER_FORWARD
    sec = dict(metric="latents/sec @ Flux.1-dev-shape 1024^2 28-step", value=round(value, 4), unit="latents/s", n_gpus=world, steps=n,
               warmup=max(1, min(args.warmup, 2)), ms_per_step=round(ms / n, 1), ms_per_forward=round(ms / n / nsteps, 2), higher_is_better=True,
               scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic (random-init weights, N(0,1) embeddings)",
               config=dict(workload=f"flux_dev_shape_1024_{nsteps}step_g3.5_b1_per_gpu", model="FluxTransformer2DModel 11.90 B params",
                           l2="23.8 GB of weights stream from HBM every forward", init_s=round(init_s, 1), parallelism=f"dp{world} (replicas)"),
               e2e=dict(value=round(n * world / (ms2 * 1e-3), 4), unit="latents/s", h2d_bytes_per_step=sum(v.numel() * 2 for v in host.values()),
                        d2h_bytes_per_step=4096 * 64 * 2),
               gpu_launches=launches, clocks=cs.summary(),
               model_flops=dict(tflop_per_latent=round(fl / 1e12, 1), achieved_tflops_per_gpu=round(value / world * fl / 1e12, 1),
                                frac_of_peak=round(value / world * fl / 1e12 / pk["tflops"], 4), peak=pk["tflops"]))
    if cx.rank == 0:
        # per-kernel rooflines from one eager forward with events around every GEMM / attention launch
        try:
            lat = torch.randn(1, 4096, 64, device=dev).to(dt)
            ids = FluxPipeline._prepare_latent_image_ids(64, 64, dev, dt)
            tid = torch.zeros(512, 3, device=dev, dtype=dt)
            kw = dict(hidden_states=lat, timestep=torch.tensor([0.5], device=dev, dtype=dt), guidance=torch.tensor([3.5], device=dev),
                      pooled_projections=res["pooled_prompt_embeds"], encoder_hidden_states=res["prompt_embeds"], txt_ids=tid, img_ids=ids, return_dict=False)
            tr(**kw)
            prof, total = profiled(lambda: tr(**kw))
            sec["roofline"] = kernel_roofline(prof, total, "conv_gemm", pk)
            sec["attention"] = kernel_roofline(prof, total, "attention", pk)
        except Exception as e:  # noqa: BLE001
            sec["roofline"] = f"failed: {type(e).__name__}: {str(e)[:160]}"
    # N > 1: ONE latent sharded over all N GPUs (Ulysses context parallelism over peer memory, SURVEY.md N2): strong scaling of
    # the single-image latency.  Runs last: it permutes the QKV weight rows of `tr` in place.
    if world > 1 and not args.no_context_parallel:
        cx.flux_state = (pipe, tr, res, call, nsteps, ms / n)  # run_b200 runs it LAST, under a watchdog (see there)
        return sec
    del pipe, tr
    torch.cuda.empty_cache()
    return sec


def flux_context_parallel(cx, pipe, tr, res, call, nsteps, replica_ms):
    from diffusers_b200.context_parallel import ContextParallelConfig
    args, dev, world = cx.args, cx.dev, cx.world
    try:
        tr.enable_parallelism(config=ContextParallelConfig(ulysses_degree=world))

        def one(seed):  # every rank runs the same sampling loop on the same seeded latents and gets the full latent back
            return pipe(generator=torch.Generator(device=dev).manual_seed(seed), **res, **call).images

        one(0)
        n = args.steps
        with ClockSampler(cx.local_rank) as cs:
            ms, launches = cx.timed(n, lambda i: one(300 + i))
        OUTPUTS.keep("flux_context_parallel_latents", cx.last)
        cx.last = None
        _, bufs = next(iter(tr._cp["plans"].values()))
        return dict(ulysses_degree=world, scaling="strong", value=round(n / (ms * 1e-3), 4), unit="latents/s", ms_per_latent=round(ms / n, 1),
                    ms_per_forward=round(ms / n / nsteps, 2), one_gpu_ms_per_latent=round(replica_ms, 1), speedup_vs_one_gpu=round(replica_ms / (ms / n), 3),
                    gpu_launches=launches, clocks=cs.summary(), barriers_per_forward=bufs["pg"].barriers // max(1, (n + 1) * nsteps),
                    collective="none: the QKV GEMM stores into the head owner's buffer, the attention epilogue into the row owner's, over NVLink peer "
                               "mappings; b200_peer_barrier between the phases")
    except Exception as e:  # noqa: BLE001  (a device-side failure poisons the context: report it, the caller must not touch the GPU again)
        cx.gpu_dead = True
        return f"failed: {type(e).__name__}: {str(e)[:200]}"


def vae_section(cx):
    """BASELINE.json configs[4]: AutoencoderKL.decode (SDXL decoder, 49.5 M params) of z (B,4,128,128) -> (B,3,1024,1024),
    batch sweep 1 / 8 / 64 - the convolution-roofline view of the path (10.47 TFLOP per image)."""
    from diffusers_b200.autoencoder_kl import AutoencoderKL
    args, dev, dt, pk = cx.args, cx.dev, cx.dt, cx.pk
    vae = AutoencoderKL.random_init(seed=0, dtype=dt, device=dev)
    sweep = {}
    with ClockSampler(cx.local_rank) as cs:
        for B in (1, 8, 64):
            g = torch.Generator().manual_seed(B)
            zh = torch.randn(B, 4, 128, 128, generator=g).to(dt).pin_memory()
            z = zh.to(dev)
            for _ in range(max(1, args.warmup if B < 64 else 1)):
                vae.decode(z, return_dict=False)
            n = args.steps
            ms, launches = cx.timed(n, lambda i: vae.decode(z, return_dict=False))
            OUTPUTS.keep(f"vae_decode_b{B}", cx.last[0])
            cx.last = None
            ms2, _ = cx.timed(n, lambda i: to_host(vae.decode(zh.to(dev, non_blocking=True), return_dict=False)[0]))
            sweep[B] = dict(images_per_s=round(B * n / (ms * 1e-3), 2), ms_per_batch=round(ms / n, 2), e2e_images_per_s=round(B * n / (ms2 * 1e-3), 2),
                            tflops=round(B * n * VAE_FLOP_PER_IMAGE / (ms * 1e-3) / 1e12, 1), launches=launches // n)
            del z
    best = max(sweep, key=lambda b: sweep[b]["images_per_s"])
    v = sweep[best]
    sec = dict(metric="images/sec @ AutoencoderKL.decode 1024^2 (SDXL VAE)", value=v["images_per_s"], unit="images/s", n_gpus=1, steps=args.steps,
               warmup=args.warmup, ms_per_step=v["ms_per_batch"], higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16",
               data="synthetic (random-init weights, N(0,1) latents)",
               config=dict(workload=f"sdxl_vae_decode_1024_b{best}", sweep={str(k): s for k, s in sweep.items()},
                           l2="activations of one image (268 MB per 128-channel 1024^2 tensor) >> L2"),
               e2e=dict(value=v["e2e_images_per_s"], unit="images/s", h2d_bytes_per_step=best * 4 * 128 * 128 * 2,
                        d2h_bytes_per_step=best * 3 * 1024 * 1024 * 2),
               gpu_launches=v["launches"], clocks=cs.summary(),
               model_flops=dict(tflop_per_image=round(VAE_FLOP_PER_IMAGE / 1e12, 2), achieved_tflops=v["tflops"],
                                frac_of_peak=round(v["tflops"] / pk["tflops"], 4), peak=pk["tflops"]))
    try:
        z1 = torch.randn(1, 4, 128, 128, device=dev).to(dt)
        prof, total = profiled(lambda: vae.decode(z1, return_dict=False))
        sec["roofline"] = kernel_roofline(prof, total, "conv_gemm", pk)
    except Exception as e:  # noqa: BLE001
        sec["roofline"] = f"failed: {type(e).__name__}: {str(e)[:160]}"
    del vae
    torch.cuda.empty_cache()
    return sec


def encoders_section(cx):
    """SURVEY.md N3, either side of the loop: prompts/s of the text encoders at their real sizes (SDXL: CLIP-L + OpenCLIP-bigG on 77
    tokens; Flux: CLIP-L + T5-XXL on 77 / 512 tokens; token ids in from pinned host memory, embeddings back to the host) and
    images/s of AutoencoderKL.encode at 1024^2.  Random-init weights of those architectures (no checkpoints offline)."""
    from diffusers_b200 import text_encoders as T
    from diffusers_b200.autoencoder_kl import AutoencoderKL
    args, dev, dt = cx.args, cx.dev, cx.dt
    if cx.world != 1:
        return "single-GPU section (run without torchrun)"
    out = {}
    mk = lambda cls, cfg, spec, seed: cls(cfg, T.random_state_dict(spec, seed=seed, dtype=dt, device=dev), dtype=dt, device=dev)  # noqa: E731
    te1 = mk(T.CLIPTextModel, T.CLIP_L_CONFIG, T.clip_text_params(T.CLIP_L_CONFIG, False), 1)
    te2 = mk(T.CLIPTextModelWithProjection, T.CLIP_BIGG_CONFIG, T.clip_text_params(T.CLIP_BIGG_CONFIG, True), 2)
    g = torch.Generator().manual_seed(3)
    ids77 = torch.randint(3, 49000, (2, 77), generator=g).pin_memory()  # prompt + negative prompt
    n = args.steps

    def sdxl_encode(i):
        ids = ids77.to(dev, non_blocking=True)
        a, b = te1(ids, output_hidden_states=True), te2(ids, output_hidden_states=True)
        return to_host(torch.cat([a.hidden_states[-2], b.hidden_states[-2]], -1)), to_host(b[0])

    sdxl_encode(0)
    ms, launches = cx.timed(n, sdxl_encode)
    OUTPUTS.keep("sdxl_text_encode_hidden_states", cx.last[0])
    OUTPUTS.keep("sdxl_text_encode_pooled", cx.last[1])
    out["sdxl_text_encode"] = dict(value=round(n / (ms * 1e-3), 2), unit="prompt pairs/s", ms=round(ms / n, 3), gpu_launches=launches // n,
                                   models="CLIPTextModel (CLIP-L, 123 M) + CLIPTextModelWithProjection (OpenCLIP bigG, 695 M), 2 x 77 tokens",
                                   h2d_bytes_per_step=ids77.numel() * 8, d2h_bytes_per_step=2 * 77 * 2048 * 2 + 2 * 1280 * 2)
    del te2
    t5 = mk(T.T5EncoderModel, T.T5_XXL_CONFIG, T.t5_encoder_params(T.T5_XXL_CONFIG), 3)
    ids512 = torch.randint(3, 32000, (1, 512), generator=g).pin_memory()

    def flux_encode(i):
        pooled = te1(ids77[:1].to(dev, non_blocking=True), output_hidden_states=False).pooler_output
        pe = t5(ids512.to(dev, non_blocking=True), output_hidden_states=False)[0]
        return to_host(pe), to_host(pooled)

    flux_encode(0)
    ms, launches = cx.timed(n, flux_encode)
    OUTPUTS.keep("flux_text_encode_prompt_embeds", cx.last[0])
    OUTPUTS.keep("flux_text_encode_pooled", cx.last[1])
    out["flux_text_encode"] = dict(value=round(n / (ms * 1e-3), 2), unit="prompts/s", ms=round(ms / n, 3), gpu_launches=launches // n,
                                   models="CLIPTextModel (CLIP-L) on 77 tokens + T5EncoderModel (T5-XXL v1.1, 4.76 B) on 512 tokens",
                                   h2d_bytes_per_step=(77 + 512) * 8, d2h_bytes_per_step=512 * 4096 * 2 + 768 * 2)
    del te1, t5
    torch.cuda.empty_cache()
    vae = AutoencoderKL.random_init(seed=0, dtype=dt, device=dev, encoder=True)
    xh = (torch.randn(1, 3, 1024, 1024, generator=g) * 0.5).clamp(-1, 1).to(dt).pin_memory()

    def enc(i):
        return to_host(vae.encode(xh.to(dev, non_blocking=True)).latent_dist.parameters)

    enc(0)
    ms, launches = cx.timed(n, enc)
    OUTPUTS.keep("vae_encode_moments", cx.last)
    cx.last = None
    out["vae_encode"] = dict(value=round(n / (ms * 1e-3), 2), unit="images/s", ms=round(ms / n, 3), gpu_launches=launches // n,
                             workload="AutoencoderKL.encode 1024^2 -> moments (SDXL VAE encoder, 34 M params)", h2d_bytes_per_step=3 * 1024 * 1024 * 2,
                             d2h_bytes_per_step=8 * 128 * 128 * 2)
    del vae
    torch.cuda.empty_cache()
    return out


def run_b200(args, rank, world, local_rank):
    cx = Ctx(args, rank, world, local_rank)
    wl = args.workload
    if wl == "flux":
        line = flux_section(cx)
    elif wl == "vae":
        line = vae_section(cx) if rank == 0 else None
    elif wl == "encoders":
        line = encoders_section(cx) if rank == 0 else None
    else:
        line = sdxl_section(cx)
        if wl == "all":
            try:
                line["flux"] = flux_section(cx)
            except Exception as e:  # noqa: BLE001  (the headline line must survive a failure of a secondary section)
                if world > 1:
                    raise  # a one-sided failure would deadlock the other ranks' collectives: fail loudly instead
                line["flux"] = f"failed: {type(e).__name__}: {str(e)[:200]}"
            if world == 1:
                try:
                    line["vae"] = vae_section(cx)
                except Exception as e:  # noqa: BLE001
                    line["vae"] = f"failed: {type(e).__name__}: {str(e)[:200]}"
                try:
                    line["encoders"] = encoders_section(cx)
                except Exception as e:  # noqa: BLE001
                    line["encoders"] = f"failed: {type(e).__name__}: {str(e)[:200]}"
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            cb = cpu_reference_subprocess(args)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "dtype", "t_step_runs_s", "run_spread") if k in cb}
    if cx.flux_state is not None:
        # ONE latent over all N GPUs (context parallelism over peer memory).  It is the only section in which a rank can wait for a
        # peer inside a kernel, so it runs last and under a watchdog: whatever happens to it, rank 0 prints the line it already has.
        # The limit covers the set-up, the warm-up latent and 10 s per timed latent (one took 1.2 s on 2 B200s, profiles/README.md).
        import threading
        limit = 240.0 + 10.0 * args.steps
        sec = line if wl == "flux" else line["flux"]
        sec["context_parallel"] = f"failed: no result within {limit:.0f} s (watchdog)"

        def give_up():
            if rank == 0:
                emit(line)
                try:
                    OUTPUTS.write()
                except Exception as e:  # noqa: BLE001  (the process ends here either way)
                    sys.stderr.write(f"--dump-outputs failed: {type(e).__name__}: {e}\n")
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)

        dog = threading.Timer(limit, give_up)
        dog.daemon = True
        dog.start()
        res = flux_context_parallel(cx, *cx.flux_state)
        dog.cancel()
        sec["context_parallel"] = res
        cx.flux_state = None
    if rank == 0 and line is not None:
        emit(line)
        OUTPUTS.write()  # after the line: a failed dump must not cost it
    if cx.gpu_dead:  # a trapped kernel left the CUDA context unusable: the line is out, skip the collective teardown
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


_JSON_FD = None


def emit(line):
    """The ONE JSON line, on the process's real stdout (everything else written to fd 1 - NCCL's version banner, library
    chatter of child processes - was diverted to stderr by main())."""
    sys.stdout.flush()
    text = json.dumps(line) + "\n"
    if _JSON_FD is None:
        sys.stdout.write(text)
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, text.encode())


def main():
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="all", choices=["all", "sdxl", "flux", "vae", "encoders"])
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1, help="images per GPU per step")
    ap.add_argument("--denoise-steps", type=int, default=50)
    ap.add_argument("--guidance-scale", type=float, default=7.5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config3", action="store_true")
    ap.add_argument("--no-context-parallel", action="store_true", help="N > 1: skip the Flux context-parallel (one latent over N GPUs) measurement")
    ap.add_argument("--no-reference-cuda", action="store_true")
    ap.add_argument("--cpu-sample", action="store_true", help="with --impl reference: print only the bounded cpu_baseline sample (used by the B200 arm)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step of each section to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    if rank == 0:
        OUTPUTS.dir = args.dump_outputs
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.cpu_sample:
            emit(cpu_reference(args, full=False))
        else:
            run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
