#!/usr/bin/env python
"""bench.py -- guided images/s on BASELINE.json config 2 (SD-1.4-shaped random-init UNet, fp16, 64x64 latent, 50 DDIM
steps, CFG 7.5, guidance active on the early steps), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA path
    python bench.py --impl reference [...]                       # the reference's algorithm on the host cores (oracle port)
    python bench.py [...] --dump-outputs DIR                     # also write the last timed image's latents to DIR

A "step" is one guided image (50 denoising steps of the per-step guidance path + the UNet passes that drive it).
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np   # noqa: E402
import torch         # noqa: E402

META_PROMPT = 'a [robot:.6,.3,.4,.55] and a [blue vase:.2,.3,.4,.55]'
# "guidance active on the early denoising steps": the preset at reference utils/shared_state.py:20
HYPER = {"strict": False, "inside_loss_scale": .2, "outside_loss_scale": .2, "shrink_factor": .15,
         "thresholds": {0: .4, 2: .8, 4: .9, 8: .9}, "use_optimizer": False, "recurse_until": 14, "recurse_steps": 3}
BASE_SEED = 28
EMBED_SEED = 1234
# BASELINE config 5: the fixed 64-seed sweep.  Every timed image of every run takes its seed from this list
# (`seed_idx % world_size == rank`, reference run.py:93-97 loops the same list sequentially), so the per-seed checksums
# printed by runs at different N can be compared for EQUALITY.
SWEEP_SEEDS = list(range(28, 92))


def peaks():
    """(HBM GB/s, dense bf16 TFLOP/s, provenance): the measured numbers of this pool's B200s when the driver left them."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d["bf16_tflops"]), "measured (MEASURED_PEAKS.json; burst figures: kernel timed alone)"
    return 6650.0, 1650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------ clock sampling
class ClockSampler:
    """SM clock + throttle reasons sampled every 200 ms while the timed regions run (pynvml, else nvidia-smi)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None

    def _loop(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {pynvml.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     pynvml.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     pynvml.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     pynvml.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self._stop.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, n in names.items():
                    if mask & bit:
                        self.reasons.add(n)
                self._stop.wait(0.2)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def start(self):
        self._thread = threading.Thread(target=self._loop, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ workload set-up
def setup_config(n_steps):
    from guided_attention_b200 import run as R, shared_state as S
    from guided_attention_b200.config import RunConfig
    import tempfile
    cfg = RunConfig(meta_prompt=META_PROMPT, output_path=tempfile.mkdtemp(prefix="ga_bench_"), half_precision=True,
                    n_inference_steps=n_steps)
    S.config = cfg
    S.curHyperParams = dict(HYPER)
    return cfg


def analytic_schedule(thresholds, n_steps, recurse_steps, recurse_until, max_refine=10):
    """UNet-pass counts of one image when no threshold is ever met (the case for a random-init UNet; the CUDA arm
    reports its measured counts next to this).  reference pipeline_guided_attention.py:925-1053, :501-581."""
    c = {"grad_fwd": 0, "bwd": 0, "cfg_fwd": 0, "loss_eval": 0}
    for i in range(n_steps):
        reps = recurse_steps if (i in thresholds and i <= recurse_until) else 1
        for _ in range(reps):
            c["grad_fwd"] += 1; c["loss_eval"] += 1
            if i in thresholds:
                c["grad_fwd"] += max_refine + 1; c["loss_eval"] += max_refine + 1; c["bwd"] += max_refine + 1
            c["cfg_fwd"] += 1
    return c


# ------------------------------------------------------------------------------------------------- reference arm
class _CpuRound:
    """One recursion round of guided step 0 of config 2 on the host cores, through the oracle port's OWN loop code
    (`OraclePipeline.__call__`, the restatement of reference pipeline_guided_attention.py:925-1053 and :475-581):
    1 evaluation forward + R refinement iterations (grad-enabled forward with explicit-softmax hooks, loss, backward
    to the latents, latent update) + the final evaluation forward with its threshold-step update + the CFG forward
    (batch 2) + DDIM step.  R = 10 is the whole round the reference runs when no threshold is met (1 + 11 forwards,
    11 backwards, 1 CFG); smaller R is a bounded sample of the same loop."""

    def __init__(self, unet_kind, threads):
        from oracle import oracle as O
        from tests.gpu_harness import setup_prompt, oracle_tokens, oracle_hyper
        from guided_attention_b200.substrate import DDIMScheduler, UNetConfig, build_unet
        from guided_attention_b200.run import synthetic_prompt_embeds
        torch.set_num_threads(threads)
        self.O = O
        cfg = setup_prompt(META_PROMPT, HYPER)
        ucfg = UNetConfig.sd14() if unet_kind == "sd14" else UNetConfig.tiny()
        self.unet = build_unet(ucfg, seed=0)
        self.embeds = synthetic_prompt_embeds(cfg.prompt, ucfg.cross_attention_dim, seed=EMBED_SEED)
        self.pipe = O.OraclePipeline(self.unet, DDIMScheduler(), oracle_tokens(cfg), oracle_hyper(cfg), recurse_steps=1,
                                     recurse_until=HYPER["recurse_until"])

    def run(self, refine, seed=BASE_SEED, denoise_steps=50):
        """Returns (seconds of the whole round, per-component seconds, pass counts)."""
        O, pipe = self.O, self.pipe
        sec = {"grad_fwd": 0.0, "cfg_fwd": 0.0, "loss_eval": 0.0, "bwd": 0.0}
        cnt = {"grad_fwd": 0, "cfg_fwd": 0, "loss_eval": 0, "bwd": 0}
        orig_unet, orig_loss, orig_update = pipe._unet, pipe._loss, O.update_latent

        def timed(key, fn):
            def wrapped(*a, **k):
                t0 = time.perf_counter()
                out = fn(*a, **k)
                sec[key] += time.perf_counter() - t0
                cnt[key] += 1
                return out
            return wrapped

        def unet(x, t, emb):
            return timed("cfg_fwd" if x.shape[0] == 2 else "grad_fwd", orig_unet)(x, t, emb)
        pipe._unet, pipe._loss, O.update_latent = unet, timed("loss_eval", orig_loss), timed("bwd", orig_update)
        lat = torch.randn(1, 4, 64, 64, generator=torch.Generator("cpu").manual_seed(seed))
        try:
            t0 = time.perf_counter()
            trace = pipe(self.embeds, lat, seed, num_inference_steps=denoise_steps, guidance_scale=7.5,
                         thresholds=HYPER["thresholds"], max_steps=1, max_refinement_steps=refine)
            total = time.perf_counter() - t0
        finally:
            pipe._unet, pipe._loss, O.update_latent = orig_unet, orig_loss, orig_update
        return total, sec, cnt, float(trace.losses[0][2])


def cpu_images_per_s(per_pass_s, schedule):
    return 1.0 / sum(per_pass_s[k] * schedule[k] for k in schedule)


def _per_pass(samples):
    """Average seconds per pass of each kind over the measured rounds."""
    out = {}
    for k in ("grad_fwd", "cfg_fwd", "loss_eval", "bwd"):
        n = sum(c[k] for _, _, c in samples)
        out[k] = sum(s[k] for _, s, _ in samples) / max(n, 1)
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    sched = analytic_schedule(HYPER["thresholds"], args.denoise_steps, HYPER["recurse_steps"], HYPER["recurse_until"])
    cpu = _CpuRound(args.unet, threads)
    samples, wall = [], []
    for i in range(args.warmup + args.steps):
        # the first timed step is the WHOLE round (10 refinement iterations); the others are bounded samples of the
        # same loop so that `--steps K --warmup W` ends within minutes on 16 host cores
        refine = args.ref_refine_first if i == args.warmup else args.ref_refine
        total, sec, cnt, _ = cpu.run(refine, denoise_steps=args.denoise_steps)
        if i >= args.warmup:
            samples.append((total, sec, cnt))
            wall.append(total)
    per_pass = _per_pass(samples)
    v = cpu_images_per_s(per_pass, sched)
    measured_passes = {k: sum(c[k] for _, _, c in samples) for k in per_pass}
    sample = (f"{args.steps} timed recursion rounds of guided step 0 through the oracle port's own loop "
              f"(OraclePipeline.__call__, fp32, explicit-softmax hooks) on {threads} host threads: the first with "
              f"{args.ref_refine_first} refinement iterations"
              + (" (the WHOLE round the reference runs: 1 + 11 forwards, 11 backwards, 1 CFG forward)"
                 if args.ref_refine_first == 10 else "") +
              f", the others with {args.ref_refine}; measured passes {measured_passes} in "
              f"{sum(wall):.1f} s; EXTRAPOLATED to one image with the analytic UNet-pass schedule {sched} "
              "(no threshold met)")
    line = {"impl": "reference", "metric": "guided_images_per_s", "value": v, "unit": "img/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / v, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "extrapolated": True, "measured_s": sum(wall), "measured_s_per_step": wall,
            "config": workload_config(args, "f32"),
            "cpu_baseline": {"value": v, "unit": "img/s", "cores": threads, "kind": "port", "sample": sample,
                             "extrapolated": True, "measured_s": sum(wall), "measured_passes": measured_passes,
                             "seconds_per_pass": per_pass, "schedule_per_image": sched},
            "e2e": {"value": v, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "one host arm, whatever --gpus says: under torchrun rank 0 alone runs it.  A ratio against an "
                    "N-GPU line compares N GPUs with ONE host and is not a per-device speed-up."}
    print(json.dumps(line))
    return 0


def workload_config(args, dtype):
    return {"workload": "BASELINE config 2: SD-1.4-shaped UNet (random init, seed 0), 64x64 latent (512^2 image), "
                        f"meta_prompt '{META_PROMPT}', seeds {BASE_SEED}+, {args.denoise_steps} DDIM steps, CFG 7.5 "
                        f"(batch 2), {dtype}, thresholds {HYPER['thresholds']} (guidance on early steps), "
                        "recurse_steps 3, attention_res 16" + ("" if args.unet == "sd14" else " [TINY UNET: NOT THE BASELINE CONFIG]"),
            "unet": args.unet, "denoise_steps": args.denoise_steps, "images_per_step_per_gpu": 1,
            "cuda_graphs": not getattr(args, "no_graphs", False),
            "control_flow": ("eager host loop" if getattr(args, "no_graphs", False) else
                             "host loop replaying graphs (one D2H read per loss evaluation)"
                             if getattr(args, "host_control", False) else
                             "device-side step driver (CUDA conditional graph nodes, no loss read back)"),
            "unet_elementwise": ("PyTorch ops (GA_FUSED_NORM=0)" if os.environ.get("GA_FUSED_NORM", "1") == "0" else
                                 "fused channels-last kernels of this repo: GroupNorm(+SiLU, +conv bias / time-embedding "
                                 "shift), conv bias + residual, GEGLU" +
                                 (" [off: %s]" % os.environ["GA_FUSED_DISABLE"] if os.environ.get("GA_FUSED_DISABLE") else "")),
            "l2_policy": "inputs larger than L2: every UNet pass streams 1.7 GB of fp16 weights (L2 is 126 MB)",
            "parallelism": f"seed-sharded, {args.gpus} process(es), no hot-path collective"}


# ------------------------------------------------------------------------------------------------------ CUDA arm
def _sha(t):
    """sha1 of the fp16 latents' bytes: the per-seed checksum compared across runs at different N (config 5)."""
    import hashlib
    return hashlib.sha1(t.detach().to(torch.float16).cpu().contiguous().numpy().tobytes()).hexdigest()[:16]


def dump_outputs(out_dir, arrays):
    """`--dump-outputs`: every array as `out_dir/<name>.npy` in float32.  The inputs are fixed by the seeds above, so two
    builds run with the same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def build_pipeline(args, dev):
    from guided_attention_b200 import run as R
    from guided_attention_b200.pipeline_guided_attention import GuidedAttention
    from guided_attention_b200.ptp_utils import AttentionStore, register_attention_control
    from guided_attention_b200.substrate import DDIMScheduler, UNetConfig, WhitespaceTokenizer, build_unet
    cfg = setup_config(args.denoise_steps)
    ucfg = UNetConfig.sd14() if args.unet == "sd14" else UNetConfig.tiny()
    unet = build_unet(ucfg, seed=0, dtype=torch.float16, device=dev)
    pipe = GuidedAttention(unet=unet, scheduler=DDIMScheduler(), tokenizer=WhitespaceTokenizer())
    cfg.stable = pipe
    pipe.use_cuda_graphs = not args.no_graphs
    pipe.device_side_control = not getattr(args, "host_control", False)
    R.register_custom_loss("toLeftOf", R.ToLeftOf())
    R.overrideConfig(cfg)
    R.parseMetaPrompt(cfg)
    store = AttentionStore()
    register_attention_control(pipe, store)
    embeds_host = R.synthetic_prompt_embeds(cfg.prompt, ucfg.cross_attention_dim, seed=EMBED_SEED).pin_memory()
    return cfg, pipe, store, embeds_host


def run_ours(args):
    from guided_attention_b200 import build as B
    B.build()
    from guided_attention_b200 import ops, shared_state as S, sweep
    import torch.distributed as dist

    rank, world, local_rank = sweep.init_distributed()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (CUDA arm) needs a GPU: the guidance path has no CPU fallback")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    cfg, pipe, store, embeds_host = build_pipeline(args, dev)

    def host_latents(seed):
        g = torch.Generator("cpu").manual_seed(seed)
        return torch.randn(1, 4, 64, 64, generator=g).pin_memory()

    def image(seed, embeds, latents):
        S.cur_seed = seed
        gen = torch.Generator("cpu").manual_seed(seed)
        out = pipe(prompt=cfg.prompt, attention_store=store, attention_res=16, guidance_scale=7.5, generator=gen,
                   latents=latents, prompt_embeds=embeds[1:2], negative_prompt_embeds=embeds[0:1],
                   num_inference_steps=args.denoise_steps, thresholds=cfg.thresholds, scale_factor=20,
                   scale_range=(1., .5), smooth_attentions=True, sigma=0.5, kernel_size=3, sd_2_1=False,
                   output_type="latent")
        return out.images

    def seed_of(step):      # timed images: the config-5 sweep list, seed_idx % world == rank
        return SWEEP_SEEDS[(step * world + rank) % len(SWEEP_SEEDS)]

    def warm_seed(w):       # warm-up images come from the far end of the list
        return SWEEP_SEEDS[-1 - ((w * world + rank) % len(SWEEP_SEEDS))]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        res = [fn(i) for i in range(n)]
        e.record()
        torch.cuda.synchronize()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        return float(ms), res

    if args.sweep64:
        return run_sweep64(args, rank, world, dev, image, host_latents, embeds_host, timed, sweep, dist, pipe)

    embeds_dev = embeds_host.to(dev, non_blocking=True)
    for w in range(args.warmup):
        image(warm_seed(w), embeds_dev, host_latents(warm_seed(w)).to(dev))

    sampler = ClockSampler(local_rank)
    sampler.start()
    # (1) device-resident inputs: `value`
    dev_lat = [host_latents(seed_of(i)).to(dev) for i in range(args.steps)]
    ops.reset_launch_counts()
    pipe._count_pass("cfg", 0)
    before = dict(pipe.pass_counts)
    ms_value, value_res = timed(lambda i: image(seed_of(i), embeds_dev, dev_lat[i]), args.steps)
    last_out = value_res[-1].detach().cpu() if args.dump_outputs else None     # the last timed step's result
    launches = ops.total_launches()
    counts = dict(ops.launch_counts)
    passes = {k: pipe.pass_counts[k] - before[k] for k in before}
    unet_passes = sum(passes.values())
    # (2) end to end: host buffers in, host buffer out, inside the timed region; final NCCL gather of the latents
    host_lat = [host_latents(seed_of(i)) for i in range(args.steps)]
    out_host = torch.empty(args.steps, 4, 64, 64, dtype=torch.float16).pin_memory()

    def e2e_step(i):
        lat = image(seed_of(i), embeds_host.to(dev, non_blocking=True), host_lat[i].to(dev, non_blocking=True))
        out_host[i].copy_(lat[0], non_blocking=True)
        return lat

    def e2e_all(_):
        res = [e2e_step(i) for i in range(args.steps)]
        if world > 1:   # the only collective of the workload: gather the final latents (32 KB / image)
            sweep.gather_results(torch.cat(res), args.steps * world, rank, world)
        torch.cuda.synchronize()
        return res
    ms_e2e, e2e_res = timed(e2e_all, 1)
    clocks = sampler.stop()

    # per-seed checksums (config 5 equality evidence): value leg == e2e leg in this process, and comparable across N
    sums = {str(seed_of(i)): _sha(value_res[i]) for i in range(args.steps)}
    same_legs = all(_sha(e2e_res[0][i]) == sums[str(seed_of(i))] for i in range(args.steps))
    if world > 1:
        everyone = [None] * world
        dist.all_gather_object(everyone, (sums, same_legs))
        sums = {k: v for d, _ in everyone for k, v in d.items()}
        same_legs = all(ok for _, ok in everyone)

    # (3) roofline: one more image with per-launch CUDA events on the launching stream
    # (CUDA events cannot be recorded inside a graph replay: this pass runs the eager loop, same kernels)
    pipe.use_cuda_graphs = False
    ops.profiler = ops.LaunchProfiler()
    image(seed_of(0), embeds_dev, dev_lat[0])
    prof = ops.profiler.summary()
    ops.profiler = None
    pipe.use_cuda_graphs = not args.no_graphs
    tensor_roof, kernel_table = roofline_from(prof)

    # (4) extension: S seeds per UNet pass (`generate_batch`), same per-seed semantics; device-resident and end to end
    batched = None
    if args.seeds_per_batch > 1:
        Sb = args.seeds_per_batch
        emb16 = embeds_dev.to(torch.float16)

        def batch_seeds(i):
            return [SWEEP_SEEDS[((i * world + rank) * Sb + j) % len(SWEEP_SEEDS)] for j in range(Sb)]

        def batch_lat(i):
            return torch.cat([host_latents(sd) for sd in batch_seeds(i)]).pin_memory()

        def batch_step(i, lat_dev=None, emb=None):
            emb = emb16 if emb is None else emb
            return pipe.generate_batch(cfg.prompt, store, batch_seeds(i), emb[1:2], emb[0:1], attention_res=16,
                                       num_inference_steps=args.denoise_steps, guidance_scale=7.5,
                                       thresholds=cfg.thresholds, latents=lat_dev)
        batch_step(0, batch_lat(0).to(dev))                          # warm-up: captures the batch-S graphs
        lat_b = batch_lat(0).to(dev)
        ms_b, res_b = timed(lambda i: batch_step(0, lat_b), 1)
        lat_bh = batch_lat(0)
        out_bh = torch.empty(Sb, 4, 64, 64, dtype=torch.float16).pin_memory()

        def batch_e2e(_):
            r = batch_step(0, lat_bh.to(dev, non_blocking=True),
                           embeds_host.to(dev, non_blocking=True).to(torch.float16))
            out_bh.copy_(r, non_blocking=True)
            torch.cuda.synchronize()
            return r
        ms_be, _ = timed(batch_e2e, 1)
        batched = {"seeds_per_batch": Sb, "value": Sb * world / (ms_b / 1e3), "unit": "img/s", "ms_per_batch": ms_b,
                   "e2e": {"value": Sb * world / (ms_be / 1e3), "unit": "img/s",
                           "h2d_bytes_per_step": int(embeds_host.numel() * 4 + Sb * 4 * 64 * 64 * 4),
                           "d2h_bytes_per_step": int(Sb * 4 * 64 * 64 * 2)},
                   "seed_checksums": {str(sd): _sha(res_b[0][j:j + 1]) for j, sd in enumerate(batch_seeds(0))},
                   "note": "extension (SURVEY 8e): S seeds advance through one UNet pass; per-seed results match the "
                           "one-seed path within the bound tested in tests/test_gpu_parity.py (batched GEMM/conv "
                           "shapes differ, so not bit-identical)"}

    # (5) the metric's second half: HBM GB/s of the attention-map kernels, live, at GPU-filling batch sizes
    # (rank 0; last, because the tail timer re-installs the prompt)
    roofline, hbm_table = None, None
    if not args.no_saturated:
        keep = (S.config, S.curHyperParams)
        torch.cuda.empty_cache()
        # kernel-only figures against a BURST peak (MEASURED_PEAKS.json: best of 10 copies on an idle GPU): let the GPU
        # idle for a few seconds after the image loops, and sample the clocks of this phase on their own
        torch.cuda.synchronize()
        time.sleep(SATURATED_IDLE_S)
        sat_sampler = ClockSampler(local_rank)
        sat_sampler.start()
        roofline, hbm_table = attn_map_roofline(dev, kernel_table)
        sat_clocks = sat_sampler.stop()
        if roofline is not None:
            roofline["clocks"] = sat_clocks
            roofline["idle_before_s"] = SATURATED_IDLE_S
        S.config, S.curHyperParams = keep
        torch.cuda.empty_cache()
    if roofline is None:
        roofline = tensor_roof
    else:
        roofline["tensor"] = tensor_roof

    n_img = args.steps * world
    value = n_img / (ms_value / 1e3)
    e2e = n_img / (ms_e2e / 1e3)
    line = {"metric": "guided_images_per_s", "value": value, "unit": "img/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_value / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic", "config": workload_config(args, "fp16"),
            "e2e": {"value": e2e, "unit": "img/s",
                    "h2d_bytes_per_step": int(embeds_host.numel() * 4 + 4 * 64 * 64 * 4),
                    "d2h_bytes_per_step": int(4 * 64 * 64 * 2)},
            "gpu_launches": launches, "gpu_launches_by_kernel": counts, "unet_passes": unet_passes,
            "unet_passes_by_program": passes, "clocks": clocks, "roofline": roofline, "kernels": kernel_table,
            "saturated_kernels": hbm_table, "batched": batched,
            "seed_checksums": sums, "value_leg_equals_e2e_leg": same_legs}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        total, sec, cnt, _ = _CpuRound(args.unet, threads).run(args.ref_refine_first, denoise_steps=args.denoise_steps)
        per_pass = {k: sec[k] / max(cnt[k], 1) for k in sec}
        n_eval = (passes["eval"] + passes["update"]) / args.steps
        per_image = {"grad_fwd": n_eval, "loss_eval": n_eval, "bwd": passes["update"] / args.steps,
                     "cfg_fwd": passes["cfg"] / args.steps}
        line["cpu_baseline"] = {
            "value": cpu_images_per_s(per_pass, per_image), "unit": "img/s", "cores": threads, "kind": "port",
            "extrapolated": True, "measured_s": total, "measured_passes": cnt, "seconds_per_pass": per_pass,
            "sample": f"one WHOLE recursion round of guided step 0 ({cnt['grad_fwd']} grad-enabled B=1 forwards with "
                      f"explicit-softmax hooks, {cnt['loss_eval']} loss evaluations, {cnt['bwd']} backwards to the "
                      f"latents, {cnt['cfg_fwd']} CFG forward) through the oracle port's own loop, fp32, {threads} "
                      f"host threads, {total:.1f} s measured; EXTRAPOLATED to one image with the UNet-pass counts "
                      f"this run measured per image: {per_image}"}
    if rank == 0:
        print(json.dumps(line))
    if args.dump_outputs:
        if world > 1:       # every rank's last image, in rank order
            parts = [None] * world
            dist.all_gather_object(parts, last_out)
            last_out = torch.cat(parts)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"final_latents": last_out})
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_sweep64(args, rank, world, dev, image, host_latents, embeds_host, timed, sweep, dist, pipe):
    """BASELINE config 5 as stated: the fixed seeds range(28, 92) through `sweep.run_seed_sweep` (static round-robin
    `seed_idx % world`), host buffers in, ONE gather of the final latents at the end (NCCL over NVLink), strong scaling.
    The line carries one checksum per seed: lines produced at different N must agree seed by seed."""
    seeds = SWEEP_SEEDS[: args.sweep_seeds]
    embeds_dev = embeds_host.to(dev)
    for w in range(max(args.warmup, 1)):        # graph capture + warm-up outside the timed region
        image(SWEEP_SEEDS[-1 - w], embeds_dev, host_latents(SWEEP_SEEDS[-1 - w]).to(dev))
    sampler = ClockSampler(dev.index)
    sampler.start()
    box = {}

    def job(_):
        full, local, failures = sweep.run_seed_sweep(
            lambda sd: image(sd, embeds_host.to(dev, non_blocking=True), host_latents(sd).to(dev, non_blocking=True))[0],
            seeds, rank, world)
        torch.cuda.synchronize()
        box["full"], box["failures"] = full, failures
        return full
    ms, _ = timed(job, 1)
    clocks = sampler.stop()
    full = box["full"]
    sums = {str(sd): _sha(full[i]) for i, sd in enumerate(seeds)}
    import hashlib
    line = {"metric": "guided_images_per_s", "mode": "sweep64", "value": len(seeds) / (ms / 1e3), "unit": "img/s",
            "n_gpus": world, "steps": 1, "warmup": max(args.warmup, 1), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": dict(workload_config(args, "fp16"), seeds=f"range({seeds[0]}, {seeds[-1] + 1})",
                           sharding="seed_idx % world_size == rank"),
            "e2e": {"value": len(seeds) / (ms / 1e3), "unit": "img/s",
                    "h2d_bytes_per_step": int(len(seeds) * (embeds_host.numel() * 4 + 4 * 64 * 64 * 4)),
                    "d2h_bytes_per_step": 0},
            "failures": box["failures"], "clocks": clocks, "seed_checksums": sums,
            "checksum_of_checksums": hashlib.sha1("".join(sums[str(sd)] for sd in seeds).encode()).hexdigest()[:16]}
    if rank == 0:
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"final_latents": full})
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


NOMINAL_HBM_GBS = 8000.0     # BASELINE.json metric: "attn-map kernel HBM GB/s vs 8 TB/s"

# (kernel, N, d, maps) -> batch at which the launch fills the GPU; the pipeline's own launches (B = 1, 2) move
# 0.7-11 MB and are launch-latency bound by size (SURVEY 8d "latency caveat")
SATURATED_IDLE_S = 5.0
SATURATED_SHAPES = [("cross_attn", 1024, 80, True, 256), ("cross_attn", 256, 160, True, 512),
                    ("cross_attn", 4096, 40, False, 128)]


def ncu_traffic(kernel, shape_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` summaries
    (tools/ncu_all.sh -> tools/ncu_summary.py), newest round first.  Returns (bytes | None, source | None)."""
    for name in ("r02b_ncu_summary.json", "r02_ncu_summary.json", "r01_ncu_final_summary.json"):
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.isfile(path):
            continue
        with open(path) as f:
            rows = json.load(f)
        # an op that is two kernels (large-launch tail forward, self-attention backward) has one row per kernel
        hit = [float(r["dram_traffic_bytes"]) for r in rows
               if r.get("bench_key") == [kernel, shape_key] and r.get("dram_traffic_bytes") is not None]
        if hit:
            return sum(hit), f"profiles/{name} (ncu --set full, same kernel and shape)"
    return None, None


def _saturated_in_subprocess(dev):
    """Runs `python -m guided_attention_b200.microbench --saturated <device>` and returns {(kind, direction, N | res): row},
    or None if the child could not be run."""
    import subprocess
    try:
        out = subprocess.run([sys.executable, "-m", "guided_attention_b200.microbench", "--saturated", str(dev)],
                             cwd=ROOT, capture_output=True, text=True, timeout=600)
        rows = [json.loads(ln) for ln in out.stdout.splitlines() if ln.startswith("{")]
        table = {}
        for r in rows:
            if r["kernel"].startswith("cross_attn"):
                table[("cross_attn", r["kernel"].split("_")[-1], r["N"])] = r
            else:
                table[("tail", r["kernel"].split("_")[-1], r["res"])] = r
        return table if len(table) == 2 * (len(SATURATED_SHAPES) + 2) else None
    except Exception:
        return None


def attn_map_roofline(dev, kernel_table):
    """The HBM-bound guidance kernels timed LIVE in this run at GPU-filling batch sizes: CUDA graph of back-to-back
    launches between two CUDA events on the launching stream, rotating buffer sets larger than L2
    (`guided_attention_b200.microbench`).  Returns (`roofline` block for the dominant attention-map kernel, table).
    Dominant = the attention-map kernel class (K1 with map accumulation, K2 with the injected map gradient, tail fwd /
    bwd) with the largest summed device time inside one image of the pipeline (`kernel_table`)."""
    from guided_attention_b200 import microbench
    peak, _, how = peaks()
    rows = []

    def add(m, kernel, key, shape):
        traffic, src = ncu_traffic(kernel, key)
        rows.append({"kernel": kernel, "key": key, "shape": shape, "us": m["us"], "bytes": m["bytes"], "gbs": m["gbs"],
                     "frac": m["gbs"] / peak, "frac_of_8tbs": m["gbs"] / NOMINAL_HBM_GBS, "traffic": traffic,
                     "traffic_source": src})
    # The measurements run in a FRESH process on the same GPU (this one keeps its UNet, graphs and pools, idle): timed
    # inside this process after ~2 000 UNet passes the same launches came out 5-20 % slower than the stand-alone sweep
    # on the same box a minute earlier (profiles/r02d_*: K1 d = 40 226 vs 184 us) -- allocator / page-table state of a
    # long-lived process, not the kernels.  `measured_in` says which way the numbers were taken.
    child = _saturated_in_subprocess(dev)
    measured_in = "fresh subprocess on the same GPU" if child is not None else "this process"

    def timed(kind, direction, **kw):
        if child is not None:
            return child[(kind, direction, kw.get("N", kw.get("res")))]
        if kind == "cross_attn":
            return microbench.time_cross_attn(kw["B"], 8, kw["N"], 77, kw["d"], torch.float16, with_acc=kw["maps"],
                                              direction=direction, device=str(dev))
        return microbench.time_tail(kw["res"], 5, 2, n_samples=kw["S"], direction=direction, device=str(dev))
    try:
        for direction in ("fwd", "bwd"):
            for _, N, d, maps, B in SATURATED_SHAPES:
                m = timed("cross_attn", direction, B=B, N=N, d=d, maps=maps)
                add(m, f"cross_attn_{direction}", f"N{N}_d{d}_maps{maps}",
                    f"B={B} H=8 N={N} T=77 d={d} fp16" + (" (maps)" if maps else ""))
            for res in (16, 32):
                m = timed("tail", direction, res=res, S=2048 if res == 16 else 512)
                add(m, f"guidance_tail_{direction}", f"res{res}",
                    f"res {res}, 5 layers x 2 slices, {2048 if res == 16 else 512} samples")
    except Exception as e:   # never lose the headline line to an auxiliary measurement
        rows.append({"error": f"{type(e).__name__}: {e}"})
        return None, rows

    def key_of(row):     # in-pipeline class -> key of the saturated measurement
        if row["kernel"].startswith("cross_attn"):
            return f"N{row['shape'][2]}_d{row['shape'][4]}_maps{row['shape'][6]}"
        if row["kernel"].startswith("guidance_tail"):
            return f"res{row['shape'][0]}"
        return None
    in_pipe = {}
    for row in kernel_table:
        k = key_of(row)
        is_map = (row["kernel"].startswith("guidance_tail") or
                  (row["kernel"].startswith("cross_attn") and row["shape"][6] == "True"))
        if k is not None and is_map:
            in_pipe[(row["kernel"], k)] = row
    ranked = sorted(in_pipe.items(), key=lambda kv: -kv[1]["total_ms"])
    top = next((r for (kern, k), _ in ranked for r in rows if r["kernel"] == kern and r["key"] == k), rows[0])
    pipe_row = in_pipe.get((top["kernel"], top["key"]))
    roof = {"bound": "hbm", "kernel": top["kernel"], "shape": top["shape"], "achieved": top["gbs"], "peak": peak,
            "unit": "GB/s", "frac": top["frac"], "frac_of_8tbs": top["frac_of_8tbs"], "traffic": top["traffic"],
            "traffic_source": top["traffic_source"], "peak_source": how, "avg_launch_us": top["us"],
            "algorithmic_bytes_per_launch": top["bytes"], "measured_in": measured_in,
            "how": "dominant attention-map kernel of the pipeline (largest summed device time among K1-with-maps, "
                   "K2-with-map-gradient, tail fwd/bwd inside one image), timed live in this run at a GPU-filling "
                   "batch: CUDA graph of back-to-back launches between CUDA events on the launching stream, rotating "
                   "buffer sets larger than L2",
            "in_pipeline_launch": None if pipe_row is None else {
                "shape": pipe_row["shape"], "launches_per_image": pipe_row["launches"],
                "kernel_us": pipe_row.get("kernel_us"), "gbs": pipe_row.get("gbs"),
                "note": "the pipeline's own launch (B = 1 or 2) moves a few MB: launch-latency bound by size"},
            "attn_map_kernels": [{k: r[k] for k in ("kernel", "shape", "us", "gbs", "frac", "frac_of_8tbs", "traffic")}
                                 for r in rows]}
    return roof, rows


def roofline_from(prof):
    """Dominant kernel = the (kernel, shape) class with the largest summed device time inside the profiled image.
    Its launch duration is then measured kernel-only: the same launch (same shape, dtype, variant choice) replayed
    back-to-back from a CUDA graph between two CUDA events on the launching stream, on rotating buffer sets larger than
    L2 (`microbench.time_cross_attn` / `time_self_attn`).  The in-pipeline event time is kept next to it: it includes
    the host gaps of the eager profiling pass and only serves to rank the kernels.
    Cross-attention / tail kernels are HBM-bound (algorithmic bytes); the self-attention kernels are tensor-pipe bound
    (algorithmic FLOPs = the 2 GEMMs of the forward / 5 of the backward, not the recomputation the kernels add)."""
    from guided_attention_b200 import microbench
    hbm_peak, tf_peak, how = peaks()
    dev = f"cuda:{torch.cuda.current_device()}"      # every rank measures on its own GPU
    table = []
    for (name, key), d in prof.items():
        avg_us = d["ms"] * 1e3 / d["launches"]
        row = {"kernel": name, "shape": list(map(str, key)), "launches": d["launches"],
               "pipeline_event_us": avg_us, "total_ms": d["ms"]}
        row["flops_issued_per_launch" if name.startswith("self_attn") else "bytes_per_launch"] = d["bytes_per_launch"]
        table.append(row)
    table.sort(key=lambda r: -r["total_ms"])
    if not table:
        return None, table
    dts = {"torch.float16": torch.float16, "torch.bfloat16": torch.bfloat16, "torch.float32": torch.float32}
    n_attn = n_unet = 0
    for row in table:
        is_attn = row["kernel"].startswith(("cross_attn", "self_attn"))
        if (is_attn and n_attn >= 8) or (not is_attn and n_unet >= 6):
            continue
        n_attn, n_unet = n_attn + int(is_attn), n_unet + int(not is_attn)
        if row["kernel"].startswith("group_norm"):
            # UNet-side fused kernels (the callers either side of the attention layers): kernel-only time of the same
            # call, next to PyTorch's own ops for that call on the same tensors
            n, hw, c, groups, silu = (int(x) for x in row["shape"][:5])
            direction = "fwd" if row["kernel"].endswith("fwd") else "fwdbwd"
            m = microbench.time_group_norm(n, c, hw, 1, groups, bool(silu), direction, "fused", device=dev)
            t = microbench.time_group_norm(n, c, hw, 1, groups, bool(silu), direction, "torch", device=dev)
            row["kernel_us" if direction == "fwd" else "fwd_plus_bwd_us"] = m["us"]
            row["gbs"], row["torch_ops_us"] = m["gbs"], t["us"]
        elif row["kernel"].startswith("geglu"):
            rows_, inner = (int(x) for x in row["shape"][:2])
            direction = "fwd" if row["kernel"].endswith("fwd") else "fwdbwd"
            m = microbench.time_geglu(rows_, inner, direction, "fused", device=dev)
            t = microbench.time_geglu(rows_, inner, direction, "torch", device=dev)
            row["kernel_us" if direction == "fwd" else "fwd_plus_bwd_us"] = m["us"]
            row["gbs"], row["torch_ops_us"] = m["gbs"], t["us"]
        if row["kernel"].startswith("cross_attn"):
            B, H, N, T, dd = (int(x) for x in row["shape"][:5])
            m = microbench.time_cross_attn(B, H, N, T, dd, dts[row["shape"][5]], with_acc=row["shape"][6] == "True",
                                           direction=row["kernel"].split("_")[-1], device=dev)
            row["kernel_us"], row["gbs"] = m["us"], m["gbs"]
        elif row["kernel"].startswith("self_attn"):
            B, H, N, dd = (int(x) for x in row["shape"][:4])
            m = microbench.time_self_attn(B, H, N, dd, dts[row["shape"][4]], direction=row["kernel"].split("_")[-1],
                                          device=dev)
            row["kernel_us"], row["tflops"], row["tflops_issued"] = m["us"], m["tflops_algorithmic"], m["tflops_issued"]
            row["algorithmic_flops_per_launch"] = m["tflops_algorithmic"] * m["us"] * 1e6
    top = next((r for r in table if "kernel_us" in r and r["kernel"].startswith(("self_attn", "cross_attn"))), table[0])
    if "tflops" in top:
        roof = {"bound": "tensor", "kernel": top["kernel"], "shape": top["shape"], "achieved": top["tflops"],
                "peak": tf_peak, "unit": "TFLOP/s", "frac": top["tflops"] / tf_peak,
                "traffic": ncu_traffic(top["kernel"], "B{}_H{}_N{}_d{}".format(*top["shape"][:4]))[0],
                "peak_source": how, "avg_launch_us": top["kernel_us"],
                "algorithmic_flops_per_launch": top["algorithmic_flops_per_launch"],
                "issued_tflops": top["tflops_issued"],
                "note": "fused exact self-attention at head_dim 40: per exponential only 4*d = 160 FLOPs of GEMM work "
                        "exist, so the SFU (16 ex2/clk/SM) caps this kernel far below the dense-GEMM peak; the "
                        "cross-attention / tail kernels (HBM-bound) are listed in `kernels` and in profiles/"}
    else:
        roof = {"bound": "hbm", "kernel": top["kernel"], "shape": top["shape"], "achieved": top.get("gbs"),
                "peak": hbm_peak, "unit": "GB/s", "frac": (top["gbs"] / hbm_peak) if "gbs" in top else None,
                "traffic": None, "peak_source": how, "avg_launch_us": top.get("kernel_us"),
                "algorithmic_bytes_per_launch": top.get("bytes_per_launch"),
                "note": "one launch at the pipeline's batch (B=1 text-cond pass, B=2 CFG pass) moves 0.7-11 MB: launch-"
                        "latency bound by size; profiles/ holds the batch sweep where the same kernels run "
                        "bandwidth-bound"}
    return roof, [r for r in table if "kernel_us" in r or "fwd_plus_bwd_us" in r][:14]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--unet", default="sd14", choices=["sd14", "tiny"], help="tiny is for plumbing checks only")
    ap.add_argument("--denoise-steps", type=int, default=50)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graphs", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--no-saturated", action="store_true", help="skip the large-batch kernel rooflines")
    ap.add_argument("--host-control", action="store_true",
                    help="A/B: drive refinement / recursion from the host (graph replays + one D2H read per evaluation) "
                         "instead of the device-side step driver")
    ap.add_argument("--seeds-per-batch", type=int, default=8,
                    help="also measure the seed-batched extension with this many seeds per UNet pass (0/1 = skip)")
    ap.add_argument("--sweep64", action="store_true",
                    help="BASELINE config 5: the fixed seeds range(28, 92) sharded seed_idx %% world, strong scaling, "
                         "per-seed checksums in the line")
    ap.add_argument("--sweep-seeds", type=int, default=64, help="with --sweep64: use the first n seeds of the list")
    ap.add_argument("--ref-refine-first", type=int, default=10,
                    help="reference arm / cpu_baseline: refinement iterations of the whole-round sample (10 = the "
                         "reference's max_refinement_steps)")
    ap.add_argument("--ref-refine", type=int, default=1,
                    help="reference arm: refinement iterations of the bounded samples after the first timed step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path returned in its last step (the final "
                         "latents of its image; with --sweep64 of every seed) as DIR/final_latents.npy in float32, to "
                         "compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the CUDA arm")
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
