"""Benchmark of the Stable Audio denoising hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config {2,3,4,5}] [--impl reference] [--dump-outputs DIR]

Default workload = BASELINE.json configs[2] (--config 3, the configuration the metric is quoted on): Stable Audio
Open 1.0 DiT (1.06 B parameters, random init), 47.55 s stereo 44.1 kHz = 1024 latent tokens, batch 4 per GPU with
classifier-free guidance (8 transformer rows), dpmpp-3m-sde sampler, synthetic conditioning; one "step" = one
sampler iteration = one CFG denoiser call + the sampler update.  `value` = denoise steps per second summed over all
ranks (weak scaling: every rank runs its own batch, sharded like the reference's generate.py:119-120).  Extra keys
report audio-seconds/s for a full 100-step generation (100 x step time + the measured Oobleck decode).
Other BASELINE configurations (SURVEY.md 8d): --config 2 = one prompt (2 rows); --config 4 = 64 prompts over 8 GPUs =
batch 8 per GPU (16 rows); --config 5 = the SA-2.0 length (6144 latents + prepend = 6145 tokens), one prompt per GPU.

--impl reference times the reference's CPU path (the oracle port of the same DiT forward) with every host thread it
can use, on a bounded sample of the same workload: the WHOLE batch of the configuration in one call through d of the
24 identical blocks, scaled by 24 / d.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "friendly-stable-audio-tools_b200")
for p in (ROOT, PKG, os.path.join(ROOT, "profiles", "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "denoise_steps_per_s"
UNIT = "steps/s"
SAO_DIT = dict(io_channels=64, embed_dim=1536, depth=24, num_heads=24, cond_token_dim=768, global_cond_dim=1536,
               project_cond_tokens=False, transformer_type="continuous_transformer")
SAO_DEC = dict(out_channels=2, channels=128, c_mults=[1, 2, 4, 8, 16], strides=[2, 4, 4, 8, 8], latent_dim=64,
               use_snake=True, final_tanh=False)
CTX_LEN = 130              # 128 T5 tokens + seconds_start + seconds_total
CFG_SCALE = 7.0
GEN_STEPS = 100
SIGMA_MIN, SIGMA_MAX = 0.3, 500.0    # generate.py:135-136
# BASELINE.json configs (1-based like SURVEY.md 8d): per-GPU batch and latent length
CONFIGS = {
    2: dict(batch=1, latent_len=1024, name="SA-Open-1.0 DiT single denoise step, one prompt (BASELINE configs[1])"),
    3: dict(batch=4, latent_len=1024, name="SA-Open-1.0 100-step generation, batch 4 per GPU (BASELINE configs[2])"),
    4: dict(batch=8, latent_len=1024, name="64 prompts over 8 GPUs = batch 8 per GPU (BASELINE configs[3])"),
    5: dict(batch=1, latent_len=6144, name="SA-2.0 length, 6144 latents (285 s), one prompt per GPU (BASELINE configs[4])"),
}
BATCH, LATENT_LEN = 4, 1024          # set from --config in main()
AUDIO_SECONDS = 2097152 / 44100.0


def set_config(idx):
    global BATCH, LATENT_LEN, AUDIO_SECONDS
    BATCH, LATENT_LEN = CONFIGS[idx]["batch"], CONFIGS[idx]["latent_len"]
    AUDIO_SECONDS = LATENT_LEN * 2048 / 44100.0


def flops_per_step(B):
    """SURVEY.md 8(d): algorithmic FLOPs of one CFG denoise step (2*B rows, cross-attention counted
    only on the B conditional rows, the uncond rows' context is null)."""
    N, D, M, ctx, ffi = LATENT_LEN + 1, 1536, CTX_LEN, 768, 6144
    self_f = 2 * N * D * 3 * D + 4 * N * N * D + 2 * N * D * D
    cross_f = 2 * N * D * D + 4 * N * M * D + 2 * N * D * D          # q, core, out (k/v are step-invariant)
    ff_f = 2 * N * D * 2 * ffi + 2 * N * ffi * D
    per_row = 24 * (self_f + ff_f) + 2 * N * 64 * D * 2
    return 2 * B * per_row + B * 24 * cross_f


def config_dict(args, extra=None):
    c = {"workload": f"SA-Open-1.0 DiT denoise step, {AUDIO_SECONDS:.2f} s stereo 44.1 kHz ({LATENT_LEN} latent tokens + 1 "
                     f"prepend), batch {BATCH} per GPU with CFG 7 ({2 * BATCH} rows), dpmpp-3m-sde update, synthetic "
                     f"T5-shaped conditioning [{CONFIGS[args.config]['name']}]",
         "baseline_config": args.config,
         "global_batch": BATCH * args.gpus, "latent_tokens": LATENT_LEN, "context_tokens": CTX_LEN,
         "parallelism": f"dp{args.gpus}", "l2_policy": "per-step working set (2.1 GB of 16-bit weights) exceeds the 126 MB L2"}
    if extra:
        c.update(extra)
    return c


# --------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons, power = [], None, set(), []
        for ts, line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(parts[1]))
                smax = float(parts[2])
                power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "power_w_max": max(power) if power else None, "samples": len(sm)}


def pick_threads(fn):
    """fp32 torch ops on a large host do not always run fastest on every hardware thread: probe all / half / a
    quarter of the threads on one call of `fn` and keep the fastest (reported as threads_used of threads_total)."""
    cores = os.cpu_count() or 1
    best, best_t = None, float("inf")
    for n in sorted({max(1, cores // d) for d in (1, 2, 4)}, reverse=True):
        torch.set_num_threads(n)
        fn()
        t0 = time.time()
        fn()
        dt = time.time() - t0
        if dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def cpu_inputs():
    g = torch.Generator().manual_seed(1)
    x = torch.randn(BATCH, 64, LATENT_LEN, generator=g)
    t = torch.full((BATCH,), 0.5)
    c = torch.randn(BATCH, CTX_LEN, 768, generator=g)
    ge = torch.randn(BATCH, 1536, generator=g)
    return x, t, c, ge


def cpu_sample(budget_s, n_calls):
    """The reference's CPU path on a bounded sample: the oracle port (oracle/dit_oracle.py, pinned to the reference
    modules by tests/golden) of ONE CFG denoiser call on the configuration's WHOLE batch (2 * BATCH rows in one call, so
    every host thread has work) through d of the 24 identical blocks; time scaled by 24 / d.  No batch extrapolation."""
    from oracle import dit_oracle as do
    x, t, c, ge = cpu_inputs()
    cfg1 = dict(SAO_DIT, depth=1)
    sd1 = do.make_dit_weights(cfg1, seed=0)
    with torch.no_grad():
        threads = pick_threads(lambda: do.dit_forward(sd1, cfg1, x, t, c, ge, cfg_scale=CFG_SCALE))
        t0 = time.time()
        do.dit_forward(sd1, cfg1, x, t, c, ge, cfg_scale=CFG_SCALE)
        block_s = time.time() - t0
    d = int(max(1, min(24, (budget_s / max(1, n_calls)) / max(block_s, 1e-3))))
    cfg = dict(SAO_DIT, depth=d)
    sd = sd1 if d == 1 else do.make_dit_weights(cfg, seed=0)
    return do, cfg, sd, (x, t, c, ge), d, threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    do, cfg, sd, (x, t, c, ge), d, threads = cpu_sample(150.0, args.steps + args.warmup)
    times = []
    with torch.no_grad():
        for i in range(args.warmup + args.steps):
            t0 = time.time()
            do.dit_forward(sd, cfg, x, t, c, ge, cfg_scale=CFG_SCALE)
            if i >= args.warmup:
                times.append(time.time() - t0)
    step_s = sum(times) / len(times) * (24.0 / d)
    value = 1.0 / step_s
    sample = (f"all {BATCH} prompts ({2 * BATCH} CFG rows) in one call through {d} of 24 blocks per step, fp32, "
              f"{threads} of {os.cpu_count()} host threads; scaled x{24.0 / d:.2f} (depth only)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "threads_total": os.cpu_count(),
                             "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# --------------------------------------------------------------------------- native arm
def build_models(device):
    from oracle import dit_oracle as do
    from oracle import oobleck_oracle as oo
    from stable_audio_tools.models.autoencoders import OobleckDecoder
    from stable_audio_tools.models.diffusion import DiTWrapper
    wrapper = DiTWrapper(**SAO_DIT)
    # random-init weights of the SA-Open-1.0 architecture (no checkpoint exists offline); the reference
    # zero-inits every branch output, which would make the step trivially sparse, so use the
    # re-randomised synthetic weights of the parity tests.
    wrapper.model.load_state_dict(do.make_dit_weights(SAO_DIT, seed=0))
    wrapper = wrapper.to(device).eval()
    dec = OobleckDecoder(**SAO_DEC)
    dec.load_state_dict(oo.make_oobleck_weights(oo.decoder_param_shapes(SAO_DEC), seed=1,
                                                transposed=oo.decoder_transposed_prefixes(SAO_DEC)))
    dec = dec.to(device).eval()
    return wrapper, dec


DUMP_MAX_ELEMENTS = 1 << 22        # per array: 16 MB of float32, so the three dumped arrays stay under 64 MB


def dump_outputs(directory, outputs):
    """Write each output as <directory>/<name>.npy in float32.  An array larger than DUMP_MAX_ELEMENTS is written as a
    fixed seeded sample of its flattened elements (the same positions in every run of the same configuration), so
    that the dumps of two builds can be compared element for element."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in outputs.items():
        flat = t.detach().reshape(-1)
        if flat.numel() > DUMP_MAX_ELEMENTS:
            idx = torch.randint(flat.numel(), (DUMP_MAX_ELEMENTS,), generator=torch.Generator().manual_seed(0))
            flat = flat[idx.sort().values.to(flat.device)]
        else:
            flat = flat.reshape(t.shape)
        np.save(os.path.join(directory, name + ".npy"), flat.float().cpu().numpy())


def cpu_baseline_leg():
    """Same bounded sample as --impl reference, ~10-20 s of host time."""
    do, cfg, sd, (x, t, c, ge), d, threads = cpu_sample(6.0, 1)
    with torch.no_grad():
        n, t0 = 0, time.time()
        while n < 2 or time.time() - t0 < 10.0:
            do.dit_forward(sd, cfg, x, t, c, ge, cfg_scale=CFG_SCALE)
            n += 1
        per = (time.time() - t0) / n
    step_s = per * (24.0 / d)
    return {"value": 1.0 / step_s, "unit": UNIT, "cores": threads, "threads_total": os.cpu_count(), "kind": "port",
            "sample": f"{n} x (all {BATCH} prompts = {2 * BATCH} CFG rows in one call, {d} of 24 blocks) fp32 on {threads} of "
                      f"{os.cpu_count()} host threads, scaled x{24.0 / d:.1f} (depth only)"}


def run_native(args):
    from stable_audio_tools import _native
    from stable_audio_tools.inference.sampling import VDenoiser, get_sigmas_polyexponential
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = world > 1
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if dist:
        import torch.distributed as td
        td.init_process_group("nccl", device_id=device)
    wrapper, dec = build_models(device)
    lib = _native.lib()

    # conditioning for the whole job is produced on rank 0 and broadcast once over NCCL (the only
    # collective of the path); each rank keeps its reference-style shard items[rank::world]
    n_total = BATCH * world
    g = torch.Generator(device="cpu").manual_seed(1234)
    cross_all = torch.randn(n_total, CTX_LEN, 768, generator=g)
    cross_all[:, 40:128] = 0.0               # padded T5 positions are exact zeros (conditioners.py:343-344)
    glob_all = torch.randn(n_total, 1536, generator=g)
    cross_all, glob_all = cross_all.to(device), glob_all.to(device)
    if dist:
        if rank != 0:
            cross_all.zero_()
            glob_all.zero_()
        td.broadcast(cross_all, 0)
        td.broadcast(glob_all, 0)
    cross = cross_all[rank::world].contiguous()
    glob = glob_all[rank::world].contiguous()
    mask = torch.ones(BATCH, CTX_LEN, device=device)
    cond = dict(cross_attn_cond=cross, cross_attn_mask=mask, global_cond=glob, cfg_scale=CFG_SCALE, batch_cfg=True,
                rescale_cfg=True)

    denoiser = VDenoiser(wrapper)
    sigmas = get_sigmas_polyexponential(GEN_STEPS, SIGMA_MIN, SIGMA_MAX, 1.0, device=device)
    sig = [float(s) for s in sigmas]
    torch.manual_seed(100 + rank)
    x0 = torch.randn(BATCH, 64, LATENT_LEN, device=device) * sigmas[0]
    ones = torch.ones(BATCH, device=device)
    import math

    from stable_audio_tools.inference.sampling import MultistepSdeStepper

    class Loop:
        """dpmpp-3m-sde, one model call per step: the product's own stepper (inference/sampling.py), which on CUDA
        runs the VDenoiser scalings + the multistep update + the noise injection as one fused kernel."""

        def __init__(self):
            self.st = MultistepSdeStepper(denoiser, x0.clone(), sigmas, order=3, extra_args=cond)
            self.n = 0

        @property
        def x(self):
            return self.st.x

        def step(self, x_in=None):
            if x_in is not None:              # e2e: this step's latents arrive from the host
                self.st.x, self.st.x_in = x_in, None
            i = self.n % (GEN_STEPS - 1)      # stay inside the non-terminal part of the schedule
            self.n += 1
            return self.st.step(i)

    def barrier():
        if dist:
            td.barrier()
        torch.cuda.synchronize()

    # one denoiser call = one CUDA-graph launch (DiffusionTransformer.cuda_graph; MultistepSdeStepper.run() switches it
    # on by itself, bench.py drives step() directly); --no-graph measures the plain enqueue path
    dit = wrapper.model
    dit.cuda_graph = not args.no_graph
    loop = Loop()
    for _ in range(max(args.warmup, 3)):
        loop.step()
    h_dit = wrapper.model._handle(device)

    # ---------------- timed region: K steps, inputs resident in HBM -------------------------
    ms8, cnt8 = (ctypes.c_float * 8)(), (ctypes.c_int * 8)()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    launches0 = _native.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.time()
    e0.record()
    for _ in range(args.steps):
        loop.step()
    e1.record()
    barrier()
    wall1 = time.time()
    launches = _native.launch_count() - launches0
    outputs = {"latents": loop.x, "denoised": loop.st.den_1}     # what the last timed step returned / estimated
    elapsed_ms = e0.elapsed_time(e1)
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    if dist:
        tmax = torch.tensor([elapsed_ms], device=device)
        td.all_reduce(tmax, op=td.ReduceOp.MAX)
        elapsed_ms = float(tmax.item())
    ms_per_step = elapsed_ms / args.steps
    value = world * args.steps / (elapsed_ms / 1e3)

    # ---------------- e2e: same steps through the public call with HOST buffers --------------
    x_host = torch.empty(BATCH, 64, LATENT_LEN, pin_memory=True).copy_(loop.x.cpu())
    out_host = torch.empty(BATCH, 64, LATENT_LEN, pin_memory=True)
    x_dev = torch.empty(BATCH, 64, LATENT_LEN, device=device)
    loop2 = Loop()
    loop2.st.den_1, loop2.st.den_2, loop2.st.h_1, loop2.st.h_2, loop2.n = loop.st.den_1, loop.st.den_2, loop.st.h_1, loop.st.h_2, loop.n
    for _ in range(max(args.warmup, 3)):
        x_dev.copy_(x_host, non_blocking=True)
        out_host.copy_(loop2.step(x_dev), non_blocking=True)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.steps):
        x_dev.copy_(x_host, non_blocking=True)                  # H2D of this step's input latents
        out_host.copy_(loop2.step(x_dev), non_blocking=True)    # D2H of this step's result
    e3.record()
    barrier()
    e2e_ms = e2.elapsed_time(e3)
    if dist:
        tmax = torch.tensor([e2e_ms], device=device)
        td.all_reduce(tmax, op=td.ReduceOp.MAX)
        e2e_ms = float(tmax.item())
    e2e_value = world * args.steps / (e2e_ms / 1e3)
    io_bytes = BATCH * 64 * LATENT_LEN * 4

    # host-side cost of enqueueing one step (launch queue empty before, no sync after): how far the
    # GPU-bound numbers above are from being launch-bound on this box's host
    host_ms = []
    for _ in range(5):
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        loop.step()
        host_ms.append((time.perf_counter() - h0) * 1e3)
    barrier()
    host_enqueue_ms = sorted(host_ms)[len(host_ms) // 2]

    # ---------------- same K steps again with per-kernel-class CUDA events (roofline) ---------
    # (a second pass: event records between kernels would defeat the programmatic dependent
    # launches the timed region above benefits from)
    dit.cuda_graph = False                                        # events between kernels: eager enqueue
    _native.check(lib.satb_dit_profile(h_dit, 1))
    _native.check(lib.satb_dit_profile_read(h_dit, ms8, cnt8))   # clear
    barrier()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(args.steps):
        loop.step()
    p1.record()
    barrier()
    profiled_ms_per_step = p0.elapsed_time(p1) / args.steps
    _native.check(lib.satb_dit_profile_read(h_dit, ms8, cnt8))
    _native.check(lib.satb_dit_profile(h_dit, 0))
    dit.cuda_graph = not args.no_graph

    # ---------------- Oobleck decode of the batch (audio-seconds/s of a full generation) ------
    lat = loop.x / max(float(loop.x.abs().max()), 1.0)
    for _ in range(3):
        audio = dec(lat[:1])
    barrier()
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0.record()
    for _ in range(3):                           # three passes over the batch; the mean pass is reported
        for b in range(BATCH):                   # one item at a time, like the reference's iterate_batch
            audio = dec(lat[b:b + 1])
    d1.record()
    torch.cuda.synchronize()
    outputs["decoded_audio"] = audio
    decode_ms = d0.elapsed_time(d1) / 3
    if dist:
        tmax = torch.tensor([decode_ms], device=device)
        td.all_reduce(tmax, op=td.ReduceOp.MAX)
        decode_ms = float(tmax.item())
    # ---------------- the decoder at the reference's own precision (split-operand mode), for the record ---------------
    dec_x3_ms = None
    if world == 1 and args.config == 3:
        from oracle import oobleck_oracle as oo
        from stable_audio_tools.models.autoencoders import OobleckDecoder
        dec3 = OobleckDecoder(**SAO_DEC, operand_dtype="fp16x3")
        dec3.load_state_dict(oo.make_oobleck_weights(oo.decoder_param_shapes(SAO_DEC), seed=1,
                                                     transposed=oo.decoder_transposed_prefixes(SAO_DEC)))
        dec3 = dec3.to(device).eval()
        dec3(lat[:1])
        torch.cuda.synchronize()
        x0_, x1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        x0_.record()
        for _ in range(2):
            dec3(lat[:1])
        x1_.record()
        torch.cuda.synchronize()
        dec_x3_ms = x0_.elapsed_time(x1_) / 2
        del dec3
    # ---------------- other BASELINE.json shapes, for the record (single GPU only) ---------------
    # configs[1]: one prompt (2 CFG rows x 1025 tokens); configs[4]: SA-2.0 length (L = 6144 latents, 1 prompt).
    extra_shapes = {}
    if world == 1 and args.config == 3:
        for name, L_x in (("single_prompt_L1024", 1024), ("single_prompt_L6144_sa2_length", 6144)):
            xs = torch.randn(1, 64, L_x, device=device)
            ts = torch.full((1,), 0.5, device=device)
            kw = dict(cross_attn_cond=cross[:1].contiguous(), cross_attn_mask=mask[:1].contiguous(),
                      global_cond=glob[:1].contiguous(), cfg_scale=CFG_SCALE, batch_cfg=True, rescale_cfg=True)
            for _ in range(3):
                wrapper(xs, ts, **kw)
            torch.cuda.synchronize()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(10):
                wrapper(xs, ts, **kw)
            s1.record()
            torch.cuda.synchronize()
            extra_shapes[name] = {"ms_per_model_call": s0.elapsed_time(s1) / 10, "rows": 2, "tokens": L_x + 1}

    # Oobleck decoder roofline bookkeeping (SURVEY.md 8d / Appendix C), per sample: ONE byte model, shared with the
    # per-layer profile tool (profiles/tools/decoder_bytes.py): 16-bit activated copies between convolutions, the raw
    # skip stream in fp16 (2 B) with fp16 operands, 128- / 256-channel ResidualUnits fused into one launch.
    import decoder_bytes
    raw_bytes = 4 if os.environ.get("SATB_RAW") == "fp32" else 2
    dec_flops, dec_bytes = decoder_bytes.totals(LATENT_LEN, raw_bytes)
    dec_ms_sample = decode_ms / BATCH
    gen_ms = GEN_STEPS * ms_per_step + decode_ms
    audio_sec_per_s = world * BATCH * AUDIO_SECONDS / (gen_ms / 1e3)

    if rank != 0:
        if dist:
            td.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)

    # ---------------- roofline of the dominant kernel (FF-in GEMM, tensor bound) --------------
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained, kernel timed inside a long step)" \
        if "bf16_tflops_sustained" in peaks else "fallback (B200_PROFILING.md sustained 1.4 PFLOP/s)"
    M = 2 * BATCH * (LATENT_LEN + 1)
    ff_in_flops = 2.0 * M * 12288 * 1536
    peak_burst = peaks.get("bf16_tflops")
    hbm_peak = peaks.get("hbm_gbs") or 6650.0
    survey_gb = decoder_bytes.SURVEY_PER_RESUNIT_FUSED_FP32_GB * LATENT_LEN / 1024.0
    ff_in_ms = ms8[0] / max(cnt8[0], 1)
    achieved = ff_in_flops / (ff_in_ms / 1e3) / 1e12 if ff_in_ms > 0 else None
    cats = ["ff_in_gemm", "ff_out_gemm", "qkv_gemm", "self_attention", "attn_out_gemm", "cross_attention", "layernorm"]
    breakdown = {c: {"ms_per_step": ms8[i] / args.steps, "launch_groups": cnt8[i] // args.steps} for i, c in enumerate(cats)}
    step_tflops = flops_per_step(BATCH) / (ms_per_step / 1e3) / 1e12

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp16 operands, fp32 accumulate (the reference's autocast dtype)", "data": "synthetic",
        "config": config_dict(args),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": io_bytes, "d2h_bytes_per_step": io_bytes},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": f"gemm_tcgen05_2cta_kernel<EpiSwiglu, 256> (FF-in {M}x12288x1536)",
                     "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": (achieved / peak_tf) if achieved else None,
                     "frac_of_burst_peak": (achieved / peak_burst) if (achieved and peak_burst) else None,
                     # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel from the
                     # `ncu --set full` capture summarised in profiles/r01_ncu_ff_in_gemm.txt (63.2 + 62.6 MB;
                     # algorithmic A + W + out = 163.7 MB, part of the 16-bit output stays in the 126 MB L2)
                     "traffic": 125806592, "traffic_unit": "bytes per launch (ncu)", "peak_source": peak_src,
                     "avg_launch_ms": ff_in_ms},
        "cuda_graph": not args.no_graph,
        "step_tflops": step_tflops, "step_frac_of_peak": step_tflops / peak_tf,
        "step_frac_of_burst_peak": (step_tflops / peak_burst) if peak_burst else None,
        "profiled_pass_ms_per_step": profiled_ms_per_step, "host_enqueue_ms_per_step": host_enqueue_ms,
        "kernel_breakdown": breakdown,
        "decode_ms_batch": decode_ms, "audio_sec_per_s_100step": audio_sec_per_s,
        "other_shapes": extra_shapes,
        "oobleck_decoder": {"ms_per_sample": dec_ms_sample, "latents": LATENT_LEN,
                            "tflops": dec_flops / (dec_ms_sample / 1e3) / 1e12,
                            "frac_of_tensor_peak": dec_flops / (dec_ms_sample / 1e3) / 1e12 / peak_tf,
                            "algorithmic_gb_per_sample": dec_bytes / 1e9, "raw_stream_bytes": raw_bytes,
                            "hbm_gbs": dec_bytes / (dec_ms_sample / 1e3) / 1e9,
                            "frac_of_hbm_peak": dec_bytes / (dec_ms_sample / 1e3) / 1e9 / hbm_peak,
                            # the same time against SURVEY.md 8(d)'s denominator (per-ResidualUnit-fused, fp32 activations)
                            "survey_gb_per_sample": survey_gb,
                            "frac_of_hbm_peak_survey_denominator": survey_gb / (dec_ms_sample / 1e3) / hbm_peak,
                            "roofline_floor_ms": max(dec_flops / (peak_tf * 1e12), dec_bytes / (hbm_peak * 1e9)) * 1e3,
                            "byte_model": "profiles/tools/decoder_bytes.py",
                            # operand_dtype="fp16x3": 3 MMAs per product, fp32 skip stream, ~73 dB instead of ~40 dB vs fp32
                            "fp16x3_ms_per_sample": dec_x3_ms,
                            "audio_sec_per_s_100step_fp16x3": (world * BATCH * AUDIO_SECONDS /
                                                               ((GEN_STEPS * ms_per_step + BATCH * dec_x3_ms) / 1e3))
                            if dec_x3_ms else None,
                            "note": "5.16 TFLOP per 1024 latents: with the 16-bit streams of this round the decoder's "
                                    "tensor time exceeds its HBM time, i.e. the bound is the tensor pipe"},
    }
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_leg()
    emit(line)
    if dist:
        td.destroy_process_group()


_REAL_STDOUT = None


def _reserve_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL writes its version banner to
    fd 1), so fd 1 is pointed at stderr for the whole run and the JSON line goes to a private duplicate."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def main():
    _reserve_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)      # seconds-long timed region: sustained clocks, not burst
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS),
                    help="BASELINE.json configuration (1-based, SURVEY.md 8d): 2 = one prompt, 3 = batch 4 (default, the one "
                         "the metric is quoted on), 4 = batch 8 per GPU (64 prompts on 8 GPUs), 5 = SA-2.0 length")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--no-graph", dest="no_graph", action="store_true", help="enqueue every kernel of a step instead of "
                    "replaying the captured CUDA graph of the denoiser call")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="after the timed steps write, as DIR/<name>.npy (float32), rank 0's latents and denoised "
                         "estimate of the last timed step and its last decoded clip; inputs are seeded, so the same "
                         "arguments give the same inputs in every run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    set_config(args.config)
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the native path only")
        run_reference(args)
    else:
        if int(os.environ.get("WORLD_SIZE", "1")) > 1:
            args.no_cpu_baseline = True     # the CPU baseline is reported at N=1 only
        run_native(args)


if __name__ == "__main__":
    main()
