#!/usr/bin/env python3
"""Benchmark of the HiFIC encode+decode forward hot path (Encoder -> Hyperprior -> Generator).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one pass of the hot path over one batch of B synthetic 3x256x256 images per GPU (weak scaling,
no data-path collective: samples are independent).  Prints ONE JSON line (rank 0):
  value     images/s with the batch already resident in HBM (CUDA events, max over ranks)
  e2e       the same through the public API with HOST buffers (pinned H2D of x, D2H of x_hat + q_bpp)
  roofline  the dominant kernel (960->960 3x3 residual conv, tcgen05 implicit GEMM) timed alone, live
  cpu_baseline  the CPU oracle (port of the reference path) on a bounded sample, rank 0 at N=1 only
  roofline_hbm  the conditional-likelihood kernel against the measured HBM peak (20 B/element), all three schedules
  train_step / gan_train_iteration  the training half of BASELINE.json's metric (fwd + losses + bwd + Adam; NCCL
                gradient all-reduce at N > 1), plus the same step with the native LPIPS trunk (single GPU)
  compress_path Model.compress / Model.decompress through the public API (GPU networks + symbol kernels + host rANS)
`--impl reference` times the reference's CPU implementation of the path (oracle port) instead.
`--dump-outputs DIR` writes what the last timed step returned (reconstruction, q_bpp) as DIR/<name>.npy, so that two builds
can be compared output for output: weights and images are seeded, the inputs are the same on every run.
"""
import argparse
import json
import logging
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("HFC_LPIPS_SYNTHETIC", "1")   # synthetic weights everywhere (no checkpoints offline): "data": "synthetic"

import torch  # noqa: E402

METRIC = "images/sec (256x256) encode+decode fwd"
RES_FLOPS_PER_IMAGE = 2.0 * 256 * 960 * 960 * 9       # one 960->960 3x3 conv on a 16x16 map
E_H_G_FLOPS_PER_IMAGE = 99.89e9                        # SURVEY.md 8d: forward, per 256x256 image


def env_int(name, default):
    return int(os.environ.get(name, default))


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(burst=float(d["bf16_tflops"]), sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    hbm=float(d["hbm_gbs"]), source="measured (MEASURED_PEAKS.json)")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        load = [s for s, p in zip(sm, power) if p > 250] or sm
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(power) if power else None}


def oracle_forward_factory(batch):
    """CPU port of the reference path (the oracle), eval mode, forward only."""
    from hific_b200 import synth
    from oracle import hific_oracle as O
    sd = synth.synth_state_dict(0)
    x = synth.synth_image(batch, 256, 256, 0)

    def step():
        with torch.no_grad():
            recon, hyper, _ = O.compression_forward(sd, x, training=False)
        return recon, hyper

    return step


def pick_cpu_threads(sample_b):
    """The CPU arm gets the thread count that serves it best: torch's intra-op pool over-subscribes badly on
    many-core hosts (128 threads were ~30x slower than 8 on this workload), so a few counts are probed with
    one untimed forward each and the fastest is used for the timed run."""
    total = os.cpu_count() or 1
    step = oracle_forward_factory(sample_b)
    best, best_dt = total, None
    for nt in sorted({total, min(total, 64), min(total, 32), min(total, 16), min(total, 8)}, reverse=True):
        torch.set_num_threads(nt)
        step()                                   # warm-up at this thread count
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if best_dt is None or dt < best_dt:
            best, best_dt = nt, dt
        if dt > 20:                              # do not burn minutes probing hopeless settings
            continue
    torch.set_num_threads(best)
    return best, sample_b


def run_reference(args, rank):
    """`--impl reference`: the reference's own CPU implementation of the path (oracle port), rank 0 only."""
    if rank != 0:
        return
    cores, sample_b = pick_cpu_threads(4)
    step = oracle_forward_factory(sample_b)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    val = sample_b * args.steps / dt
    sample = (f"{args.steps} forward passes of {sample_b}x3x256x256 (bounded sample of the B={args.batch} workload: the CPU arm "
              f"runs batch {sample_b}, the GPU arm batch {args.batch}; images/s is per image)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, sample_b),
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(args, batch):
    return {"workload": f"c2 shapes: compression (no GAN) regime=low, batch={batch}/GPU 3x256x256, "
                        "Encoder+Hyperprior(analysis, factorized+conditional likelihood, synthesis)+Generator forward "
                        "(eval mode, ANS bypassed)",
            "per_gpu_batch": batch, "image": "3x256x256", "latent_channels": 220, "n_residual_blocks": 9,
            "l2": "no explicit flush: per-step working set (363 MB packed fp16 weights + activations) exceeds the 126 MB L2"}


def run_train_step(args, cfg, model, dev, dist, rank, world, x_host, timed):
    """One training step of the compression model as train.py runs it (train.py:137-141, 54-59): forward, losses
    (rate + distortion + LPIPS), backward through the hand-written kernels, gradient all-reduce over NCCL when
    world > 1 (coalesced, after backward), Adam on the amortization and the hyper-latent parameter groups."""
    from hific_b200.config import ModelModes
    from hific_b200.dist import allreduce_gradients
    from hific_b200.optim import Adam
    B = args.train_batch or args.batch
    model.enable_cuda_graph(False)
    model.model_mode = ModelModes.TRAINING
    model.train()
    amort = [p for m in model.amortization_models for p in m.parameters()]
    hyper = list(model.Hyperprior.hyperlatent_likelihood.parameters())
    opt_a = Adam(amort, lr=1e-4)
    opt_h = Adam(hyper, lr=1e-4)
    x = x_host[:B].to(dev)
    params = amort + hyper
    # multi-GPU: three ways to get the gradients averaged and the step taken, all timed at every N > 1 (the fastest is the
    # headline, the others are reported beside it -- DESIGN.md section 4):
    #   plain      one coalesced in-place NCCL all-reduce after backward, then Adam
    #   pipelined  the same collective cut in 64 MB buckets on a side stream, the Adam launch of bucket i waiting for
    #              bucket i only (hific_b200.dist.allreduce_then_step): Adam runs underneath the rest of the collective
    #   in-backward 32 MB buckets handed over layer by layer from inside the network Functions
    #              (hific_b200.dist.InBackwardGradientReducer)
    # The two non-plain modes are self-checked against the plain all-reduce once before timing; a mode that disagrees
    # (or raises) is dropped on every rank.
    PLAIN = "after backward, one coalesced NCCL all-reduce"
    modes = {"plain": PLAIN} if dist is not None else {"single": "none (single GPU)"}
    reducer = None
    if dist is not None and os.environ.get("HFC_OVERLAP_ALLREDUCE", "1") != "0":
        from hific_b200.dist import InBackwardGradientReducer, allreduce_then_step, reducer_group
        probe = [amort[0], amort[len(amort) // 2], amort[-1], hyper[0]]

        class _NoStep:                       # allreduce_then_step's communication half alone (gradients stay inspectable)
            def __init__(self, ps):
                self.param_groups = [{"params": ps}]

            def step_subset(self, group, ps):
                pass

            def step(self):
                pass

        def grads_once(mode):
            for p in params:
                p.grad = None
            torch.manual_seed(1234)
            loss = model(x, train_generator=True)['compression']
            if mode == "in-backward":
                with reducer:
                    loss.backward()
                reducer.reduce_rest(hyper)
            elif mode == "pipelined":
                loss.backward()
                allreduce_then_step(_NoStep(amort), dist, world)
                allreduce_gradients(hyper, dist, world)
            else:
                loss.backward()
                allreduce_gradients(params, dist, world)
            torch.cuda.synchronize()
            return [p.grad.detach().clone() for p in probe]

        def agree(ok):
            flag = torch.tensor([1.0 if ok else 0.0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            return flag.item() >= 1.0

        def close(ref, got):
            return all(torch.allclose(a, b, rtol=2e-2, atol=1e-3 * float(a.abs().max()) + 1e-12) for a, b in zip(ref, got))

        try:
            reducer = InBackwardGradientReducer(dist, world, group=reducer_group(dist))
            grads_once("in-backward")                              # calibrates the loss scales (per-Function hand-over)
            ref = grads_once("plain")
        except Exception:
            reducer, ref = None, None
        if agree(ref is not None):
            for mode, label in (("in-backward", "overlapped with backward: {n} buckets of <= 32 MB handed over layer by layer from inside "
                                                "the network Functions, all-reduced (ncclAvg, in place) on a side stream"),
                                ("pipelined", "after backward, in 64 MB buckets on a side stream, the Adam launch of bucket i waiting for "
                                              "bucket i only (allreduce_then_step)")):
                try:
                    ok = close(ref, grads_once(mode)) and (mode != "in-backward" or reducer.buckets_launched >= 8)
                except Exception:                    # every rank must still reach the agreement collective below
                    ok = False
                if agree(ok):
                    modes[mode] = label.format(n=reducer.buckets_launched if reducer is not None else 0) + \
                        " (self-check against the plain all-reduce passed)"
        for p in params:
            p.grad = None

    def step(mark=None, mode="plain"):
        mark = mark or (lambda: None)
        mark()
        losses = model(x, train_generator=True)
        mark()
        if mode == "in-backward":
            with reducer:
                losses['compression'].backward()
            mark()
            reducer.reduce_rest(hyper)
            mark()
            opt_a.step()
        elif mode == "pipelined":
            losses['compression'].backward()
            mark()
            mark()
            allreduce_then_step(opt_a, dist, world)
            allreduce_gradients(hyper, dist, world)
        else:
            losses['compression'].backward()
            mark()
            if dist is not None:
                allreduce_gradients(params, dist, world)
            mark()
            opt_a.step()
        opt_a.zero_grad()
        opt_h.step()
        opt_h.zero_grad()
        mark()

    def measure(mode):
        for _ in range(3):
            step(mode=mode)
        steps = max(3, args.steps // 4)
        ms = timed(lambda: step(mode=mode), steps)
        # where the step goes (3 extra untimed steps, events on the compute stream, median) and what the host needs to
        # enqueue one step onto an idle GPU (a step whose enqueue time approaches its GPU time is launch-bound)
        rows, host = [], []
        for _ in range(3):
            evs = []

            def mark():
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                evs.append(e)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            step(mark, mode)
            host.append((time.perf_counter() - t0) * 1e3)
            torch.cuda.synchronize()
            rows.append([evs[i].elapsed_time(evs[i + 1]) for i in range(4)])
        med = [sorted(r[i] for r in rows)[1] for i in range(4)]
        phases = {"forward_and_losses_ms": med[0], "backward_ms": med[1], "gradient_allreduce_after_backward_ms": med[2],
                  "adam_ms": med[3], "host_enqueue_ms": sorted(host)[1],
                  "note": "one step from an idle GPU, CUDA events on the compute stream; in-backward: the waits for the buckets "
                          "are inside backward_ms; pipelined: the collective and Adam are both inside adam_ms"}
        return ms, steps, phases

    other = None
    try:
        results = {m: measure(m) for m in modes}
        best = min(results, key=lambda m: results[m][0] / results[m][1])
        ms, steps, phases = results[best]
        reduce_mode = modes[best]
        if len(results) > 1:
            reduce_mode += " (the fastest of the modes timed at this N)"
            other = [{"ms_per_step": r[0] / r[1], "gradient_allreduce": modes[m], "phases": r[2]} for m, r in results.items() if m != best]
    except NotImplementedError as e:      # a piece of the backward is missing: report it, do not fake a number
        return {"unavailable": str(e)[:200]}
    finally:
        model.model_mode = ModelModes.EVALUATION
        model.eval()
    return {"ms_per_step": ms / steps, "images_per_s": world * B * steps / (ms * 1e-3), "steps": steps,
            "per_gpu_batch": B, "n_gpus": world, "gradient_allreduce": reduce_mode, "phases": phases,
            "other_allreduce_modes": other,
            "lpips_trunk": os.environ.get("HFC_LPIPS_TRUNK", "native"),
            "dtype": ("bf16 x bf16 backward GEMMs (HFC_GRAD_FMT=bf16)" if os.environ.get("HFC_GRAD_FMT", "fp16").lower() == "bf16" else
                      "fp16 x fp16 backward GEMMs (10-bit mantissa as TF32; power-of-two loss scale per backward Function), "
                      "fp16-operand forward, fp32 accumulate, fp32 elementwise / Adam"),
            "what": "compression model (no GAN): fwd + rate/distortion/LPIPS losses + bwd + 2x Adam (hific_b200.optim.Adam, one launch each); "
                    f"LPIPS AlexNet trunk: {os.environ.get('HFC_LPIPS_TRUNK', 'native')}; gradient all-reduce over NCCL when n_gpus > 1"}


def run_gan_steps(args, dev, dist, rank, world, x_host, timed, batch=None, regime="low", label="c4 shapes"):
    """The alternating generator / discriminator iterations of COMPRESSION_GAN training (configs c3 / c4;
    train.py:137-141): every iteration runs the full forward (E, H, G, D, all losses); generator iterations
    back-propagate the compression loss (+ beta * G loss, through D into G) and step the two Adam optimizers,
    discriminator iterations back-propagate the D loss and step the discriminator's Adam."""
    from hific_b200 import synth
    from hific_b200.config import ModelModes, ModelTypes, hific_args
    from hific_b200.dist import allreduce_gradients
    from hific_b200.model import Model
    from hific_b200.optim import Adam
    B = batch or args.gan_batch or args.train_batch or args.batch
    cfg = hific_args()
    cfg.batch_size = B
    cfg.regime = regime                                   # default_config.py: target rate / lambda_A follow the regime
    cfg.target_rate, cfg.lambda_A = cfg.target_rate_map[regime], cfg.lambda_A_map[regime]
    model = Model(cfg, logging.getLogger("bench-gan"), model_mode=ModelModes.TRAINING, model_type=ModelTypes.COMPRESSION_GAN)
    model.load_state_dict(synth.synth_state_dict(0, gan=True), strict=True)
    model.to(dev).train()
    amort = [p for m in model.amortization_models for p in m.parameters()]
    hyper = list(model.Hyperprior.hyperlatent_likelihood.parameters())
    disc = list(model.Discriminator.parameters())
    opt_a, opt_h, opt_d = (Adam(g, lr=1e-4) for g in (amort, hyper, disc))
    x = x_host[:B].to(dev)

    def allreduce(params):
        if dist is not None:
            allreduce_gradients(params, dist, world)

    # plain after-backward all-reduce by default: the in-backward reducer measured slower at every N tried (train_step times
    # both modes and says so); HFC_OVERLAP_ALLREDUCE=1 selects it here
    reducer = None
    if dist is not None and os.environ.get("HFC_OVERLAP_ALLREDUCE", "") == "1":
        from hific_b200.dist import InBackwardGradientReducer, reducer_group
        reducer = InBackwardGradientReducer(dist, world, group=reducer_group(dist))

    def g_step():
        losses = model(x, train_generator=True)
        if reducer is not None:                 # E / H / G gradients reduced from inside their backward; the discriminator's
            with reducer:                       # (stale, un-stepped on G iterations: train.py:54-59) stay local as before
                losses['compression'].backward()
            reducer.reduce_rest(hyper)
        else:
            losses['compression'].backward()
            allreduce(amort + hyper)
        opt_a.step(); opt_a.zero_grad()
        opt_h.step(); opt_h.zero_grad()

    def d_step():
        losses = model(x, train_generator=False)
        losses['disc'].backward()
        allreduce(disc)
        opt_d.step(); opt_d.zero_grad()

    try:
        for _ in range(5):                                  # >= 5 warm-up pairs: cuDNN autotune (LPIPS trunk), allocator, plans
            g_step(); d_step()
        steps = max(10, args.steps // 2)
        # every iteration is timed on its own (barrier + events, max over ranks) and the MEDIAN is reported: a 5-step mean
        # let one allocator / autotune hiccup move the figure by 60 % in round 1 (56.8 vs 34.7 ms)
        tg = sorted(timed(g_step, 1) for _ in range(steps))
        td = sorted(timed(d_step, 1) for _ in range(steps))
        ms_g, ms_d = tg[len(tg) // 2] * steps, td[len(td) // 2] * steps
    except NotImplementedError as e:
        return {"unavailable": str(e)[:200]}
    pair = (ms_g + ms_d) / steps
    return {"config": f"{label}: compression_gan regime={regime} batch={B}/GPU 3x256x256",
            "ms_per_generator_iteration": ms_g / steps, "ms_per_discriminator_iteration": ms_d / steps,
            "ms_per_generator_iteration_min_max": [tg[0], tg[-1]], "ms_per_discriminator_iteration_min_max": [td[0], td[-1]],
            "timing": f"median of {steps} individually timed iterations after 5 warm-up pairs",
            "ms_per_iteration": pair / 2, "images_per_s": world * B * 2 / (pair * 1e-3), "steps": steps, "per_gpu_batch": B,
            "n_gpus": world,
            "what": "COMPRESSION_GAN alternating iterations (train.py:137-141): full forward incl. discriminator and "
                    "LPIPS every iteration; G iterations: backward of the compression loss + 2x Adam; D iterations: "
                    "backward of the D loss + Adam; gradient all-reduce (NCCL) when n_gpus > 1"}



def _event_times(fn, warmup, reps):
    """Per-call CUDA-event times (ms) of `fn` on the current stream, after `warmup` untimed calls."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


def run_eager_cudnn(args, dev, x_host, ours_fwd_ms, ours_train_ms):
    """The real bar (BASELINE.md 4.5, SURVEY.md 8d): the reference's modules under torch-eager + cuDNN on THIS GPU.
    /root/reference does not exist on the GPU box, so the arithmetic is the oracle's functional restatement of
    Encoder / Hyperprior / Generator (src/network/encoder.py:104-111, src/hyperprior.py:277-330,
    src/network/generator.py:145-169; pinned bit-exactly to the real modules, tests/test_oracle_golden.py) run on `cuda`:
    the same F.conv2d / F.conv_transpose2d / elementwise calls the reference issues, dispatched to cuDNN by torch.
    Timed with cuDNN's TF32 convolutions (torch's default, what the reference gets on an Ampere+ GPU; cudnn.benchmark on
    as train.py:29 sets it) and with TF32 off (strict fp32).  c2 forward (eval) and the c2 training step
    (rate + distortion + LPIPS, backward, 2 x torch.optim.Adam as train.py:287-300)."""
    import torchvision
    from hific_b200 import synth
    from hific_b200.config import mse_lpips_args
    from oracle import hific_oracle as O
    B = args.batch
    cfgc = mse_lpips_args()
    cfg = dict(lambda_A=cfgc.lambda_A, lambda_B=cfgc.lambda_B, lambda_schedule=cfgc.lambda_schedule,
               target_rate=cfgc.target_rate, target_schedule=cfgc.target_schedule, k_M=cfgc.k_M, k_P=cfgc.k_P)
    sd = {k: v.to(dev) for k, v in synth.synth_state_dict(0).items()}
    x = x_host[:B].to(dev)
    state = torch.random.get_rng_state()
    torch.manual_seed(1234)
    trunk = torchvision.models.alexnet(weights=None).features.to(dev).eval()
    torch.random.set_rng_state(state)
    for p in trunk.parameters():
        p.requires_grad = False
    lins = [torch.rand(c, device=dev) * 0.02 for c in (64, 192, 384, 256, 256)]
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    out = {"what": "oracle restatement of the reference modules on cuda (torch eager + cuDNN), same synthetic weights / "
                   f"inputs, batch {B}; cudnn.benchmark = True (train.py:29)", "per_gpu_batch": B}
    try:
        torch.backends.cudnn.benchmark = True
        for tag, tf32 in (("tf32", True), ("fp32", False)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32

            def fwd():
                with torch.no_grad():
                    return O.compression_forward(sd, x, training=False)
            ts = _event_times(fwd, 3, 10)
            ms = statistics.median(ts)
            out[f"forward_{tag}"] = {"ms_per_step": ms, "images_per_s": B / (ms * 1e-3),
                                     "ours_speedup": (ms / ours_fwd_ms) if ours_fwd_ms else None}
            if args.no_train:
                continue
            sdg = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in sd.items()}
            amort = [v for k, v in sdg.items() if v.requires_grad and "hyperlatent_likelihood" not in k]
            hyper = [v for k, v in sdg.items() if v.requires_grad and "hyperlatent_likelihood" in k]
            opt_a, opt_h = torch.optim.Adam(amort, lr=1e-4), torch.optim.Adam(hyper, lr=1e-4)

            def train():
                nz = torch.rand((B, 320, 4, 4), device=dev) - 0.5
                ny = torch.rand((B, 220, 16, 16), device=dev) - 0.5
                recon, hyp, _ = O.compression_forward(sdg, x, True, False, nz, ny)
                rate, _ = O.weighted_rate_loss(cfg, hyp.total_nbpp, hyp.total_qbpp, 1)       # .item() sync, as losses.py:21
                loss = rate + cfg["k_M"] * O.distortion_loss(recon, x) + \
                    cfg["k_P"] * O.lpips_forward(trunk, lins, recon, x).mean()
                loss.backward()
                opt_a.step(); opt_h.step()
                opt_a.zero_grad(); opt_h.zero_grad()
            ts = _event_times(train, 3, 8)
            ms = statistics.median(ts)
            out[f"train_step_{tag}"] = {"ms_per_step": ms, "images_per_s": B / (ms * 1e-3),
                                        "ours_speedup": (ms / ours_train_ms) if ours_train_ms else None}
            del sdg, amort, hyper, opt_a, opt_h
            torch.cuda.empty_cache()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    return out


def run_c5_inference(model, dev, peaks, rank):
    """Config c5 (BASELINE.json): compress.py's inference path at batch 8 x 3 x 1024 x 1024, encode -> latents -> decode
    with the entropy coder bypassed (compress.py:143-150, `model(data, writeout=False)` in EVALUATION mode)."""
    B5 = 8
    from hific_b200 import synth
    x = synth.synth_image(B5, 1024, 1024, seed=7 + rank).to(dev)

    def step():
        with torch.no_grad():
            return model(x, writeout=False)
    ts = _event_times(step, 3, 10)
    ms = statistics.median(ts)
    flops = E_H_G_FLOPS_PER_IMAGE * 16 * B5
    return {"workload": "c5: compress.py inference path, batch 8 x 3x1024x1024, E + H + G forward, eval mode, ANS bypassed",
            "ms_per_step": ms, "images_per_s": B5 / (ms * 1e-3), "images_256_equiv_per_s": 16 * B5 / (ms * 1e-3),
            "tflops_per_step_algorithmic": flops / 1e12, "step_tensor_frac": flops / (ms * 1e-3) / 1e12 / peaks["sustained"],
            "timing": "median of 10 CUDA-event-timed steps after 3 warm-ups; inputs resident in HBM; working set >> L2"}


def cpu_c1_train_step(cores):
    """Config c1 (BASELINE.json configs[0], BASELINE.md 4.3): compression (no GAN), regime low, batch 4 x 3x256x256,
    ONE forward + backward step on the host cores through the oracle (rate + distortion loss; torch CPU autograd)."""
    from hific_b200 import synth
    from oracle import hific_oracle as O
    torch.set_num_threads(cores)
    sd = synth.synth_state_dict(0)
    sdg = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in sd.items()}
    x = synth.synth_image(4, 256, 256, 0)
    nz, ny = torch.rand((4, 320, 4, 4)) - 0.5, torch.rand((4, 220, 16, 16)) - 0.5
    k_M = 0.075 * 2 ** (-5)

    def step():
        for v in sdg.values():
            v.grad = None
        recon, hyp, _ = O.compression_forward(sdg, x, True, False, nz, ny)
        (2.0 * hyp.total_nbpp + k_M * O.distortion_loss(recon, x)).backward()
    step()
    n, t0 = 0, time.perf_counter()
    while n < 2 or (time.perf_counter() - t0 < 8 and n < 10):
        step()
        n += 1
    dt = (time.perf_counter() - t0) / n
    return {"ms_per_step": 1e3 * dt, "images_per_s": 4 / dt, "cores": cores, "steps": n,
            "what": "c1: batch 4 x 3x256x256 forward + backward (rate + distortion) through the CPU oracle, torch fp32"}


def ncu_dram_traffic(profile, kernel_substr):
    """DRAM bytes (read + write) per launch of a kernel from a committed `ncu --set full` summary under profiles/
    (tools/ncu_summary.py format); None when the file or the kernel is missing."""
    path = os.path.join(ROOT, "profiles", profile)
    if not os.path.exists(path):
        return None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    try:
        for rec in json.load(open(path)):
            if kernel_substr in rec.get("Kernel Name", ""):
                tot = 0.0
                for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    val, u = rec[k].split()
                    tot += float(val) * unit[u]
                return tot
    except (KeyError, ValueError, OSError):
        return None
    return None


def run_likelihood_roofline(dev, peaks, batch):
    """HBM roofline of the conditional-likelihood kernel at this batch's latent size (north_star: >= 60 % of HBM peak at
    batch 32): 20 B/element algorithmic traffic (SURVEY.md 8d), CUDA events around single launches on the launching
    stream, L2 flushed (256 MiB memset) before every launch.  All three schedules of the kernel are timed; `schedule` is the
    one hfc_latent_likelihood uses by default."""
    from hific_b200 import ops
    n = batch * 220 * 16 * 16
    g = torch.Generator(device=dev).manual_seed(0)
    y = torch.randn(n, device=dev, generator=g).view(batch, 220, 16, 16) * 2
    mu = torch.randn(n, device=dev, generator=g).view_as(y)
    s = torch.rand(n, device=dev, generator=g).view_as(y) * 2
    nz = torch.rand(n, device=dev, generator=g).view_as(y) - 0.5
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    default = os.environ.get("HFC_LIKELIHOOD_V")
    res = {}
    try:
        for v in ("1", "2", "3", "4"):
            os.environ["HFC_LIKELIHOOD_V"] = v
            sums = torch.zeros(2, dtype=torch.float64, device=dev)
            for _ in range(3):
                ops.latent_likelihood(y, mu, s, nz, sums=sums)
            ts = []
            for _ in range(20):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ops.latent_likelihood(y, mu, s, nz, sums=sums)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            ms = sum(ts) / len(ts)
            gbs = 20.0 * n / (ms * 1e-3) / 1e9
            res[v] = {"ms_per_launch": ms, "achieved": gbs, "frac": gbs / peaks["hbm"]}
    finally:
        if default is None:
            os.environ.pop("HFC_LIKELIHOOD_V", None)
        else:
            os.environ["HFC_LIKELIHOOD_V"] = default
    # what the machine gives a PLAIN copy of the same traffic at this size (16 B/element read, 4 B/element written, L2
    # flushed, same event bracket): at 36 MB a launch is mostly DRAM ramp + drain, so the floor is far from the 2 GB-copy
    # peak the fraction is quoted against -- the kernel's distance to this floor is what a better schedule could still win
    src = torch.empty(4 * n, dtype=torch.float32, device=dev).normal_()
    dst = torch.empty(n, dtype=torch.float32, device=dev)
    ts = []
    for _ in range(3):
        dst.copy_(src[:n])
    for _ in range(20):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.sum(src.view(4, n), dim=0, out=dst)          # reads 16 B/element, writes 4 B/element, trivial arithmetic
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    floor_ms = sorted(ts)[len(ts) // 2]
    floor = {"ms_per_launch": floor_ms, "achieved": 20.0 * n / (floor_ms * 1e-3) / 1e9,
             "frac": 20.0 * n / (floor_ms * 1e-3) / 1e9 / peaks["hbm"],
             "what": "torch.sum over a (4, n) fp32 view -> (n,): the same 20 B/element with no arithmetic to speak of"}
    used = default if default in ("1", "2", "3", "4") else "3"         # HFC_LIKELIHOOD_DEFAULT_VARIANT in csrc/elementwise.cu
    return {"kernel": "latent_likelihood_kernel (y, mean, scale, noise -> y_hat, 2 log-likelihood sums), %d elements" % n,
            "bound": "hbm", "achieved": res[used]["achieved"], "peak": peaks["hbm"], "unit": "GB/s",
            "frac": res[used]["frac"],
            "traffic": ncu_dram_traffic("r01_ncu_symbols_likelihood.json", "latent_likelihood_v2_kernel<1, 1>"),
            "traffic_source": "dram bytes of one launch at this size, profiles/r01_ncu_symbols_likelihood.json (ncu --set full)",
            "ms_per_launch": res[used]["ms_per_launch"],
            "algorithmic_bytes_per_launch": 20 * n, "schedule": used, "schedules": res, "same_traffic_floor": floor,
            "peak_source": peaks["source"] + ", HBM copy bandwidth", "l2": "flushed (256 MiB memset) before every timed launch"}


def run_symbols_roofline(dev, peaks):
    """HBM roofline of the compress-path kernel at the c5 latent size (8 x 220 x 64 x 64): hfc_quantize_symbols with
    symbols + table indices + Shannon estimate = 12 B read + 8 B written per element (DESIGN.md 3.7); CUDA events, L2
    flushed before every launch."""
    from hific_b200 import ops
    from hific_b200._lib import SYM_BATCH_STEPS, SYM_PIXEL_STEPS
    from hific_b200.compression.prior_model import prior_scale_table
    table = torch.clamp(prior_scale_table(), 0.11).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {}
    for name, shape, layout in (("batch_steps_8x220x64x64", (8, 220, 64, 64), SYM_BATCH_STEPS),
                                ("pixel_steps_1x220x64x64", (1, 220, 64, 64), SYM_PIXEL_STEPS)):
        g = torch.Generator(device=dev).manual_seed(0)
        y = torch.randn(shape, device=dev, generator=g) * 3
        mu = torch.randn(shape, device=dev, generator=g)
        sc = torch.rand(shape, device=dev, generator=g) * 3
        for _ in range(3):
            ops.quantize_symbols(y, mu, sc, table, 0.11, "gaussian", layout, want_bits=True)
        ts = []
        for _ in range(10):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ops.quantize_symbols(y, mu, sc, table, 0.11, "gaussian", layout, want_bits=True)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ms = sorted(ts)[len(ts) // 2]          # median: the output allocations inside the wrapper add jitter
        gbs = 20.0 * y.numel() / (ms * 1e-3) / 1e9
        out[name] = {"ms_per_launch": ms, "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs / peaks["hbm"],
                     "algorithmic_bytes_per_launch": 20 * y.numel()}
    out["kernel"] = "quantize_symbols_{flat,transposed}_kernel (symbols, table indices, Shannon estimate), bound: hbm"
    return out


def run_compress_path(model, dev, x_host):
    """compress.py's path through the public API (Model.compress -> CompressionOutput -> Model.decompress): GPU networks
    and symbol kernels + the host rANS coder; wall clock with a device synchronisation on both sides."""
    model.enable_cuda_graph(False)
    t0 = time.perf_counter()
    model.Hyperprior.hyperprior_entropy_model.build_tables()          # compress.py:61,122 (host, once per checkpoint)
    out = {"hyper_table_build_s": time.perf_counter() - t0}
    for b in sorted({1, min(8, x_host.shape[0])}):
        x = x_host[:b].to(dev)
        co = model.compress(x, silent=True)
        model.decompress(co)
        torch.cuda.synchronize()
        n = 3
        t0 = time.perf_counter()
        for _ in range(n):
            co = model.compress(x, silent=True)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        for _ in range(n):
            rec = model.decompress(co)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        out[f"batch{b}"] = {"compress_ms": 1e3 * (t1 - t0) / n, "decompress_ms": 1e3 * (t2 - t1) / n,
                            "message_bytes": 4 * (len(co.hyperlatents_encoded) + len(co.latents_encoded)),
                            "estimated_bits": co.total_bits, "coder_lanes": "channels" if b == 1 else "C*H*W"}
    out["what"] = ("Model.compress / Model.decompress on b x 3x256x256 (random-init weights: ~10 bpp, far above a trained "
                   "model's rate): Encoder/Hyperprior/Generator kernels + hfc_quantize_symbols / hfc_scale_indices / "
                   "hfc_dequantize_symbols on the GPU, rANS coder (bit-compatible with the reference's) on one host core")
    return out


def dump_outputs(out_dir, outputs, rank, world, budget=64 << 20):
    """Write each output tensor as out_dir/<name>.npy in float32 (`<name>_rank<r>.npy` at N > 1).  A tensor larger than
    its share of `budget` is replaced by a fixed, seeded sample of its flattened elements (the same indices on every run
    with the same arguments)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = budget // (world * len(outputs))
    for name, t in outputs.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, f"{name}.npy" if world == 1 else f"{name}_rank{rank}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step measurement")
    ap.add_argument("--train-batch", type=int, default=0, help="per-GPU batch of the training step (default: --batch)")
    ap.add_argument("--gan-batch", type=int, default=0, help="per-GPU batch of the GAN iterations (default: the training batch)")
    ap.add_argument("--no-gan", action="store_true", help="skip the COMPRESSION_GAN alternating-iteration measurement")
    ap.add_argument("--no-compress", action="store_true", help="skip the Model.compress / decompress measurement")
    ap.add_argument("--no-eager", action="store_true", help="skip the torch-eager + cuDNN comparison and the c5 inference leg")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying a CUDA graph")
    ap.add_argument("--profile", action="store_true",
                    help="profiling mode (ncu): device-resident steps only, no e2e / roofline / CPU legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)

    if args.impl == "reference":
        run_reference(args, rank)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hific_b200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from hific_b200 import ops, synth
    from hific_b200.config import ModelModes, ModelTypes, mse_lpips_args
    from hific_b200.model import Model

    cfg = mse_lpips_args()
    cfg.batch_size = args.batch
    model = Model(cfg, logging.getLogger("bench"), model_mode=ModelModes.EVALUATION, model_type=ModelTypes.COMPRESSION)
    model.load_state_dict(synth.synth_state_dict(0), strict=False)    # identical weights on every rank; EVALUATION mode adds coder tables
    model.to(dev).eval()
    B = args.batch
    x_host = synth.synth_image(B, 256, 256, seed=1 + rank).pin_memory()  # rank-offset data seed
    x_dev = x_host.to(dev)
    out_host = torch.empty((B, 3, 256, 256), dtype=torch.float32).pin_memory()
    bpp_host = torch.empty((), dtype=torch.float32).pin_memory()

    last = {}

    def step_device():
        with torch.no_grad():
            last["reconstruction"], last["q_bpp"] = model(x_dev, writeout=False)
            return last["reconstruction"], last["q_bpp"]

    # end to end through the public API with HOST buffers: every step copies its input from pinned host memory and
    # its result back; hific_b200.pipeline.PipelinedForward double-buffers the copies on their own streams so that
    # they overlap the kernels of the neighbouring steps (all copies stay inside the timed region)
    from hific_b200.pipeline import PipelinedForward
    pipe = PipelinedForward(model, depth=2)
    pending = []

    def step_e2e():
        pending.append(pipe.submit(x_host))
        if len(pending) > 1:
            recon_h, bpp_h = pipe.result(pending.pop(0))      # the host consumes the previous step's result
            assert recon_h.shape == out_host.shape

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, finalize=None):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            fn()
        if finalize is not None:
            finalize()              # e.g. make the timing stream wait for copies still in flight on side streams
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    # kernels launched per step, counted on one eager step (graph replays do not pass through the C ABI)
    step_device()
    torch.cuda.synchronize()
    l0 = ops.launch_count()
    step_device()
    launches_per_step = ops.launch_count() - l0
    use_graph = not (args.no_graph or args.profile)
    if use_graph:
        model.enable_cuda_graph(True)
    for _ in range(args.warmup if args.profile else max(args.warmup, 3)):
        step_device()
    torch.cuda.synchronize()
    if args.profile:
        ms = timed(step_device, args.steps)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last, rank, world)
        if rank == 0:
            print(json.dumps({"profile_mode": True, "ms_per_step_under_profiler": ms / args.steps}))
        return

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms = timed(step_device, args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last, rank, world)
    launches = launches_per_step * args.steps
    for _ in range(2):
        step_e2e()
    pipe.drain()
    pending.clear()
    ms_e2e = timed(step_e2e, args.steps, finalize=pipe.drain)
    clocks = sampler.stop() if rank == 0 else None

    # --- roofline of the dominant kernel, timed alone on this stream (rank 0) ---
    roof = None
    if rank == 0:
        peaks = measured_peaks()
        plan = model.Generator._plans.get(torch.empty((B, 220, 16, 16), device=dev))
        blk = model.Generator.resblock_0
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        plain = plan.res_convs[0][0]
        fused = plan.fused[0][0] if plan.fused is not None else None

        def run_plain():
            plain(plan.act_a, blk.conv1.weight, blk.conv1.bias, out=plan.rows)

        def run_fused():       # what the step launches 18 x: conv + ChannelNorm + ReLU + reflected border in one kernel
            fused.call_widenorm(plan.act_a, blk.conv1.weight, blk.conv1.bias, blk.norm1.gamma, blk.norm1.beta, out_act=plan.act_b)

        def time_alone(fn, reps=20):
            for _ in range(3):
                fn()
            tot = 0.0
            for _ in range(reps):
                flush.zero_()                               # evict weights/activations: cold-L2 launch, as in the step
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                tot += e0.elapsed_time(e1)
            return tot / reps

        flops = RES_FLOPS_PER_IMAGE * B
        ms_plain = time_alone(run_plain)
        ms_fused = time_alone(run_fused) if fused is not None else None
        k_ms = ms_fused if fused is not None else ms_plain
        achieved = flops / (k_ms * 1e-3) / 1e12
        ncu_file, ncu_kernel = (("r02_ncu_resconv_widenorm.json", "conv_igemm_kernel<1, 2, 1, 0>") if fused is not None
                                else ("r01_ncu_resconv_v9.json", "conv_igemm_kernel<1, 2>"))
        roof = {"kernel": ("conv_igemm_kernel<pair, 2 N tiles, widenorm> (Generator residual conv 960->960 3x3 fused with its 960-channel "
                           "ChannelNorm + ReLU + reflected border: the launch the step issues 18 x; M=%d N=960 K=8640)" % (B * 256))
                if fused is not None else
                "conv_igemm_kernel (Generator residual conv 960->960 3x3, M=%d N=960 K=8640)" % (B * 256),
                "bound": "tensor", "achieved": achieved, "peak": peaks["burst"], "unit": "TFLOP/s",
                "frac": achieved / peaks["burst"],
                "traffic": ncu_dram_traffic(ncu_file, ncu_kernel),
                "traffic_source": f"dram__bytes_read.sum + dram__bytes_write.sum of one launch, profiles/{ncu_file} "
                                  "(ncu --set full; the operands of this GEMM are L2-resident re-reads, DRAM sees the weights once)",
                "ms_per_launch": k_ms,
                "algorithmic_flops_per_launch": flops, "peak_source": peaks["source"] + ", bf16 burst",
                "l2": "flushed (256 MiB memset) before every timed launch",
                "conv_alone": {"what": "the same GEMM without the fused norm epilogue (fp32 rows out; round 1's dominant kernel, "
                                       "still the training forward's)", "ms_per_launch": ms_plain,
                               "frac": flops / (ms_plain * 1e-3) / 1e12 / peaks["burst"]},
                "step_tensor_frac": (E_H_G_FLOPS_PER_IMAGE * B / (ms / args.steps * 1e-3) / 1e12) / peaks["sustained"]}

    # --- training step (config c2: compression model, fwd + bwd + Adam), second half of BASELINE.json's metric ---
    train = None
    if not args.no_train:
        train = run_train_step(args, cfg, model, dev, dist, rank, world, x_host, timed)

    gan = gan_c3 = None
    if not args.no_train and not args.no_gan:
        # c4 shapes (regime low, batch 32 per GPU) at every N: the weak-scaling series of the GAN step; at N = 1 also c3
        # exactly as BASELINE.json states it (regime med, batch 16)
        gan = run_gan_steps(args, dev, dist, rank, world, x_host, timed, regime="low", label="c4 shapes")
        if world == 1 and not args.gan_batch:
            gan_c3 = run_gan_steps(args, dev, dist, rank, world, x_host, timed, batch=16, regime="med", label="c3")

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores, sb = pick_cpu_threads(4)
        step = oracle_forward_factory(sb)
        step()
        n, t0 = 0, time.perf_counter()
        while n < 3 or (time.perf_counter() - t0 < 10 and n < 50):
            step()
            n += 1
        dt = time.perf_counter() - t0
        cpu = {"value": sb * n / dt, "unit": "images/s", "cores": cores, "kind": "port",
               "sample": f"{n} forward passes of {sb}x3x256x256 through the CPU oracle (torch fp32, best of probed thread counts: {cores} of {os.cpu_count()} cores)",
               "batch_note": f"CPU sample batch {sb} vs GPU batch {B}: throughput in images/s is per image, the batch differs"}
        try:
            cpu["c1_train_step"] = cpu_c1_train_step(cores)
        except Exception as e:
            cpu["c1_train_step"] = {"unavailable": repr(e)[:200]}

    # --- compress / decompress through the public API, then the HBM roofline of the likelihood kernel (rank 0) ---
    comp, lik = None, None
    if rank == 0 and world == 1 and not args.no_compress:
        try:
            comp = run_compress_path(model, dev, x_host)
        except Exception as e:          # never lose the headline line to an auxiliary measurement
            comp = {"unavailable": repr(e)[:300]}
    if rank == 0:
        try:
            lik = run_likelihood_roofline(dev, measured_peaks(), B)
        except Exception as e:
            lik = {"unavailable": repr(e)[:300]}
        if isinstance(comp, dict) and "unavailable" not in comp:
            try:
                comp["symbols_kernel"] = run_symbols_roofline(dev, measured_peaks())
            except Exception as e:
                comp["symbols_kernel"] = {"unavailable": repr(e)[:300]}

    # --- the training step once more with the LPIPS AlexNet trunk on cuDNN + torch autograd (HFC_LPIPS_TRUNK=cudnn; the
    # native tcgen05 trunk is the default since round 2): kept so that the choice stays backed by a number.  Single GPU.
    if world == 1 and isinstance(train, dict) and "ms_per_step" in train and os.environ.get("HFC_LPIPS_TRUNK") is None:
        try:
            os.environ["HFC_LPIPS_TRUNK"] = "cudnn"
            t2 = run_train_step(args, cfg, model, dev, dist, rank, world, x_host, timed)
            train["with_cudnn_lpips_trunk"] = {k: t2[k] for k in ("ms_per_step", "images_per_s") if k in t2} or t2
        except Exception as e:
            train["with_cudnn_lpips_trunk"] = {"unavailable": repr(e)[:200]}
        finally:
            os.environ.pop("HFC_LPIPS_TRUNK", None)

    eager = c5 = None
    if rank == 0 and world == 1 and not args.no_eager:
        model.enable_cuda_graph(use_graph)
        try:
            c5 = run_c5_inference(model, dev, measured_peaks(), rank)
        except Exception as e:
            c5 = {"unavailable": repr(e)[:300]}
        torch.cuda.empty_cache()
        try:
            eager = run_eager_cudnn(args, dev, x_host, ms / args.steps,
                                    train.get("ms_per_step") if isinstance(train, dict) else None)
        except Exception as e:
            eager = {"unavailable": repr(e)[:300]}

    if rank == 0:
        per_step = ms / args.steps
        print(json.dumps({
            "metric": METRIC, "value": world * B * args.steps / (ms * 1e-3), "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16 operands, fp32 accumulate (tcgen05 kind::f16); fp32 elementwise",
            "data": "synthetic", "config": workload_config(args, B),
            "e2e": {"value": world * B * args.steps / (ms_e2e * 1e-3), "unit": "images/s",
                    "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": out_host.numel() * 4 + 4,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches, "gpu_launches_per_step": launches_per_step, "cuda_graph": use_graph,
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
            "tflops_per_step_algorithmic": E_H_G_FLOPS_PER_IMAGE * B / 1e12,
            "train_step_ms": train.get("ms_per_step") if isinstance(train, dict) else None,
            "train_step_dtype": train.get("dtype") if isinstance(train, dict) else None,
            "gan_generator_iteration_ms": gan.get("ms_per_generator_iteration") if isinstance(gan, dict) else None,
            "gan_discriminator_iteration_ms": gan.get("ms_per_discriminator_iteration") if isinstance(gan, dict) else None,
            "eager_cudnn": eager, "c5_inference": c5,
            "train_step": train, "gan_train_iteration": gan, "c3_gan_train_iteration": gan_c3,
            "roofline_hbm": lik, "compress_path": comp,
        }))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
