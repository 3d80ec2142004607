#!/usr/bin/env python
"""bench.py -- SD1.5 LoRA-r4 512px training step (BASELINE.json configs[1]) on N x B200.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun)
  python bench.py --impl reference ...                     (the reference's CPU path, oracle port)
  python bench.py --impl reference-cuda ...                (the reference's path on the same GPU: torch eager)

One "step" = one full Dreambooth LoRA training step at bs = 1 per GPU: text encoder (48 LoRA
sites) -> UNet (144 LoRA sites) forward, MSE, backward (dX, dA, dB; W frozen), gradient
all-reduce over the LoRA arena, global-norm clip + AdamW. Synthetic latents / token ids and
random-initialised SD1.5-shaped weights (no datasets or checkpoints offline).

Prints ONE JSON line (rank 0). `value` = images/s with inputs resident in HBM; `e2e` = the same
through the public step_host() call with pinned-host inputs (H2D) and a D2H loss read per step;
`roofline` = the fused tcgen05 LoRA-linear kernel (all 384 fwd + dX launches of one step, real
site shapes) timed live with CUDA events: algorithmic bytes / time vs the measured HBM peak;
`cpu_baseline` = the oracle port of the reference's step on the host cores (rank 0, N = 1).
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

import torch  # noqa: E402

METRIC = "sd15_lora_r4_512px_train_images_per_sec"
UNIT = "images/s"
WORKLOAD = "SD1.5 UNet+text_encoder LoRA rank=4 512x512 bf16 bs=1/GPU dreambooth step (configs[1])"


def bench_config(args, world, lora_sites=None, lora_params=None):
    """The `config` object of the JSON line -- identical keys and values for every arm of the same
    invocation, so the driver can check that both arms ran the same workload."""
    if args.tiny:
        wl = "TINY smoke config (not a bench)"
    elif args.extended:
        wl = ("SD1.5 --use_extended_lora (ResBlock Conv2d LoRA, dropout 0.1) UNet+text_encoder 512x512 bf16 "
              "bs=1/GPU (configs[2] shape)")
    elif args.res == 768 and args.rank == 16:
        wl = ("SD1.5 UNet+text_encoder LoRA rank=16 768x768 bf16 bs=1/GPU LoRA-tuning step of cli_lora_pti "
              "(configs[3] shape)")
    elif args.res != 512 or args.rank != 4:
        wl = f"SD1.5 UNet+text_encoder LoRA rank={args.rank} {args.res}x{args.res} bf16 bs=1/GPU dreambooth step"
    else:
        wl = WORKLOAD
    return {"workload": wl, "extended": bool(args.extended), "resolution": args.res, "rank": args.rank,
            "global_batch": world, "parallelism": f"dp{world}",
            "l2": "working set per step (>=1.7 GB frozen weights + activations) exceeds the 126 MB L2; no explicit flush"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def wait_ready(self, timeout=3.0):
        """nvidia-smi needs a few hundred ms before its first sample: block until it is producing."""
        t0 = time.time()
        while self.proc is not None and not self.lines and time.time() - t0 < timeout:
            time.sleep(0.02)

    def mark(self):
        """Start of the timed region (the GPU is idle and the host is about to enqueue it)."""
        self.i0 = len(self.lines)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        i1 = len(self.lines)                       # host has synchronised: the timed region is over
        time.sleep(0.08)
        self.proc.terminate()
        i0 = getattr(self, "i0", 0)
        window = self.lines[i0:max(i1, i0 + 1)] or self.lines[-1:]
        sm, mx, reasons = [], [], set()
        for ln in window:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                  "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "samples": len(sm),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
def build_models(device, dtype, seed=0, tiny=False):
    from lora_b200.host.clip import build_text_encoder
    from lora_b200.host.unet_sd15 import UNet2DConditionModel, UNetConfig
    torch.manual_seed(seed)
    with torch.device(device):
        unet = UNet2DConditionModel(UNetConfig.tiny() if tiny else UNetConfig.sd15())
        text = build_text_encoder(tiny=tiny)
    unet.requires_grad_(False)
    text.requires_grad_(False)
    unet, text = unet.to(dtype), text.to(dtype)
    if torch.device(device).type == "cuda":
        # NHWC activations/weights for the conv/GroupNorm host layers: cuDNN's tensor-core convs
        # are NHWC-native (avoids an NCHW<->NHWC transpose around every conv)
        unet = unet.to(memory_format=torch.channels_last)
    return unet, text


def site_shapes(model, tokens_by_module):
    """(M, K, N, r, has_bias) for every LoraInjectedLinear of `model`; M from the recorded calls."""
    out = []
    for m in model.modules():
        if type(m).__name__ == "LoraInjectedLinear":
            out.append((tokens_by_module[id(m)], m.linear.in_features, m.linear.out_features, m.r,
                        m.linear.bias is not None))
    return out


def fused_linear_bytes(M, K, N, r, bias, e=2):
    """SURVEY.md 8(d): algorithmic bytes of one fused LoRA-linear launch (16-bit operands):
    X + W + down + up + Y (+ bias fp32) (+ T fp32 [M,16] side output)."""
    return e * (M * K + N * K + r * K + M * N) + 4 * N * r + (4 * N if bias else 0) + 4 * M * 16


def site_families(models, tokens_by_module):
    """Launch groups of the fused kernel in one step: families of sites that share an input run as ONE
    grouped launch (lora_b200/grouping.py, learned during the eager steps), every other site alone.
    Returns a list of lists of (M, K, N, r, has_bias)."""
    fam_of, fams = {}, []
    for model in models:
        for mod in model.modules():
            st = mod.__dict__.get("_lb_groups")
            if st is None:
                continue
            for fam in {id(f): f for f in st.groups.values() if f is not None}.values():
                if not any(id(m) in fam_of for m in fam):
                    for m in fam:
                        fam_of[id(m)] = len(fams)
                    fams.append(list(fam))
    out, done = [], set()
    shape = lambda m: (tokens_by_module[id(m)], m.linear.in_features, m.linear.out_features, m.r,
                       m.linear.bias is not None)
    for model in models:
        for m in model.modules():
            if type(m).__name__ != "LoraInjectedLinear":
                continue
            f = fam_of.get(id(m))
            if f is None:
                out.append([shape(m)])
            elif f not in done:
                done.add(f)
                out.append([shape(x) for x in fams[f]])
    return out


def roofline_sweep(trainer, families, iters=10, eager_once=False):
    """Every fused-kernel launch of one step (forward: X[M,K]->Y[M,N]; dX: gY[M,N]->dX[M,K]; families
    as grouped launches) with private buffers per site, captured in one CUDA graph, CUDA-event timed."""
    from lora_b200 import ops
    dev = trainer.device
    dt = trainer.cfg.compute_dtype
    launches = []
    total_bytes = 0
    for fam in families:
        for bwd in (False, True):
            probs = []
            xs = None
            for (M, K, N, r, bias) in fam:
                m, k, n = (M, N, K) if bwd else (M, K, N)
                if bwd or xs is None:                 # forward: the family shares ONE input
                    x = torch.randn(m, k, device=dev, dtype=dt)
                    xs = x if not bwd else None
                    total_bytes += 2 * m * k
                else:
                    x = xs
                w = torch.randn(n, k, device=dev, dtype=dt) * 0.02
                a = torch.randn(r, k, device=dev)
                b = torch.randn(n, r, device=dev) * 0.01
                d16 = ops.cast_rows_pad16(a, k, 1, r, k, dt)
                bb = torch.zeros(n, device=dev) if (bias and not bwd) else None
                probs.append((x, w, bb, d16, b, r, 1, None, 1.0, r))
                total_bytes += fused_linear_bytes(m, k, n, r, bb is not None) - 2 * m * k
            launches.append(probs)

    def run():
        for probs in launches:
            if len(probs) == 1:
                (x, w, bb, d16, b, rs, cs, dg, sc, r) = probs[0]
                ops.fused_linear(x, w, bb, d16, b, rs, cs, dg, sc, r, dt, True)
            else:
                ops.fused_linear_grouped(probs, dt, True)

    if eager_once:     # ncu mode: the LAST len(launches) fused-kernel launches of the process
        run(); torch.cuda.synchronize(); run(); torch.cuda.synchronize()
        return total_bytes, float("nan"), len(launches)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run(); run()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    return total_bytes, ms, len(launches)


def conv_bytes(n, cin, cout, k, H, W, r, e=2):
    """SURVEY.md 8(d): a conv site counts the activation ONCE (not im2col-expanded): X + W + down + Y
    (16-bit) + up (fp32) + bias (fp32) + T [pixels,16] fp32."""
    P, taps = n * H * W, k * k
    return e * (P * cin + cout * taps * cin + r * taps * cin + P * cout) + 4 * cout * r + 4 * cout + 4 * P * 16


def conv_sweep(trainer, conv_sites, iters=10):
    """Every fused LoRA-conv launch of one extended step: forward (dropout mask fused into the drain,
    the configs[2] default p = 0.1) and the input gradient (per-tap T groups), real ResnetBlock2D
    shapes, private buffers, one CUDA graph, CUDA-event timed."""
    from lora_b200 import ops
    dev, dt = trainer.device, trainer.cfg.compute_dtype
    seed = torch.zeros(1, device=dev, dtype=torch.int64)
    launches, total = [], 0
    for (n, cin, cout, k, H, W, r) in conv_sites:
        taps, pad = k * k, k // 2
        x = torch.randn(n, cin, H, W, device=dev, dtype=dt).contiguous(memory_format=torch.channels_last)
        gy = torch.randn(n, cout, H, W, device=dev, dtype=dt).contiguous(memory_format=torch.channels_last)
        w = torch.randn(cout, cin, k, k, device=dev) * 0.02
        wf, wb = ops.cast_conv_weight(w, dt, True, True)
        A = torch.randn(r, cin, k, k, device=dev)
        B = torch.randn(cout, r, device=dev) * 0.01
        d16 = ops.conv_down16(A, dt, {})
        bt16 = ops.cast_rows_pad16(B, 1, r, r, cout, dt)
        bias = torch.zeros(cout, device=dev)
        A32 = A.contiguous()
        launches.append(lambda x=x, wf=wf, bias=bias, d16=d16, B=B, r=r, cout=cout, k=k, pad=pad:
                        ops.fused_conv2d(x, wf, bias, d16, B, 0, r, 1, 0, None, 1.0, r, cout, k, k, pad, pad, False,
                                         dt, True, drop_p=0.1, seed=seed))
        launches.append(lambda gy=gy, wb=wb, bt16=bt16, A32=A32, r=r, cin=cin, k=k, pad=pad, taps=taps:
                        ops.fused_conv2d(gy, wb, None, bt16, A32, taps - 1, taps, cin * taps, -1, None, 1.0, r, cin,
                                         k, k, k - 1 - pad, k - 1 - pad, True, dt, True))
        total += conv_bytes(n, cin, cout, k, H, W, r) + conv_bytes(n, cout, cin, k, H, W, r)

    def run():
        for f in launches:
            f()

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run(); run()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return total, e0.elapsed_time(e1) / iters, len(launches)


def record_tokens(unet, text):
    """Forward hooks: rows (tokens) seen by each LoRA linear in one step."""
    seen = {}
    hooks = []
    for model in (unet, text):
        for m in model.modules():
            if type(m).__name__ == "LoraInjectedLinear":
                hooks.append(m.register_forward_pre_hook(
                    lambda mod, inp: seen.__setitem__(id(mod), inp[0].numel() // inp[0].shape[-1])))
    return seen, hooks


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, trainer, loss):
    """What the timed step hands its caller after the last timed step, as float32 .npy files: the
    loss and every trained LoRA factor (the fp32 masters the model's Parameters view, unet sites
    then text encoder, up before down). Above DUMP_LIMIT_BYTES the factors are a fixed seeded sample."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    p = trainer.arena.p.detach().cpu()
    factors = torch.cat([p[o:o + n] for _, _, _, o, n in trainer.arena.entries])
    limit = (DUMP_LIMIT_BYTES - 4096) // 4          # room for the .npy headers and loss.npy
    if factors.numel() > limit:
        idx = torch.randperm(factors.numel(), generator=torch.Generator().manual_seed(0))[:limit]
        factors = factors[idx.sort().values]
    np.save(os.path.join(out_dir, "loss.npy"), np.asarray([loss], dtype=np.float32))
    np.save(os.path.join(out_dir, "lora_factors.npy"), factors.numpy().astype(np.float32))


def run_native(args):
    import torch.distributed as dist
    from lora_b200 import ops
    import lora_b200 as L
    from lora_b200.train import LoraTrainStep, StepConfig

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (native arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    torch.backends.cudnn.benchmark = True   # host-model convs: let cuDNN pick its kernels in warm-up
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # An externally set NCCL_DEBUG (the driver's communicator check reads NCCL's INFO lines) is
        # honoured as is; only when nobody asked for NCCL logging do we default to WARN. In both cases
        # stdout must carry exactly ONE JSON line, and NCCL prints its version banner / INFO lines to
        # STDOUT at communicator creation -- so fd 1 is parked on stderr while the communicator is
        # built (the lines are not lost: they land on stderr).
        if "NCCL_DEBUG" not in os.environ:
            os.environ["NCCL_DEBUG"] = os.environ.get("LB_NCCL_DEBUG", "WARN")
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.ones(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    dt = torch.bfloat16
    res = args.res
    L_lat = res // 8
    unet, text = build_models(dev, dt, seed=0, tiny=args.tiny)
    if args.extended:   # configs[2]: --use_extended_lora (ResnetBlock2D conv sites; class-default dropout 0.1)
        L.inject_trainable_lora_extended(unet, r=args.rank)
    else:
        L.inject_trainable_lora(unet, r=args.rank)
    L.inject_trainable_lora(text, target_replace_module={"CLIPAttention"}, r=args.rank)
    # reference init has up = 0 (lora.py:51); give the up factors small non-zero values so the
    # LoRA branch and all three gradients are numerically exercised (SURVEY.md 8d)
    g = torch.Generator(device=dev).manual_seed(1)
    for m in list(unet.modules()) + list(text.modules()):
        if type(m).__name__ in ("LoraInjectedLinear", "LoraInjectedConv2d"):
            m.lora_up.weight.data.normal_(0.0, 0.01, generator=g)

    cfg = StepConfig(compute_dtype=dt, use_cuda_graph=not args.no_graph,
                     capture_collective=args.capture_collective, peer_allreduce=not args.nccl_allreduce)
    seq = 77
    trainer = LoraTrainStep(unet, text, cfg, latent_shape=(1, 4, L_lat, L_lat), seq_len=seq, device=dev)
    vocab = text.config.vocab_size
    torch.manual_seed(1234 + rank)
    n_data = 4
    host_lat = [(torch.randn(1, 4, L_lat, L_lat) * 0.18215).pin_memory() for _ in range(n_data)]
    host_ids = [torch.randint(0, vocab, (1, seq)).pin_memory() for _ in range(n_data)]
    trainer.latents.copy_(host_lat[0]); trainer.input_ids.copy_(host_ids[0])

    if not args.no_group:
        L.set_grouping(True)             # q/k/v-type sites that share an input: one launch per family
    seen, hooks = record_tokens(unet, text)
    conv_seen = {}
    if args.extended:
        for m in unet.modules():
            if type(m).__name__ == "LoraInjectedConv2d":
                hooks.append(m.register_forward_pre_hook(
                    lambda mod, inp: conv_seen.__setitem__(id(mod), (inp[0].shape[0], mod.conv.in_channels,
                                                                     mod.conv.out_channels, mod.conv.kernel_size[0],
                                                                     inp[0].shape[2], inp[0].shape[3], mod.r))))
    trainer._body()                      # eager step 1: records tokens per site, learns site families
    ops.LAUNCH_COUNT = 0
    trainer._body()                      # eager step 2: the steady-state launch count
    launches_per_step = ops.LAUNCH_COUNT
    if args.roofline_only:               # ncu DRAM-traffic mode: one eager sweep of the fused kernel
        fams = site_families((unet, text), seen)
        rb, _, n_l = roofline_sweep(trainer, fams, eager_once=True)
        print(json.dumps({"roofline_only": True, "launches": n_l, "algorithmic_bytes": rb}), flush=True)
        return None
    if args.profile_steps:               # ncu launch-list mode: a few eager steps, nothing else
        for _ in range(args.profile_steps):
            trainer._body()
        torch.cuda.synchronize()
        return None
    for h in hooks:
        h.remove()
    torch.cuda.synchronize()
    trainer.prepare()                    # warm-up + CUDA-graph capture

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing (value)
    for _ in range(max(args.warmup, 3)):
        trainer.step_device()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_ready()
    barrier()
    if rank == 0:
        sampler.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        trainer.step_device()
    e1.record()
    barrier()
    ms_dev = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    loss_dev = float(trainer.loss.item())

    # ---------------- end-to-end timing (public step_host API, pinned host inputs, D2H loss)
    for i in range(3):
        trainer.step_host(host_lat[i % n_data], host_ids[i % n_data])
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for i in range(args.steps):
        hl = trainer.step_host(host_lat[i % n_data], host_ids[i % n_data])
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    loss_e2e = float(hl.item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, trainer, loss_e2e)

    t = torch.tensor([ms_dev, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = float(t[0]), float(t[1])

    out = None
    if rank == 0:
        shapes = site_shapes(unet, seen) + site_shapes(text, seen)
        fams = site_families((unet, text), seen)
        hbm_peak, peak_src = load_peaks()
        rb, rms, n_l = roofline_sweep(trainer, fams)
        achieved = rb / (rms * 1e-3) / 1e9
        traffic = None   # DRAM bytes of the same 384 launches, from the committed ncu capture
        tpath = os.path.join(ROOT, "profiles", "fused_linear_dram_traffic.json")
        if os.path.exists(tpath) and not args.tiny and not args.extended and args.res == 512 and args.rank == 4:
            with open(tpath) as fh:
                traffic = json.load(fh).get("dram_bytes_per_sweep")
        value = world * args.steps / (ms_dev * 1e-3)
        conv_roof = None
        if args.extended and conv_seen:
            cb, cms, cn = conv_sweep(trainer, list(conv_seen.values()))
            c_ach = cb / (cms * 1e-3) / 1e9
            conv_roof = {"bound": "hbm", "kernel": "fused_lora_kernel<CONV>: forward (dropout fused in the drain) + input "
                         "gradient (per-tap T groups) of every LoRA conv site of one extended step",
                         "sites": 2 * len(conv_seen), "achieved": c_ach, "peak": hbm_peak, "unit": "GB/s",
                         "frac": c_ach / hbm_peak, "launches": cn, "algorithmic_bytes": cb, "ms_per_sweep": cms,
                         "avg_launch_us": cms * 1e3 / cn, "share_of_step": cms / (ms_dev / args.steps),
                         "peak_source": peak_src}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic latents/token ids, random-init SD1.5-shaped weights",
            "config": bench_config(args, world),
            "engine": {"lora_sites": len(shapes), "lora_params": trainer.arena.n_params,
                       "cuda_graph": trainer.graph is not None, "grouped_launches": not args.no_group,
                       "graph_error": trainer.graph_error, "loss": loss_dev,
                       "graphs_per_step": (0 if trainer.graph is None else (1 if trainer.graph_update is None else 2)),
                       "grad_exchange": ("none (1 rank)" if world == 1 else
                                         ("nvlink peer reads inside lb_optim_step_dp" if trainer.peer_allreduce
                                          else "nccl all_reduce"))},
            "e2e": {"value": world * args.steps / (ms_e2e * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": trainer.h2d_bytes(), "d2h_bytes_per_step": trainer.d2h_bytes(),
                    "loss": loss_e2e},
            "gpu_launches": int(launches_per_step * args.steps * 2),
            "gpu_launches_per_step": int(launches_per_step),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "fused_lora_kernel / fused_lora_grouped_kernel / fused_lora_persistent_kernel: every forward + dX launch of the fused LoRA-linear path in one step (families grouped as in the step)",
                         "sites": 2 * len(shapes),
                         "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak, "traffic": traffic,
                         "launches": n_l, "algorithmic_bytes": rb, "ms_per_sweep": rms,
                         "avg_launch_us": rms * 1e3 / n_l,
                         "share_of_step": rms / (ms_dev / args.steps), "peak_source": peak_src},
        }
        if conv_roof is not None:
            out["roofline_conv"] = conv_roof
        if world == 1 and not args.no_cuda_baseline:
            # the reference's operator modules (oracle port) in the same host models on THIS GPU:
            # torch eager (what the reference runs) and, generously, the same step graph-replayed
            del trainer
            torch.cuda.empty_cache()
            try:
                out["cuda_eager_baseline"] = cuda_reference(dev, args, steps=args.steps, warmup=max(args.warmup, 3))
            except Exception as e:   # a baseline must never take the native line down
                out["cuda_eager_baseline"] = {"error": f"{type(e).__name__}: {e}"}
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_reference(res, args.rank, budget_s=args.cpu_budget, tiny=args.tiny)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


# ------------------------------------------------------------------------------------------------
def cpu_reference(res, rank_r, budget_s=30.0, max_steps=None, warmup=1, tiny=False):
    """The reference's own path on the host cores: oracle port (oracle/ref_modules.py,
    oracle/ref_step.py: torch-eager fp32 LoRA modules + torch.optim.AdamW + clip_grad_norm_) in
    the same SD1.5-shaped host models, full steps at the bench resolution."""
    from oracle.ref_modules import ref_inject
    from oracle.ref_step import RefDreamboothStep
    from lora_b200.host.ddpm import DDPMNoiser
    # all the host threads torch can use (torchrun exports OMP_NUM_THREADS=1 for its children)
    ncpu = os.cpu_count() or 1
    want = int(os.environ.get("LB_CPU_THREADS", "0")) or (ncpu // 2 if ncpu >= 16 else ncpu)
    if torch.get_num_threads() < want:
        torch.set_num_threads(want)
    unet, text = build_models("cpu", torch.float32, seed=0, tiny=tiny)
    us = ref_inject(unet, {"CrossAttention", "Attention", "GEGLU"}, r=rank_r)
    ts = ref_inject(text, {"CLIPAttention"}, r=rank_r)
    stepper = RefDreamboothStep(unet, text, DDPMNoiser(), us, ts)
    L_lat = res // 8
    torch.manual_seed(1234)
    lat = torch.randn(1, 4, L_lat, L_lat) * 0.18215
    ids = torch.randint(0, text.config.vocab_size, (1, 77))
    cores = torch.get_num_threads()
    t_w = time.perf_counter()
    for _ in range(warmup):
        stepper.step(lat, ids)
    t_w = (time.perf_counter() - t_w) / max(warmup, 1)
    if budget_s is None:            # --impl reference: exactly the requested number of steps
        n = max(1, int(max_steps))
    else:                           # cpu_baseline block of the native line: a bounded sample
        n = max(1, int(budget_s / max(t_w, 1e-3)))
        if max_steps is not None:
            n = min(n, max_steps)
    t0 = time.perf_counter()
    for _ in range(n):
        loss = stepper.step(lat, ids)
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n} full training step(s) at {res}x{res}, bs=1, fp32, torch eager "
                      f"{torch.__version__}, after {warmup} warm-up; os.cpu_count()={os.cpu_count()}",
            "ms_per_step": dt / n * 1e3, "steps": n, "loss": float(loss)}


def cuda_reference(dev, args, steps, warmup):
    """The reference's LoRA path on the SAME B200: its operator modules (oracle/ref_modules.py, the
    three-GEMM + elementwise torch formulation of lora.py:53-58,130-135) injected into the same host
    models, its step (oracle/ref_step.py: torch.optim.AdamW + clip_grad_norm_), torch eager -- the
    stock way the reference runs on a GPU. Also timed as ONE CUDA-graph replay per step (something
    the reference does not do) so that launch latency is taken out of the comparison. Two precision
    set-ups: "bf16_model" = the native arm's host-model dtype (the reference casts its LoRA modules
    to the weight dtype, lora.py:295); "autocast" = accelerate's mixed_precision=bf16
    (fp32 weights + torch.autocast, train_lora_dreambooth.py:489-494)."""
    from oracle.ref_modules import ref_inject
    from oracle.ref_step import RefDreamboothStep
    from lora_b200.host.ddpm import DDPMNoiser
    L_lat = args.res // 8
    out = {"unit": UNIT, "kind": "port", "steps": steps, "warmup": warmup,
           "what": "oracle port of the reference step (RefLoraSite modules, torch.optim.AdamW, clip_grad_norm_) "
                   f"on cuda, torch {torch.__version__}"}
    for mode in (("bf16_model", "autocast") if not args.tiny else ("bf16_model",)):
        mdt = torch.bfloat16 if mode == "bf16_model" else torch.float32
        unet, text = build_models(dev, mdt, seed=0, tiny=args.tiny)
        targets = {"CrossAttention", "Attention", "GEGLU"}
        if args.extended:
            us = ref_inject(unet, targets | {"ResnetBlock2D"}, r=args.rank, extended=True)
        else:
            us = ref_inject(unet, targets, r=args.rank)
        ts = ref_inject(text, {"CLIPAttention"}, r=args.rank)
        g = torch.Generator(device=dev).manual_seed(1)
        for st in us + ts:
            st.up.data.normal_(0.0, 0.01, generator=g)
        stepper = RefDreamboothStep(unet, text, DDPMNoiser(device=dev), us, ts,
                                    autocast_dtype=(torch.bfloat16 if mode == "autocast" else None), capturable=True)
        torch.manual_seed(1234)
        lat = torch.randn(1, 4, L_lat, L_lat, device=dev) * 0.18215
        ids = torch.randint(0, text.config.vocab_size, (1, 77), device=dev)
        loss_buf = torch.zeros((), device=dev)

        def body():
            loss_buf.copy_(stepper.step(lat, ids))

        def timed(fn):
            for _ in range(warmup):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / steps

        ms_eager = timed(body)
        res = {"eager_ms_per_step": ms_eager, "eager_images_per_s": 1e3 / ms_eager, "loss": float(loss_buf)}
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                body()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                body()
            ms_graph = timed(gr.replay)
            res.update({"graphed_ms_per_step": ms_graph, "graphed_images_per_s": 1e3 / ms_graph})
            del gr
        except Exception as e:
            res["graph_error"] = f"{type(e).__name__}: {e}"
            torch.cuda.synchronize()
        out[mode] = res
        del stepper, unet, text, us, ts
        torch.cuda.empty_cache()
    best = out["bf16_model"]
    out["value"] = best["eager_images_per_s"]
    out["graphed_value"] = best.get("graphed_images_per_s")
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU path (oracle port; the reference package itself
    cannot be imported: diffusers/accelerate/fire are absent) on the host cores, EXACTLY --steps
    steps after --warmup warm-ups, rank 0 only. Imports nothing that maps liblora_b200.so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    world = int(os.environ.get("WORLD_SIZE", "1"))
    warm = max(args.warmup, 1)
    cb = cpu_reference(args.res, args.rank, budget_s=None, max_steps=args.steps, warmup=warm, tiny=args.tiny)
    try:
        from lora_b200 import _C
        so_mapped = _C.is_loaded()
    except Exception:
        so_mapped = None
    return {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT,
        "n_gpus": world, "steps": cb["steps"], "warmup": warm,
        "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic latents/token ids, random-init SD1.5-shaped weights",
        "config": bench_config(args, world),
        "engine": {"note": "reference = pure-Python lora_diffusion on torch eager; it cannot be imported on this box "
                           "(diffusers/accelerate/fire absent), so its step is the oracle port on the host cores",
                   "native_library_mapped": so_mapped, "loss": cb["loss"]},
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def run_reference_cuda(args):
    """--impl reference-cuda: the reference's path on the same GPU (see cuda_reference)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    if not torch.cuda.is_available():
        return {"impl": "reference-cuda", "unavailable": "no CUDA device"}
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    torch.backends.cudnn.benchmark = True
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    cb = cuda_reference(dev, args, steps=args.steps, warmup=max(args.warmup, 3))
    clocks = sampler.stop()
    return {
        "impl": "reference-cuda", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": 1,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": 1e3 / cb["value"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic latents/token ids, random-init SD1.5-shaped weights",
        "config": bench_config(args, world), "cuda_eager_baseline": cb, "clocks": clocks, "gpu_launches": 0,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference", "reference-cuda"])
    ap.add_argument("--res", type=int, default=512)
    ap.add_argument("--rank", type=int, default=4)
    ap.add_argument("--tiny", action="store_true", help="toy widths (smoke only, not a bench)")
    ap.add_argument("--extended", action="store_true", help="configs[2]: extended (conv) LoRA sites")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-group", action="store_true", help="one launch per LoRA site (no grouped launches)")
    ap.add_argument("--capture-collective", action="store_true",
                    help="EXPERIMENTAL: all-reduce inside ONE step graph (thread-local capture mode); run under timeout")
    ap.add_argument("--nccl-allreduce", action="store_true",
                    help="N > 1: NCCL all-reduce between two graphs instead of the all-reduce fused into the optimizer launch")
    ap.add_argument("--profile-steps", type=int, default=0, help="run N eager steps and exit (for ncu)")
    ap.add_argument("--roofline-only", action="store_true", help="one eager sweep of the fused kernel (for ncu)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cuda-baseline", action="store_true", help="skip the reference-on-this-GPU block")
    ap.add_argument("--cpu-budget", type=float, default=25.0, help="seconds of CPU-baseline work")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's loss and LoRA factors as DIR/<name>.npy")
    args = ap.parse_args()
    out = (run_reference(args) if args.impl == "reference" else
           run_reference_cuda(args) if args.impl == "reference-cuda" else run_native(args))
    if out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
