#!/usr/bin/env python
"""Benchmark of the Swapping-Autoencoder training hot path on B200 (DESIGN.md §7).

  python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU (native-PyTorch) path = oracle port
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/*.npy

A "step" is one ``train_one_step`` call — a discriminator OR a generator half-step over one batch, exactly the unit
the reference's own iteration counter advances by (reference util/iter_counter.py:54, SURVEY.md §8(d)); lazy R1
runs inside every 16th discriminator step.  Metric: training images / second at 256x256 with the reference's
default networks (BASELINE.json), per-GPU batch 32 (weak scaling).  One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

RES = 256
PER_GPU_BATCH = 32
CPU_SAMPLE_BATCH = 2


# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1425.5), d.get("hbm_gbs", 6480.8), "measured"
    return 1400.0, 6650.0, "fallback"


# ----------------------------------------------------------------------------------------------------------------
def cpu_step_rate(steps, warmup, batch=CPU_SAMPLE_BATCH, threads=None):
    """Reference CPU path (oracle port of the native-PyTorch fallback): D/G half-steps at 256x256, default nets."""
    from oracle import sae_oracle as O
    from swapping_autoencoder_pytorch_b200 import default_options
    # all host cores up to 32: beyond that the reference's many small ATen ops only lose time to oversubscription
    threads = threads or min(os.cpu_count() or 1, 32)
    torch.set_num_threads(threads)
    opt = default_options(num_gpus=0, batch_size=batch, crop_size=RES)
    model = O.OracleModel(opt, O.init_state_dict(opt, seed=0))
    trainer = O.OracleTrainer(model)
    real = torch.randn(batch, 3, RES, RES, generator=torch.Generator().manual_seed(0)).clamp(-1, 1)
    for _ in range(warmup):
        trainer.train_one_step(real)
    t0 = time.perf_counter()
    for _ in range(steps):
        trainer.train_one_step(real)
    dt = time.perf_counter() - t0
    return steps * batch / dt, dt / max(steps, 1), threads


def cpu_config1_ms(threads=None, iters=3):
    """BASELINE configs[0]: single 64x64 random image, E -> G forward + L1 reconstruction loss on the reference's CPU path
    (``netE_num_downsampling_sp=3``: the default 4 cannot run at 64x64, SURVEY.md §0.5 / reference encoder.py:106)."""
    from oracle import sae_oracle as O
    from swapping_autoencoder_pytorch_b200 import default_options
    torch.set_num_threads(threads or min(os.cpu_count() or 1, 32))
    opt = default_options(num_gpus=0, batch_size=1, crop_size=64, netE_num_downsampling_sp=3)
    model = O.OracleModel(opt, O.init_state_dict(opt, seed=0))
    x = torch.randn(1, 3, 64, 64, generator=torch.Generator().manual_seed(0)).clamp(-1, 1)
    best = None
    with torch.no_grad():
        for _ in range(iters + 1):
            t0 = time.perf_counter()
            loss = (model.autoencode(x) - x).abs().mean()
            dt = (time.perf_counter() - t0) * 1e3
            best = dt if best is None else min(best, dt)
    assert float(loss) == float(loss)
    return best


def gpu_context_rate(device, batch, steps=4, warmup=2):
    """CONTEXT ONLY (BASELINE.md §3 "kernel to beat"): the reference's own operator formulation — plain torch ops, cuDNN /
    cuBLAS convolutions with ``allow_tf32`` on (the reference's default), ``upfirdn2d_native``-style FIR — run on the same
    B200 through the oracle port (the Python reference and its JIT-built extensions cannot travel to the GPU box).
    Nothing of this library is on that path and nothing of it is on the product path."""
    from oracle import sae_oracle as O
    from swapping_autoencoder_pytorch_b200 import default_options
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.benchmark = True
    opt = default_options(num_gpus=0, batch_size=batch, crop_size=RES)
    sd = {k: v.to(device) for k, v in O.init_state_dict(opt, seed=0).items()}
    trainer = O.OracleTrainer(O.OracleModel(opt, sd))
    real = torch.randn(batch, 3, RES, RES, generator=torch.Generator().manual_seed(0)).clamp(-1, 1).to(device)
    for _ in range(warmup):
        trainer.train_one_step(real)
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        trainer.train_one_step(real)
    e1.record()
    torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1) / steps
    del trainer, sd
    torch.cuda.empty_cache()
    return batch / (ms * 1e-3), ms


def run_reference(args, rank):
    if rank != 0:
        return
    value, sec_per_step, threads = cpu_step_rate(args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": "training images/sec", "value": value, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "256x256 default E/G/D/Dpatch D/G half-steps (CPU sample)", "resolution": RES,
                   "sample_batch": CPU_SAMPLE_BATCH},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "port",
                         "sample": "%d half-steps (D,G alternating) of batch %d at %dx%d, default nets, fp32, oracle port of the "
                                   "reference's native-PyTorch path" % (args.steps, CPU_SAMPLE_BATCH, RES, RES),
                         "config1_64x64_autoencode_l1_ms": cpu_config1_ms(threads)},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
def _numel(out):
    if torch.is_tensor(out):
        return out.numel()
    if isinstance(out, (tuple, list)):
        return sum(_numel(o) for o in out if o is not None)
    return 0


def kernel_rooflines(trainer, images, device):
    """One eager D + one G half-step with every launch of (a) the implicit-GEMM conv family and (b) the bandwidth-bound
    kernels (FIR, bias/activation, modulate, resampling merges) bracketed by CUDA events on the launching stream.
    Returns (per-impl conv totals, bandwidth totals [bytes, seconds, launches], per-shape conv table rows)."""
    from swapping_autoencoder_pytorch_b200 import backend
    k = backend.kernels()
    conv_rec, mem_rec = [], []
    conv_names = ("conv_fprop", "conv_dgrad", "conv_wgrad")
    mem_names = ("upfirdn2d", "fir_act_backward", "bias_act", "bias_act_backward", "modulate", "modulate_backward",
                 "add_scale", "upsample2x_add_scale", "upsample2x_backward", "pad_channels", "reflect_pad",
                 "reflect_pad_backward", "fir_bias_act", "fir_bias_act_backward", "crop_gather", "crop_gather_backward")
    mem_names = tuple(n for n in mem_names if hasattr(k, n))
    orig = {n: getattr(k, n) for n in conv_names + mem_names}

    def wrap_conv(name, direction):
        fn = orig[name]

        def timed(a, b, g, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(a, b, g, **kw)
            e1.record()
            flops = 2.0 * g.N * g.P * g.Q * g.K * g.R * g.S * g.C
            nbytes = 4.0 * (g.N * g.H * g.W * g.C + g.N * g.P * g.Q * g.K + g.K * g.R * g.S * g.C)
            conv_rec.append((e0, e1, flops, nbytes, k.conv_impl_for(g, direction), g.key(), name))
            return out
        return timed

    def wrap_mem(name):
        fn = orig[name]

        def timed(*a, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*a, **kw)
            e1.record()
            if out is not None:
                # algorithmic bytes: every full-size tensor argument read once, every result written once
                big = [t for t in list(a) + list(kw.values()) if torch.is_tensor(t) and t.numel() >= 4096]
                mem_rec.append((e0, e1, 4.0 * (sum(t.numel() for t in big) + _numel(out)), name))
            return out
        return timed
    try:
        for i, n in enumerate(conv_names):
            setattr(k, n, wrap_conv(n, i))
        for n in mem_names:
            setattr(k, n, wrap_mem(n))
        trainer.train_one_step({"real_A": images}, 0)
        trainer.train_one_step({"real_A": images}, 0)
        torch.cuda.synchronize(device)
    finally:
        for n, fn in orig.items():
            setattr(k, n, fn)
    tot = {1: [0.0, 0.0, 0], 2: [0.0, 0.0, 0]}
    per_shape = {}
    for e0, e1, flops, nbytes, impl, key, name in conv_rec:
        t = tot.setdefault(impl, [0.0, 0.0, 0])
        sec = e0.elapsed_time(e1) * 1e-3
        t[0] += flops
        t[1] += sec
        t[2] += 1
        ps = per_shape.setdefault((name, impl) + key, [0.0, 0.0, 0, 0.0])
        ps[0] += flops
        ps[1] += sec
        ps[2] += 1
        ps[3] += nbytes
    mem = {}
    for e0, e1, nbytes, name in mem_rec:
        m = mem.setdefault(name, [0.0, 0.0, 0])
        m[0] += nbytes
        m[1] += e0.elapsed_time(e1) * 1e-3
        m[2] += 1
    dump = os.environ.get("SAE_BENCH_CONV_TABLE")
    if dump:
        with open(dump, "w") as f:
            f.write("dir impl N H W C K R S P Q stride pad_t pad_l | calls ms TFLOP/s GB/s\n")
            for kk, v in sorted(per_shape.items(), key=lambda kv: -kv[1][1]):
                f.write("%s %s | %d %.3f %.1f %.0f\n" % (kk[0], " ".join(str(x) for x in kk[1:]), v[2], v[1] * 1e3,
                                                        v[0] / max(v[1], 1e-12) / 1e12, v[3] / max(v[1], 1e-12) / 1e9))
            f.write("\nbandwidth-bound kernels: name | calls ms GB/s\n")
            for n, v in sorted(mem.items(), key=lambda kv: -kv[1][1]):
                f.write("%s | %d %.3f %.0f\n" % (n, v[2], v[1] * 1e3, v[0] / max(v[1], 1e-12) / 1e9))
    return tot, mem, per_shape


def r1_position(d_steps, every):
    """(c0, n): value of the discriminator iteration counter before a loop of ``d_steps`` discriminator half-steps such that
    the loop contains n = max(1, round(d_steps / every)) lazy-R1 evaluations (never fewer than the cadence asks for, so the
    rate is not flattered), the first of them in the middle of the loop / of the first cadence window."""
    if d_steps <= 0:
        return 0, 0
    target = max(1, int(round(d_steps / every)))
    best = None
    for c0 in range(every):
        if (c0 + d_steps) // every - c0 // every != target:
            continue
        first = every - c0
        score = abs(first - (min(d_steps, every) + 1) / 2.0)
        if best is None or score < best[0]:
            best = (score, c0)
    return (best[1] if best else 0), target


DUMP_SAMPLE = 4096


def dump_outputs(out_dir, losses, named_params):
    """Writes what the last timed half-step hands its caller — its losses (``loss.<name>.npy``, float64) and the parameters
    it leaves behind (``param.<name>.npy``, float32; tensors above DUMP_SAMPLE elements at DUMP_SAMPLE indices drawn from a
    fixed seed: 1.6 MB in all for the default nets) — so that two builds can be compared output for output on identical inputs.
    The inputs are seeded and the kernels reduce in a fixed order, so repeated runs of one build write the same values."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for k, v in losses.items():
        np.save(os.path.join(out_dir, "loss.%s.npy" % k), np.asarray(float(v), dtype=np.float64))
    for name, p in named_params:
        flat = p.detach().float().reshape(-1).cpu().numpy()
        if flat.size > DUMP_SAMPLE:
            flat = flat[np.sort(np.random.RandomState(0).choice(flat.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(out_dir, "param.%s.npy" % name), flat)


def run_ours(args, rank, world, local):
    import swapping_autoencoder_pytorch_b200 as S
    from swapping_autoencoder_pytorch_b200 import _lib, backend
    import torch.distributed as dist

    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    backend.kernels()          # loads libsae_b200.so; raises if it is missing (no fallback)
    PER_GPU_BATCH = args.per_gpu_batch
    # each half-step runs as a CUDA graph replay (graphs.py) unless SAE_CUDA_GRAPHS=0
    use_graphs = os.environ.get("SAE_CUDA_GRAPHS", "1") != "0"
    opt = S.default_options(num_gpus=1, batch_size=PER_GPU_BATCH * world, crop_size=RES, cuda_graphs=use_graphs,
                            batch_discriminator_passes=os.environ.get("SAE_BATCH_D", "1") == "1")
    torch.manual_seed(0)
    model = S.create_model(opt)
    trainer = S.create_optimizer(opt, model)
    every = opt.R1_once_every

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def timed_loop(fetch, sample_clocks):
        """EXACTLY args.steps half-steps starting with a discriminator step; the lazy-R1 counter is positioned so that the
        loop holds max(1, round(D-steps / 16)) R1 evaluations whatever --steps and the warm-up were."""
        d_steps = (args.steps + 1) // 2
        c0, _ = r1_position(d_steps, every)
        trainer.train_mode_counter = 0
        trainer.discriminator_iter_counter = c0
        barrier()
        sampler = ClockSampler(local) if (rank == 0 and sample_clocks) else None
        if sampler:
            sampler.start()
        n0 = _lib.launch_count() + (trainer.graphs.replayed_launches if trainer.graphs else 0)
        if trainer.graphs is not None:
            trainer.graphs.phase_events = []
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        kinds = []
        ev[0].record()
        for i in range(args.steps):
            out = trainer.train_one_step({"real_A": fetch()}, 0)     # losses are read back (D2H) inside
            kinds.append("D+R1" if "D_R1" in out else ("D" if "D_total" in out else "G"))
            ev[i + 1].record()
        barrier()
        ms = ev[0].elapsed_time(ev[-1])
        per_kind = {}
        for i, kd in enumerate(kinds):
            per_kind.setdefault(kd, []).append(ev[i].elapsed_time(ev[i + 1]))
        launches = _lib.launch_count() + (trainer.graphs.replayed_launches if trainer.graphs else 0) - n0
        clocks = sampler.stop() if sampler else None
        # per-phase device time of the replayed half-steps on this rank: graph replay (forward + backward [+ Adam at N = 1]),
        # then bucket pack + all-reduce + Adam (N > 1); "gap" = what is left of the step (input copy, host gaps, waiting for peers)
        phases = None
        if trainer.graphs is not None and trainer.graphs.phase_events:
            pe, trainer.graphs.phase_events = trainer.graphs.phase_events, None
            rep = sum(e[0].elapsed_time(e[1]) for _, e in pe) / len(pe)
            tail = sum(e[1].elapsed_time(e[2]) for _, e in pe) / len(pe)
            phases = {"graph_replay_ms": rep, "exchange_and_adam_ms": tail, "gap_ms": ms / args.steps - (rep + tail) * len(pe) / args.steps,
                      "replays": len(pe)}
        if world > 1:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return {"ms": ms, "launches": launches, "clocks": clocks, "r1": kinds.count("D+R1"), "phases": phases,
                "per_kind_ms": {kd: sum(v) / len(v) for kd, v in per_kind.items()}, "last_losses": out}

    def warm(resident):
        # at least 4 untimed half-steps: D, G, D, G — both step kinds twice, so the caching allocator and every kernel
        # variant have reached steady state before the timed region
        n_warm = max(args.warmup, int(os.environ.get("SAE_BENCH_MIN_WARM", "4")))   # (profiling runs under ncu lower it)
        for _ in range(n_warm):
            trainer.train_one_step({"real_A": resident}, 0)
        if trainer.graphs is not None and trainer.graphs.enabled:
            trainer.graphs.warm_up(resident)          # capture the D, G and R1 graphs before the timed region
        if (trainer.graphs is None or trainer.graphs.disabled) and os.environ.get("SAE_BENCH_SKIP_R1_WARM") != "1":
            # eager execution: the lazy-R1 evaluation must not meet the caching allocator's cold start inside the timed region
            trainer.discriminator_iter_counter = every - 1
            trainer.train_mode_counter = 0
            trainer.train_one_step({"real_A": resident}, 0)      # D + R1
            trainer.train_one_step({"real_A": resident}, 0)      # G
            torch.cuda.synchronize(device)
        return n_warm

    def measure(per_gpu_batch, sample_clocks):
        gen = torch.Generator().manual_seed(1234 + rank)
        host = torch.randn(per_gpu_batch, 3, RES, RES, generator=gen).clamp(-1, 1).pin_memory()
        resident = host.to(device)
        n_warm = warm(resident)
        dev = timed_loop(lambda: resident, sample_clocks)
        e2e = timed_loop(lambda: host.to(device, non_blocking=True), False)
        return host, resident, n_warm, dev, e2e

    host, resident, n_warm, dev, e2e = measure(PER_GPU_BATCH, True)
    images = args.steps * PER_GPU_BATCH * world
    if args.dump_outputs and rank == 0:
        # the e2e loop ran last: its final half-step is the last timed step
        dump_outputs(args.dump_outputs, e2e["last_losses"], model.singlegpu_model.named_parameters())

    strong = None
    if world > 1 and 32 % world == 0 and (32 // world) % 2 == 0 and not args.no_strong:
        # strong scaling (SURVEY.md §9.1): the metric's global batch of 32 split over the ranks
        pb = 32 // world
        _, _, _, sdev, se2e = measure(pb, False)
        strong = {"scaling": "strong", "global_batch": 32, "per_gpu_batch": pb,
                  "value": args.steps * 32 / (sdev["ms"] * 1e-3), "ms_per_step": sdev["ms"] / args.steps,
                  "e2e_value": args.steps * 32 / (se2e["ms"] * 1e-3), "r1_evaluations": sdev["r1"], "unit": "images/s"}

    # the per-launch instrumentation pass needs eager launches.  It runs on the stream the half-steps were warmed up and
    # captured on: autograd binds a parameter's gradient-accumulation node to the stream it was created on, and running
    # the eager pass elsewhere would make every backward hop streams (torch warns about exactly that)
    side = trainer.graphs.stream if (trainer.graphs is not None and trainer.graphs.stream is not None) else torch.cuda.current_stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        if trainer.graphs is not None:
            trainer.graphs.enabled = False
            for _ in range(2):                    # a warm caching allocator under the eager launches
                trainer.train_one_step({"real_A": resident}, 0)
            torch.cuda.synchronize(device)
        trainer.train_mode_counter = 0
        trainer.discriminator_iter_counter = 0
        roof, mem, per_shape = kernel_rooflines(trainer, resident, device)
    torch.cuda.current_stream().wait_stream(side)
    graph_state = "off"
    if trainer.graphs is not None:
        g = trainer.graphs
        graph_state = ("off (capture failed: %s)" % g.disabled) if g.disabled else \
            "on (%s captured; %s)" % ("/".join(sorted(set(k[0] for k in g.captured))), g.describe(world))
    peak_tf, peak_bw, peak_src = measured_peaks()
    dom = 2 if roof.get(2, [0, 0, 0])[2] > 0 else 1
    fl, sec, cnt = roof[dom]
    achieved = fl / sec / 1e12 if sec > 0 else 0.0
    traffic, traffic_note = None, None
    for name in ("r2_traffic.json", "r1_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
            traffic_note = "%s: dram read+write per launch from %s; algorithmic bytes %d" % (tj["kernel"], tj["source"],
                                                                                             tj["algorithmic_bytes"])
            break
    tf32_nominal = 1125.0      # dense kind::tf32 rate = half the nominal 2250 TFLOP/s bf16 rate (B200_PROFILING.md)
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": achieved / peak_tf if peak_tf else None, "traffic": traffic, "traffic_note": traffic_note,
                "peak_tf32_nominal": tf32_nominal, "frac_of_tf32_nominal": achieved / tf32_nominal,
                "kernel": "conv implicit GEMM (%s)" % ("tcgen05+TMA TF32" if dom == 2 else "mma.sync TF32 generic"),
                "launches_timed": cnt, "peak_source": peak_src + " bf16 dense sustained; kind::tf32 peaks at half of it",
                "by_impl": {("tcgen05" if i == 2 else "generic"): {"tflops": (v[0] / v[1] / 1e12 if v[1] > 0 else 0.0),
                                                                  "share_of_flops": v[0] / max(sum(x[0] for x in roof.values()), 1.0),
                                                                  "launches": v[2]} for i, v in roof.items()}}
    # second entry: everything whose roofline is HBM — the pointwise / FIR / resampling kernels and the conv launches whose
    # arithmetic intensity is below the machine balance (1x1 convs, 32/64-channel layers, 3-channel outputs)
    balance = tf32_nominal * 1e12 / (peak_bw * 1e9)
    mb, ms_, mc = 0.0, 0.0, 0
    for v in mem.values():
        mb, ms_, mc = mb + v[0], ms_ + v[1], mc + v[2]
    cb, cs, cc = 0.0, 0.0, 0
    for v in per_shape.values():
        if v[0] / max(v[3], 1.0) < balance:
            cb, cs, cc = cb + v[3], cs + v[1], cc + v[2]
    roofline_hbm = {"bound": "hbm", "unit": "GB/s", "peak": peak_bw,
                    "achieved": (mb + cb) / max(ms_ + cs, 1e-12) / 1e9, "frac": (mb + cb) / max(ms_ + cs, 1e-12) / 1e9 / peak_bw,
                    "pointwise_fir": {"achieved": mb / max(ms_, 1e-12) / 1e9, "launches": mc, "ms": ms_ * 1e3,
                                      "by_kernel": {n: round(v[0] / max(v[1], 1e-12) / 1e9) for n, v in mem.items()}},
                    "low_intensity_convs": {"achieved": cb / max(cs, 1e-12) / 1e9, "launches": cc, "ms": cs * 1e3,
                                            "rule": "FLOP / algorithmic byte < %.0f" % balance},
                    "note": "algorithmic bytes (each operand read once, each result written once) / CUDA-event time, "
                            "eager instrumented D + G half-step"}

    if trainer.graphs is not None:
        trainer.graphs.release()          # no captured kernels (possibly NCCL ones) outlive the measurements
    if rank != 0:
        return
    # bounded CPU sample (one D + one G half-step on 2 images, plus BASELINE configs[0]); N = 1 only
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        v, _, threads = cpu_step_rate(2, 0)
        cpu = {"value": v, "unit": "images/s", "cores": threads, "kind": "port",
               "sample": "1 D + 1 G half-step, batch %d at %dx%d, default nets, fp32 oracle port of the reference's "
                         "native-PyTorch CPU path" % (CPU_SAMPLE_BATCH, RES, RES),
               "config1_64x64_autoencode_l1_ms": cpu_config1_ms(threads)}
    ctx = None
    if world == 1 and not args.no_gpu_context:
        del trainer, model
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        for b in (PER_GPU_BATCH, PER_GPU_BATCH // 2, PER_GPU_BATCH // 4):
            try:
                v, ms_step = gpu_context_rate(device, b)
                ctx = {"value": v, "unit": "images/s", "ms_per_step": ms_step, "batch": b,
                       "what": "CONTEXT, not the product: the reference's operator formulation (oracle port) as plain torch ops "
                               "on this B200 — cuDNN/cuBLAS convolutions with allow_tf32=True, native-PyTorch upfirdn2d / "
                               "bias-act, eager, stock Adam; 4 half-steps after 2 warm-up"}
                break
            except torch.cuda.OutOfMemoryError:
                torch.cuda.empty_cache()
            except Exception as e:      # noqa: BLE001 — context only, never fails the bench
                ctx = {"error": "%s: %s" % (type(e).__name__, str(e)[:200])}
                break
    pk = dev["per_kind_ms"]
    cadence = None
    if "D" in pk and "G" in pk and "D+R1" in pk:
        period = every * pk["D"] + every * pk["G"] + (pk["D+R1"] - pk["D"])
        cadence = {"images_per_s_at_1_in_%d" % every: 2 * every * PER_GPU_BATCH * world / (period * 1e-3),
                   "ms": {"D": pk["D"], "G": pk["G"], "R1_extra": pk["D+R1"] - pk["D"]},
                   "note": "rank-0 per-kind half-step times from the device-timed loop, weighted 16 D : 16 G : 1 R1"}
    loss_bytes = 8 * 4
    line = {
        "metric": "training images/sec", "value": images / (dev["ms"] * 1e-3), "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": n_warm, "ms_per_step": dev["ms"] / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "tf32", "data": "synthetic",
        "config": {"workload": "256x256 default E/G/D/Dpatch, alternating D/G half-steps with lazy R1 (BASELINE configs[1] "
                               "shape at the metric's bs=32)", "resolution": RES, "per_gpu_batch": PER_GPU_BATCH,
                   "global_batch": PER_GPU_BATCH * world, "parallelism": "dp%d" % world,
                   "r1_evaluations_in_timed_region": dev["r1"], "r1_evaluations_in_e2e_region": e2e["r1"],
                   "r1_once_every": every,
                   "r1_policy": "counter positioned so every timed loop holds max(1, round(D-steps/16)) evaluations",
                   "cuda_graphs": graph_state,
                   "l2": "activations per step exceed the 126 MB L2 by >100x; no explicit flush"},
        "clocks": dev["clocks"],
        "e2e": {"value": images / (e2e["ms"] * 1e-3), "unit": "images/s",
                "h2d_bytes_per_step": host.numel() * 4, "d2h_bytes_per_step": loss_bytes},
        "gpu_launches": int(dev["launches"]),
        "phases_rank0": dev["phases"],
        "roofline": roofline,
        "roofline_hbm": roofline_hbm,
    }
    if cadence is not None:
        line["cadence"] = cadence
    if strong is not None:
        line["strong"] = strong
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if ctx is not None:
        line["reference_gpu_context"] = ctx
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # default 32 half-steps = 16 discriminator steps = exactly one lazy-R1 evaluation at the reference's cadence; for any other
    # --steps the loop still holds max(1, round(D-steps / 16)) evaluations (r1_position)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-context", action="store_true", help="skip the torch/cuDNN context leg (N = 1 only)")
    ap.add_argument("--no-strong", action="store_true", help="N > 1: skip the strong-scaling sub-result (global batch 32)")
    ap.add_argument("--per-gpu-batch", type=int, default=PER_GPU_BATCH,
                    help="experiments only (host-overhead probes); the reported metric is defined at the default 32")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's losses and a seeded sample of the updated "
                         "parameters to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of this library's timed path; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    from swapping_autoencoder_pytorch_b200.parallel import init_distributed
    rank, world, local = init_distributed("nccl")
    try:
        run_ours(args, rank, world, local)
    finally:
        import gc
        import torch.distributed as dist
        gc.collect()
        torch.cuda.synchronize()
        if dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
