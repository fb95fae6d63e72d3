#!/usr/bin/env python
"""Decoding with a texture code MAP [N, C, h, w] against decoding with a texture code vector [N, C], inference (no_grad), CUDA-event
timed after warm-up, median of the timed runs: the vector code, the native map path (modulation affine at the map's resolution +
sae_modulate_spatial) and the glue map path (SAE_SPATIAL_STYLE=glue: map interpolated to every layer's resolution, 1x1 conv there).
Peak memory is torch.cuda.max_memory_allocated above what was allocated before the decode.  Configurations: 256^2 default nets at
batch 8 and the ffhq1024 option set at 1024^2 with the largest batch the glue path fits in.  Then the HBM rate of
sae_modulate_spatial forward / backward at the 256^2 layer shape, from ALGORITHMIC bytes (forward: read x + write out = 8 B per
element; backward: read dy, x + write dx = 12 B per element), L2 flushed between runs, against the 6481 GB/s copy peak."""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from swapping_autoencoder_pytorch_b200 import backend, default_options, networks  # noqa: E402

DEV = "cuda"
COPY_PEAK_GBS = 6481.0
FFHQ1024 = dict(crop_size=1024, netG_scale_capacity=0.8, netE_num_downsampling_sp=5, netE_scale_capacity=0.4, global_code_ch=1536,
                patch_size=256)


def timed(fn, warmup=2, iters=5, flush=None):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def peak_bytes(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def generator(over):
    opt = default_options(**dict(num_gpus=1, **over))
    torch.manual_seed(0)
    return opt, networks.create_network(opt, opt.netG, "generator").to(DEV).eval()


def decodes(opt, g, batch, map_hw):
    gen = torch.Generator(device=DEV).manual_seed(1)
    sp_hw = opt.crop_size // 2 ** opt.netE_num_downsampling_sp
    sp = torch.randn(batch, opt.spatial_code_ch, sp_hw, sp_hw, device=DEV, generator=gen)
    code = torch.randn(batch, opt.global_code_ch, device=DEV, generator=gen)
    code_map = torch.randn(batch, opt.global_code_ch, map_hw, map_hw, device=DEV, generator=gen)
    return sp, code, code_map


def run_glue(fn):
    k = backend.kernels()
    prev, k.spatial_style = k.spatial_style, "glue"
    try:
        return fn()
    finally:
        k.spatial_style = prev


def bench_config(label, over, batches, map_hw=16):
    opt, g = generator(over)
    batch = None
    with torch.no_grad():
        for b in batches:                       # largest batch the glue path fits in
            sp, code, code_map = decodes(opt, g, b, map_hw)
            try:
                run_glue(lambda: g(sp, code_map))
                batch = b
                break
            except torch.cuda.OutOfMemoryError:
                del sp, code, code_map
                torch.cuda.empty_cache()
        if batch is None:
            print("%s: the glue path does not fit at batch %s" % (label, batches[-1]))
            return
        rows = {}
        for tag, fn in (("vector code", lambda: g(sp, code)), ("native map", lambda: g(sp, code_map)),
                        ("glue map", lambda: run_glue(lambda: g(sp, code_map)))):
            torch.cuda.empty_cache()
            rows[tag] = (timed(fn), peak_bytes(fn))
    print("%s, batch %d, %dx%d code map" % (label, batch, map_hw, map_hw))
    print("  %-12s %10s %10s %12s %10s" % ("decode", "ms", "x vector", "peak MB", "x vector"))
    v_ms, v_mem = rows["vector code"]
    for tag, (ms, mem) in rows.items():
        print("  %-12s %10.3f %10.2f %12.1f %10.2f" % (tag, ms, ms / v_ms, mem / 1e6, mem / v_mem), flush=True)


def bench_kernel():
    k = backend.kernels()
    flush = torch.empty(256 * 1024 * 1024 // 4, device=DEV)
    print("sae_modulate_spatial at the 256^2 layer shape (algorithmic bytes, L2 flushed)")
    print("  %-44s %9s %9s %8s" % ("shape", "ms", "GB/s", "of copy"))
    for n, c, demod in ((8, 128, True), (8, 128, False), (8, 256, True)):
        gen = torch.Generator(device=DEV).manual_seed(2)
        x = torch.randn(n, 256, 256, c, device=DEV, generator=gen)
        dy = torch.randn_like(x)
        s = torch.randn(n, 16, 16, c, device=DEV, generator=gen)
        elems = x.numel()
        for name, fn, nbytes in (("fwd", lambda: k.modulate_spatial(x, s, demod), 8 * elems),
                                 ("bwd", lambda: k.modulate_spatial_backward(dy, x, s, demod), 12 * elems)):
            ms = timed(fn, iters=10, flush=flush)
            gbs = nbytes / ms / 1e6
            print("  %-44s %9.3f %9.0f %7.0f%%" % ("%s N=%d 256x256 C=%d demod=%d (16x16 map)" % (name, n, c, demod), ms, gbs,
                                                    100 * gbs / COPY_PEAK_GBS), flush=True)


def main():
    assert torch.cuda.is_available(), "spatial_code_bench.py measures on the GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    print("device: %s | nvidia-smi: %s" % (torch.cuda.get_device_name(), smi))
    bench_config("256x256 default nets", {}, [8])
    bench_config("1024x1024 ffhq1024 option set", FFHQ1024, [8, 4, 2, 1])
    bench_kernel()


if __name__ == "__main__":
    main()
