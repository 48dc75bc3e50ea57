#!/usr/bin/env python
"""bench.py -- closed-loop encode + decode throughput of the B200-native block codec.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--config B8_lowrate] [--images PER_GPU] [--height 512] [--width 768] [--lanes 0|1]
                    [--dump-outputs DIR]

One "step" = compress + decompress of one batch of synthetic HxW RGB images (default 768x512, the
Kodak size BASELINE.json quotes) with random-init weights of the named architecture.  Metric: Mpixel/s
of the encode+decode round trip (a pixel counts once per round trip), whole job over all N GPUs
(image-sharded, weak scaling, no data-path collective).  Prints ONE JSON line on rank 0.

--dump-outputs DIR writes what the last timed step returned (see dump_outputs) as DIR/<name>.npy on rank 0.  Inputs
and weights are seeded, so two builds run with the same arguments can be compared output for output.

--impl reference times the reference's CPU implementation of the same path (the oracle port of
graphs/models/BlockBasedImgCompLossy_net.py:319-452; the Python reference itself cannot travel to
the GPU box) on a bounded sample of the same workload, using all host threads.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# SURVEY.md section 8(d) / Appendix C: live MACs per block (masked taps excluded)
def macs_per_block(cfg):
    B, N, M = int(cfg.block_size), int(cfg.N), int(cfg.M)
    cin, C2, C3 = 3 * B * B, N // 8 * 7, N // 8 * 6
    E1, E2, E3 = N // 8 * 12, N // 8 * 10, N // 8 * 8
    t1 = 5 if int(cfg.KS[1]) == 3 else 1
    enc = cin * N + 4 * cin * N + N * N + N * C2 + C2 * C2 + C2 * C3 + C3 * C3 + C3 * M
    dec = M * N + 4 * cin * N + N * N + N * C2 + C2 * C2 + C2 * C3 + C3 * C3 + C3 * cin
    ent = 4 * cin * E1 + t1 * E1 * E2 + E2 * E3 + E3 * 2 * M
    return dict(encode=enc + dec + ent, decode=dec + ent)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tf_sustained=d.get("bf16_tflops_sustained", 1381.8), tf_burst=d.get("bf16_tflops", 1670.2),
                    hbm=d.get("hbm_gbs", 6555.8), source="measured")
    return dict(tf_sustained=1400.0, tf_burst=1590.0, hbm=6650.0, source="fallback")


def measured_traffic(args):
    """roofline.traffic comes from an ncu --set full capture of THIS command (scripts/ncu_traffic.py parses the report
    into profiles/ncu_traffic.json keyed by workload); it is null when no capture of the workload being run exists."""
    key = f"{args.config}:{args.images}:{args.width}x{args.height}:lanes{args.lanes}"
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        rec = json.load(open(p)).get(key)
    except Exception:
        rec = None
    if not rec:
        return dict(traffic=None, traffic_note=f"no ncu --set full capture for workload {key} under profiles/ncu_traffic.json")
    return dict(traffic=rec["dram_bytes_per_launch"], traffic_note=rec["note"])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [v for v in sm if mx and v > 0.3 * mx] or sm
        return dict(sm_mhz=statistics.median(busy) if busy else None, sm_max_mhz=mx, reasons=sorted(reasons),
                    samples=len(sm))


def synth_batch_gpu(n, H, W, seed, dev):
    """Smooth-plus-noise synthetic 8-bit RGB images (SURVEY.md 8(d)), generated on the device: (n,3,H,W) uint8."""
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    low = torch.rand(n, 3, max(H // 16, 2), max(W // 16, 2), generator=g, device=dev)
    up = torch.nn.functional.interpolate(low, size=(H, W), mode="bicubic", align_corners=False)
    img = (up + 0.05 * torch.randn(n, 3, H, W, generator=g, device=dev)).clamp_(0, 1)
    return img.mul_(255).round_().to(torch.uint8)


DUMP_ELEMENTS = 1 << 22      # per array (16 MB of float32): at most ~48 MB in all, plus 8 bytes per image for lens


def dump_outputs(dirname, zhat, lens, streams, zdec):
    """Writes what one encode + decode step hands its caller, as float32 / float64 arrays DIR/<name>.npy:
    zhat and zdec (encoder and decoder reconstruction, flattened), lens (bytes of each image's stream) and streams
    (n, k: the bytes of each stream at k fixed fractions of its length).  An array larger than DUMP_ELEMENTS is a fixed,
    seeded sample whose positions depend only on the shape, the same in every run and build."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    flat_zhat, flat_zdec = zhat.reshape(-1), zdec.reshape(-1)
    if flat_zhat.numel() > DUMP_ELEMENTS:
        pos = np.sort(np.random.default_rng(0).choice(flat_zhat.numel(), DUMP_ELEMENTS, replace=False))
        pos = torch.from_numpy(pos).to(zhat.device)
        flat_zhat, flat_zdec = flat_zhat[pos], flat_zdec[pos]
    k = max(1, min(2048, DUMP_ELEMENTS // lens.shape[0]))
    frac = np.sort(np.random.default_rng(1).random(k))
    at = (torch.from_numpy(frac).to(lens.device)[None, :] * lens.double()[:, None]).long()
    out = dict(zhat=flat_zhat.float(), zdec=flat_zdec.float(), lens=lens.double(),
               streams=torch.gather(streams, 1, at).float())
    for name, t in out.items():
        np.save(os.path.join(dirname, f"{name}.npy"), t.cpu().numpy())


def cpu_baseline(cfg, H, W, max_blocks, threads):
    """The oracle port of the reference's compress()/decompress() loops (torch CPU fp32 convs exactly as
    NET:363-398) timed on a bounded sample: the first `max_blocks` blocks in raster order of one image.
    threads = 1 is the reference's own CPU setting (AGENT:565-566 torch.set_num_threads(1))."""
    import torch
    import lbic_b200
    from lbic_b200 import weights
    from oracle import nets
    torch.set_num_threads(threads)
    torch.use_deterministic_algorithms(True)      # AGENT:562
    B = int(cfg.block_size)
    sd = weights.synth_state_dict(cfg, 1337)
    P = nets.effective_params(sd, cfg)
    tabs = nets.build_tables()
    img = weights.synth_images(1, H, W, seed0=1000)
    x = nets.arrange_block_pixels_to_channel_dim(img - 0.5, B)
    nets.compress_loop(P, x, max_blocks=4)                      # warm-up
    t0 = time.perf_counter()
    syms, idxs, zhat = nets.compress_loop(P, x, max_blocks=max_blocks)
    t_enc = time.perf_counter() - t0
    from oracle import native
    T = native.Tables(*[t.numpy() for t in tabs])
    nb = min(max_blocks, x.shape[2] * x.shape[3])
    flat_s = syms.reshape(-1, cfg.M)[:nb].reshape(-1).numpy()
    flat_i = idxs.reshape(-1, cfg.M)[:nb].reshape(-1).numpy()
    stream = native.rans_encode(flat_s, flat_i, T)
    t0 = time.perf_counter()
    nets.decompress_loop(P, tabs, stream, x.shape, max_blocks=max_blocks)
    t_dec = time.perf_counter() - t0
    px = nb * B * B
    return dict(enc_s=t_enc, dec_s=t_dec, pixels=px, blocks=nb,
                mpix_s=px / (t_enc + t_dec) / 1e6, enc_mpix_s=px / t_enc / 1e6, dec_mpix_s=px / t_dec / 1e6)


def run_reference(args, cfg, rank):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_baseline(cfg, args.height, args.width, args.ref_blocks, threads)
        if i >= args.warmup:
            vals.append(r)
    t = sum(v["enc_s"] + v["dec_s"] for v in vals)
    px = sum(v["pixels"] for v in vals)
    value = px / t / 1e6
    sample = (f"first {vals[0]['blocks']} raster-order blocks of one {args.width}x{args.height} image per step, "
              f"compress loop + decompress loop, torch CPU fp32, {threads} threads")
    line = dict(metric="encode+decode Mpixel/s", value=value, unit="Mpixel/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * t / len(vals), higher_is_better=True, scaling=args.scaling,
                vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                config=workload_config(args, cfg),
                cpu_baseline=dict(value=value, unit="Mpixel/s", cores=threads, kind="port", sample=sample),
                e2e=dict(value=value, unit="Mpixel/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def workload_config(args, cfg):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    split = (f"{args.images} images per GPU (weak scaling)" if args.scaling == "weak" else
             f"{args.total_images} images in total, image-sharded over {world} GPU(s) = {args.images} per GPU (strong scaling)")
    return dict(workload=f"{args.config} (B{cfg.block_size}, KS{''.join(map(str, cfg.KS))}, N{cfg.N} M{cfg.M}) "
                         f"compress+decompress of synthetic {args.width}x{args.height} RGB images, {split}, "
                         f"random-init conditioned weights",
                images_per_gpu=args.images, height=args.height, width=args.width,
                container="reference (1 rANS stream per image)" if args.lanes == 1 else "lane (1 rANS stream per block row)",
                l2="inputs larger than L2 (batch of input blocks > 126 MB)" if args.images * args.height * args.width * 12 > 126e6
                else "inputs smaller than L2; L2 flushed between steps",
                **({} if (args.latent_gain == 60.0 and args.scale_span == 5.2) else
                   {"synthetic_rate": f"latent_gain {args.latent_gain}, scale_span {args.scale_span} (see bpp)"}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="B8_lowrate")
    ap.add_argument("--images", type=int, default=1024, help="images per GPU per step (weak scaling)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="strong: --total-images are image-sharded over the N GPUs (BASELINE config 3)")
    ap.add_argument("--total-images", type=int, default=1024, help="batch of the whole job under --scaling strong")
    ap.add_argument("--height", type=int, default=512)
    ap.add_argument("--width", type=int, default=768)
    ap.add_argument("--lanes", type=int, default=0, help="1 = reference container, 0 = lane container")
    ap.add_argument("--ref-blocks", type=int, default=1536, help="blocks per step of the CPU reference arm")
    ap.add_argument("--cpu-blocks", type=int, default=6144, help="blocks of the cpu_baseline sample (6144 = one whole 768x512 B8 image, ~10 s)")
    ap.add_argument("--core", default="tcgen05", choices=["tcgen05", "simt"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--latent-gain", type=float, default=60.0,
                    help="rate of the synthetic model (weights.synth_state_dict): 60 / 5.2 = ~11 bpp (default), 2.5 / 2.0 = ~1 bpp")
    ap.add_argument("--scale-span", type=float, default=5.2)
    ap.add_argument("--no-reference-container", action="store_true")
    ap.add_argument("--no-single-image", action="store_true", help="skip the one-image latency leg")
    ap.add_argument("--refc-images", type=int, default=2048,
                    help="second, larger batch for the reference-container round trip (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (--impl b200)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    sys.dont_write_bytecode = True          # the tree may be read-only: nothing is cached in it

    import lbic_b200
    cfg = lbic_b200.load_config(args.config)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.scaling == "strong":
        if args.total_images % world:
            raise SystemExit(f"--total-images {args.total_images} is not divisible by {world} GPUs")
        args.images = args.total_images // world

    if args.impl == "reference":
        run_reference(args, cfg, rank)
        return

    import torch
    from lbic_b200 import weights
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    from lbic_b200.net import BlockBasedImgCompLossyNetv9

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a B200: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    B, H, W, n = int(cfg.block_size), args.height, args.width, args.images
    Hb, Wb = H // B, W // B
    m = BlockBasedImgCompLossyNetv9(cfg, device=dev)
    m.load_state_dict(weights.synth_state_dict(cfg, 1337, latent_gain=args.latent_gain, scale_span=args.scale_span))
    m.update(force=True)
    m.set_gemm_core(args.core)
    img_u8 = synth_batch_gpu(n, H, W, 1000 + rank, dev)
    # ToTensor (a TRUE division by 255: a tensor divisor, because torch's CUDA kernel for `x / python_scalar` multiplies by
    # the reciprocal and differs from the reference's CPU division in the last bit), AGENT:581, 588-589
    x = arrange_block_pixels_to_channel_dim(
        torch.true_divide(img_u8.float(), torch.full((), 255.0, device=dev)) - 0.5, B)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if x.numel() * 4 < 126e6 else None

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    enc_out = m.encode_device(x, lanes=args.lanes)      # allocates outputs + workspace
    zdec = None

    def step():
        nonlocal zdec
        if flush is not None:
            flush.zero_()
        o = m.encode_device(x, lanes=args.lanes, out=enc_out)
        zdec = m.decode_device(o.streams, o.lens, n, Hb, Wb, lanes=args.lanes)

    def timed(fn, k):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(k):
            fn()
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = m.launch_count()
    ms_total = timed(step, args.steps)
    launches = m.launch_count() - l0
    clocks = sampler.stop() if sampler else None
    parity_ok = bool(torch.equal(zdec, enc_out.zhat))   # the last timed step
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, enc_out.zhat, enc_out.lens, enc_out.streams, zdec)
    pixels_step = world * n * H * W
    value = pixels_step * args.steps / (ms_total * 1e-3) / 1e6

    # separate encode-only / decode-only timings (same warm state)
    ms_enc = timed(lambda: m.encode_device(x, lanes=args.lanes, out=enc_out), args.steps)
    ms_dec = timed(lambda: m.decode_device(enc_out.streams, enc_out.lens, n, Hb, Wb, lanes=args.lanes), args.steps)
    bytes_total = int(enc_out.lens.sum().item())

    # roofline of the dominant kernel (gemm_ws_kernel): one more encode with per-launch CUDA events
    m.set_profiling(True)
    m.encode_device(x, lanes=args.lanes, out=enc_out)
    prof = m.get_profile()
    m.set_profiling(False)
    # per-layer split: the dataflow launch covers a whole step, so this pass uses one launch per layer
    m.set_option("flow", 0)
    m.set_profiling(True)
    m.encode_device(x, lanes=args.lanes, out=enc_out)
    layers = m.get_layer_profile()
    m.set_profiling(False)
    m.set_option("flow", 1)
    peaks = load_peaks()
    ach = prof["gemm_flops"] / (prof["gemm_ms"] * 1e-3) / 1e12 if prof["gemm_ms"] > 0 else 0.0
    macs = macs_per_block(cfg)
    roofline = dict(bound="tensor", kernel="gemm_flow_kernel / gemm_ws_kernel<PAIR> (cta_group::2) + gemm_tc_kernel (tcgen05 kind::f16, fp16 hi/lo operand split, 3 MMAs per product, fp32 TMEM accumulate)",
                    achieved=ach, peak=peaks["tf_sustained"], unit="TFLOP/s", frac=ach / peaks["tf_sustained"],
                    passes=3, frac_pass_adjusted=3 * ach / peaks["tf_sustained"], peak_source=peaks["source"] + " sustained",
                    launches=prof["gemm_launches"], avg_launch_us=1e3 * prof["gemm_ms"] / max(1, prof["gemm_launches"]),
                    gemm_share_of_encode=prof["gemm_ms"] / (ms_enc / args.steps),
                    algorithmic_flop_per_pixel=dict(encode=2 * macs["encode"] / (B * B), decode=2 * macs["decode"] / (B * B)),
                    **measured_traffic(args),
                    binding_resource="data movement under the board's power cap: a 256 x 192 tile costs 26-27 k cycles whatever its K "
                                     "(its MMAs need 10-21 k); ablation: of a layer's time the mainloop is ~60 %, the epilogue's "
                                     "global stores 13-26 %, its arithmetic 3-12 %; not DRAM bound, not instruction bound (TMA "
                                     "stores change nothing); ncu: tensor pipe 57-62 %, L2 34 %, DRAM 36 % of peak "
                                     "(profiles/r2_flow_epilogue.md); the tensor peak is the contract's denominator",
                    layers_tflops_per_layer_launches={k: round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 1)
                                                      for k, v in layers.items() if v["ms"] > 0})

    # the reference's own container (one rANS stream per image, NET:359-360): its decode is serial in raster order,
    # so it is reported beside the headline instead of inside it
    refc = None
    if args.lanes != 1 and not args.no_reference_container:
        o1 = m.encode_device(x, lanes=1)                                     # warm-up of both directions
        z1 = m.decode_device(o1.streams, o1.lens, n, Hb, Wb, lanes=1)
        torch.cuda.synchronize()
        ms_e1 = min(timed(lambda: m.encode_device(x, lanes=1, out=o1), 1) for _ in range(2))
        ms_d1 = min(timed(lambda: m.decode_device(o1.streams, o1.lens, n, Hb, Wb, lanes=1), 1) for _ in range(2))
        z1 = m.decode_device(o1.streams, o1.lens, n, Hb, Wb, lanes=1)
        refc = dict(container="reference (1 rANS64 stream per image)", images_per_gpu=n,
                    value=pixels_step / ((ms_e1 + ms_d1) * 1e-3) / 1e6, unit="Mpixel/s (encode+decode round trip)",
                    encode_mpix_s=pixels_step / (ms_e1 * 1e-3) / 1e6, decode_mpix_s=pixels_step / (ms_d1 * 1e-3) / 1e6,
                    enc_dec_identical=bool(torch.equal(z1, o1.zhat)), bpp=8.0 * int(o1.lens.sum().item()) / (n * H * W))
        del o1, z1

    # end to end through the reference-facing host call: 8-bit images in pinned host memory -> bitstreams in host memory
    # (ToTensor, -0.5, padding, space-to-depth, compress: AGENT:581-592) -> 8-bit reconstructions in host memory
    # (decompress, depth-to-space, 8-bit quantisation: AGENT:598, 610, 628); H2D + D2H copies inside the timed region
    e2e = None
    if not args.no_e2e:
        import numpy as np
        from lbic_b200 import _lib
        L = _lib.lib()
        ih = torch.empty(img_u8.shape, dtype=torch.uint8).pin_memory()
        ih.copy_(img_u8)
        oh = torch.empty(img_u8.shape, dtype=torch.uint8).pin_memory()
        cap = int(min(enc_out.streams.shape[1], ((int(enc_out.lens.max().item()) * 2 + 4096) + 3) // 4 * 4))
        sh = torch.empty(n, cap, dtype=torch.uint8).pin_memory()
        lh = torch.zeros(n, dtype=torch.int32).pin_memory()

        def e2e_step():
            _lib.check(L.lbic_encode_images_u8_host(m._need(), ih.data_ptr(), n, H, W, None, sh.data_ptr(), cap,
                                                    lh.data_ptr(), args.lanes))
            _lib.check(L.lbic_decode_images_u8_host(m._need(), sh.data_ptr(), lh.data_ptr(), cap, n, H, W, oh.data_ptr(),
                                                    args.lanes))
        e2e_step()
        ms_e2e = timed(e2e_step, args.steps)
        lens_h = lh.numpy().astype(np.int64)
        from lbic_b200.layout import arrange_channel_dim_to_block_pixels
        want = (arrange_channel_dim_to_block_pixels(enc_out.zhat, B) + 0.5).mul_(255).add_(0.5).clamp_(0, 255).to(torch.uint8)
        e2e = dict(value=pixels_step * args.steps / (ms_e2e * 1e-3) / 1e6, unit="Mpixel/s",
                   h2d_bytes_per_step=ih.numel() + int(lens_h.sum()) + 4 * n,
                   d2h_bytes_per_step=int(lens_h.sum()) + 4 * n + oh.numel(),
                   api="lbic_encode_images_u8_host + lbic_decode_images_u8_host (8-bit images and bitstreams in pinned host "
                       "memory; copies overlapped with the wavefront in bands of block rows)",
                   parity=bool(torch.equal(oh.to(dev), want)), ratio_to_device_value=None)
        e2e["ratio_to_device_value"] = e2e["value"] / value
        del ih, oh, sh, want

    # The reference container's decode is Hb * Wb strictly serial steps whose time does not depend on the number of
    # images (profiles/r2_wave_latency.md), so its throughput grows with the batch: the same round trip at a larger one.
    if refc is not None and args.refc_images > n and args.lanes != 1:
        n2 = args.refc_images
        free_b, _ = torch.cuda.mem_get_info()
        need = 30e6 * n2 * (H * W) / (512 * 768)           # ~27 MB of workspace + I/O per 768x512 image (B8 N768)
        ok = torch.tensor([1 if free_b + torch.cuda.memory_reserved() > need * 1.3 else 0], device=dev)
        if dist is not None:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)          # every rank takes the same branch (the timing has barriers)
        if int(ok.item()):
            x2 = x.repeat((n2 + n - 1) // n, 1, 1, 1)[:n2].contiguous()
            o2 = m.encode_device(x2, lanes=1)
            z2 = m.decode_device(o2.streams, o2.lens, n2, Hb, Wb, lanes=1)
            torch.cuda.synchronize()
            ms_e2 = timed(lambda: m.encode_device(x2, lanes=1, out=o2), 1)
            ms_d2 = timed(lambda: m.decode_device(o2.streams, o2.lens, n2, Hb, Wb, lanes=1), 1)
            px2 = world * n2 * H * W
            refc["larger_batch"] = dict(images_per_gpu=n2, value=px2 / ((ms_e2 + ms_d2) * 1e-3) / 1e6,
                                        encode_mpix_s=px2 / (ms_e2 * 1e-3) / 1e6, decode_mpix_s=px2 / (ms_d2 * 1e-3) / 1e6,
                                        enc_dec_identical=bool(torch.equal(z2, o2.zhat)))
            del x2, o2, z2
            torch.cuda.empty_cache()

    # The reference's own call pattern is ONE image per compress / decompress call (eval_model, AGENT:578-599): a chain of
    # Hb + 2 Wb dependent wavefront steps, i.e. latency, not throughput (the persistent wavefront kernel, gemm_wave.cu).
    single = None
    if not args.no_single_image:
        x1 = x[:1].contiguous()
        o1 = m.encode_device(x1, lanes=args.lanes)
        z1 = m.decode_device(o1.streams, o1.lens, 1, Hb, Wb, lanes=args.lanes)
        torch.cuda.synchronize()
        l1 = m.launch_count()
        ms_e = min(timed(lambda: m.encode_device(x1, lanes=args.lanes, out=o1), 1) for _ in range(3))
        le = (m.launch_count() - l1) // 3
        ms_d = min(timed(lambda: m.decode_device(o1.streams, o1.lens, 1, Hb, Wb, lanes=args.lanes), 1) for _ in range(3))
        z1 = m.decode_device(o1.streams, o1.lens, 1, Hb, Wb, lanes=args.lanes)
        single = dict(images=1, size=f"{W}x{H}", encode_ms=ms_e, decode_ms=ms_d, launches_per_encode=int(le),
                      container="reference" if args.lanes == 1 else "lane", timing="device-resident, CUDA events, best of 3",
                      enc_dec_identical=bool(torch.equal(z1, o1.zhat)))
        del x1, o1, z1

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:   # reported at N=1 only (host cores are shared by the ranks)
        threads = os.cpu_count() or 1
        r = cpu_baseline(cfg, H, W, args.cpu_blocks, threads)
        cpu = dict(value=r["mpix_s"], unit="Mpixel/s", cores=threads, kind="port",
                   sample=f"first {r['blocks']} raster-order blocks of one {W}x{H} image: oracle port of the reference "
                          f"compress loop ({r['enc_s']:.1f} s) + decompress loop ({r['dec_s']:.1f} s), torch CPU fp32",
                   encode_mpix_s=r["enc_mpix_s"], decode_mpix_s=r["dec_mpix_s"])
        # the reference's own CPU setting is ONE thread (AGENT:565-566): a smaller sample of the same loops
        r1 = cpu_baseline(cfg, H, W, max(16, args.cpu_blocks // 16), 1)
        cpu["one_thread"] = dict(value=r1["mpix_s"], cores=1, encode_mpix_s=r1["enc_mpix_s"], decode_mpix_s=r1["dec_mpix_s"],
                                 sample=f"first {r1['blocks']} blocks, torch.set_num_threads(1) as agents/blkbsdimgcomp_agent.py:565-566")

    if rank == 0:
        line = dict(metric="encode+decode Mpixel/s", value=value, unit="Mpixel/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms_total / args.steps, higher_is_better=True, scaling=args.scaling,
                    vs_baseline=None, dtype="f16x3->f32", data="synthetic", config=workload_config(args, cfg),
                    encode_mpix_s=pixels_step * args.steps / (ms_enc * 1e-3) / 1e6,
                    decode_mpix_s=pixels_step * args.steps / (ms_dec * 1e-3) / 1e6,
                    bpp=8.0 * bytes_total / (n * H * W), enc_dec_identical=parity_ok,
                    gpu_launches=int(launches), clocks=clocks, roofline=roofline, e2e=e2e, cpu_baseline=cpu,
                    reference_container=refc, single_image=single,
                    gemm_core=args.core)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
