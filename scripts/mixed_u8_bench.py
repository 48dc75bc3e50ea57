"""Mixed-size batches of 8-bit images from host memory (lbic_encode_images_u8_host_mixed /
lbic_decode_images_u8_host_mixed) against the device-resident mixed call and against ImageCodec.encode_many /
decode_many plus an 8-bit conversion.  B8_lowrate, lane container, the two sets of scripts/mixed_batch_bench.py.
Device-resident: CUDA events; host calls: host clock around calls that end synchronised; best of --reps timed passes
after one warm-up pass of every mode.  Checks that every route gives the same streams and 8-bit images.
    python scripts/mixed_u8_bench.py --set kodak   > profiles/r3_mixed_u8_kodak.json
    python scripts/mixed_u8_bench.py --set dataset > profiles/r3_mixed_u8_dataset.json
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import lbic_b200  # noqa: E402
from lbic_b200 import _lib, weights  # noqa: E402
from lbic_b200.codec import ImageCodec, pack_container  # noqa: E402
from lbic_b200.layout import arrange_block_pixels_to_channel_dim, arrange_channel_dim_to_block_pixels  # noqa: E402
from lbic_b200.net import BlockBasedImgCompLossyNetv9  # noqa: E402
from mixed_batch_bench import image_sizes  # noqa: E402


def best(fn, reps, device_events):
    times, out = [], None
    for _ in range(reps):
        torch.cuda.synchronize()
        if device_events:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = fn()
            b.record()
            torch.cuda.synchronize()
            times.append(a.elapsed_time(b))
        else:
            t0 = time.perf_counter()
            out = fn()
            times.append((time.perf_counter() - t0) * 1e3)
    return min(times), times, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--set", choices=["kodak", "dataset"], required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=2024)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    cfg = lbic_b200.load_config("B8_lowrate")
    m = BlockBasedImgCompLossyNetv9(cfg, device=dev)
    m.load_state_dict(weights.synth_state_dict(cfg, 1337))
    m.update(force=True)
    B = int(cfg.block_size)
    sizes = image_sizes(args.set, args.seed)
    imgs = [weights.synth_image_u8(H, W, seed=args.seed + i) for i, (H, W) in enumerate(sizes)]
    mpix = sum(H * W for H, W in sizes) / 1e6
    # device-resident blocks built the reference way (CPU true division, -0.5, space-to-depth; sizes are multiples of B)
    xs = [arrange_block_pixels_to_channel_dim((torch.from_numpy(a[None]).float().div(255) - 0.5).to(dev), B).contiguous()
          for a in imgs]
    shapes = [tuple(x.shape[2:]) for x in xs]
    codec = ImageCodec(m, lanes=0)
    hwc = [np.ascontiguousarray(a.transpose(1, 2, 0)) for a in imgs]
    res, outs = {}, {}

    def dev_enc():
        return m.encode_device_mixed(xs, lanes=0)

    def dev_dec(o):
        return lambda: m.decode_device_mixed(o.streams, o.lens, shapes, lanes=0)

    # the C calls alone: inputs packed once into pinned memory, outputs into pinned buffers (what a caller that keeps its
    # images in pinned memory pays); the python methods add the packing and unpacking copies on the host thread
    n = len(sizes)
    packed, _ = m._pack_u8(imgs, False)
    packed = packed[: sum(3 * H * W for H, W in sizes)].clone().pin_memory()
    rec_pin = torch.empty_like(packed).pin_memory()
    dec_pin = torch.empty_like(packed).pin_memory()
    Hs = (ctypes.c_int * n)(*[s[0] for s in sizes])
    Ws = (ctypes.c_int * n)(*[s[1] for s in sizes])
    cap = (max(m.stream_bound(-(-H // B), -(-W // B), 0) for H, W in sizes) + 3) // 4 * 4
    streams = torch.empty(n, cap, dtype=torch.uint8).pin_memory()
    call_lens = torch.zeros(n, dtype=torch.int32).pin_memory()

    def call_enc():
        _lib.check(_lib.lib().lbic_encode_images_u8_host_mixed(m._need(), packed.data_ptr(), n, Hs, Ws, rec_pin.data_ptr(),
                                                               streams.data_ptr(), cap, call_lens.data_ptr(), 0))
        return streams, call_lens

    def call_dec(_):
        def f():
            _lib.check(_lib.lib().lbic_decode_images_u8_host_mixed(m._need(), streams.data_ptr(), call_lens.data_ptr(), cap, n,
                                                                   Hs, Ws, dec_pin.data_ptr(), 0))
            return dec_pin
        return f

    def u8_enc():
        return m.compress_images_u8_mixed(imgs, lanes=0, return_recon=True)

    def u8_dec(s):
        return lambda: m.decompress_images_u8_mixed(s, sizes, lanes=0)

    def codec_enc():
        return codec.encode_many(hwc)

    def codec_dec(blobs):
        return lambda: [r[0].mul(255).add_(0.5).clamp_(0, 255).to(torch.uint8).cpu().numpy()
                        for r in codec.decode_many(blobs)]

    modes = [("device_resident", dev_enc, dev_dec, True, None),
             ("u8_host_call_bands16", call_enc, call_dec, False, 16), ("u8_host_call_bands1", call_enc, call_dec, False, 1),
             ("u8_host_call_bands16_again", call_enc, call_dec, False, 16),
             ("u8_host_call_bands1_again", call_enc, call_dec, False, 1),
             ("u8_host_python_methods", u8_enc, u8_dec, False, 16),
             ("encode_many_decode_many", codec_enc, codec_dec, False, None)]
    for name, enc, dec, ev, bands in modes:
        if bands:
            m.set_option("host_bands", bands)
        e = enc()                                   # warm-up
        dec(e if not isinstance(e, tuple) else e[0])()
        m.check_errors()
        t_enc, all_enc, e = best(enc, args.reps, ev)
        key = e if not isinstance(e, tuple) else e[0]
        t_dec, all_dec, d = best(dec(key), args.reps, ev)
        m.check_errors()
        res[name] = dict(encode_ms=t_enc, decode_ms=t_dec, encode_ms_all=all_enc, decode_ms_all=all_dec,
                         encode_mpix_s=mpix / (t_enc / 1e3), decode_mpix_s=mpix / (t_dec / 1e3),
                         round_trip_mpix_s=mpix / ((t_enc + t_dec) / 1e3))
        outs[name] = (e, d)
    m.set_option("host_bands", 16)
    # identical outputs: streams of every route, 8-bit images of the u8 calls against save_image's quantisation of the
    # device-resident reconstructions
    de, dd = outs["device_resident"]
    dev_lens = de.lens.cpu().tolist()
    dev_streams = [de.streams[i, : dev_lens[i]].cpu().numpy().tobytes() for i in range(len(xs))]
    want_u8 = [(arrange_channel_dim_to_block_pixels(z, B) + 0.5).mul(255).add_(0.5).clamp_(0, 255).to(torch.uint8)
               .cpu().numpy()[0] for z in dd]
    identical = True
    (s, rec), dec_imgs = outs["u8_host_python_methods"]
    identical &= s == dev_streams
    identical &= all(np.array_equal(a, b) and np.array_equal(c, b) for a, b, c in zip(rec, want_u8, dec_imgs))
    want_packed = np.concatenate([w.reshape(-1) for w in want_u8])
    identical &= np.array_equal(rec_pin.numpy(), want_packed) and np.array_equal(dec_pin.numpy(), want_packed)
    identical &= call_lens.tolist() == dev_lens
    identical &= [streams[i, : int(call_lens[i])].numpy().tobytes() for i in range(n)] == dev_streams
    blobs, codec_imgs = outs["encode_many_decode_many"]
    identical &= blobs == [pack_container(s, H=H, W=W, B=B, KS=codec.KS, N=codec.N, M=codec.M, lanes=0)
                           for s, (H, W) in zip(dev_streams, sizes)]
    identical &= all(np.array_equal(a, b) for a, b in zip(codec_imgs, want_u8))
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    rt = {k: v["round_trip_mpix_s"] for k, v in res.items()}
    print(json.dumps(dict(
        set=args.set, config="B8_lowrate", container="lane", images=len(imgs), mpixel=mpix,
        u8_bytes_each_way=int(sum(3 * H * W for H, W in sizes)), gpu=gpu, reps=args.reps,
        timing="device-resident: CUDA events; host calls: host clock, call ends synchronised; best of reps after one "
               "warm-up pass. u8_host_call_*: the C calls alone, images, reconstructions and streams in pinned host "
               "memory; u8_host_python_methods: compress_images_u8_mixed / decompress_images_u8_mixed from numpy arrays "
               "(packing into and unpacking from pinned staging included); encode_many_decode_many: ImageCodec on HWC "
               "arrays plus save_image's 8-bit conversion",
        all_outputs_identical=bool(identical),
        e2e_over_device_bands16=max(rt["u8_host_call_bands16"], rt["u8_host_call_bands16_again"]) / rt["device_resident"],
        e2e_over_device_bands1=max(rt["u8_host_call_bands1"], rt["u8_host_call_bands1_again"]) / rt["device_resident"],
        python_methods_over_device=rt["u8_host_python_methods"] / rt["device_resident"],
        python_methods_over_encode_many=rt["u8_host_python_methods"] / rt["encode_many_decode_many"],
        modes=res), indent=1))


if __name__ == "__main__":
    main()
