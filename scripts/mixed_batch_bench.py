"""Throughput of a set of differently sized images: one call per image, one call per distinct shape, and one mixed-size
call (lbic_encode_mixed / lbic_decode_mixed).  B8_lowrate, lane container, device-resident, CUDA events, best of
--reps timed passes after one warm-up pass of every mode.  Also checks that the mixed call's streams and
reconstructions equal the per-image calls'.
    python scripts/mixed_batch_bench.py --set kodak   > profiles/r3_mixed_batch_kodak.json
    python scripts/mixed_batch_bench.py --set dataset > profiles/r3_mixed_batch_dataset.json
Run one process per set.
"""
import argparse
import json
import os
import random
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lbic_b200  # noqa: E402
from lbic_b200 import weights  # noqa: E402
from lbic_b200.layout import arrange_block_pixels_to_channel_dim  # noqa: E402
from lbic_b200.net import BlockBasedImgCompLossyNetv9  # noqa: E402


def image_sizes(which, seed):
    """(H, W) pixel sizes, multiples of the block size 8."""
    rng = random.Random(seed)
    if which == "kodak":   # 24 images, mostly landscape 768x512, a few portrait 512x768
        portrait = set(rng.sample(range(24), 4))
        return [(768, 512) if i in portrait else (512, 768) for i in range(24)]
    sizes = set()          # 256 distinct sizes, 256 to 1024 pixels per side
    while len(sizes) < 256:
        sizes.add((8 * rng.randint(32, 128), 8 * rng.randint(32, 128)))
    return sorted(sizes, key=lambda s: rng.random())


def timed(fn, reps):
    times, out = [], None
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return min(times), times, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--set", choices=["kodak", "dataset"], required=True)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--seed", type=int, default=2024)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    cfg = lbic_b200.load_config("B8_lowrate")
    m = BlockBasedImgCompLossyNetv9(cfg, device=dev)
    m.load_state_dict(weights.synth_state_dict(cfg, 1337))
    m.update(force=True)
    B = int(cfg.block_size)
    sizes = image_sizes(args.set, args.seed)
    xs = []
    for i, (H, W) in enumerate(sizes):
        img = weights.synth_images(1, H, W, seed0=args.seed + i).to(dev)
        xs.append(arrange_block_pixels_to_channel_dim(img - 0.5, B).contiguous())
    shapes = [tuple(x.shape[2:]) for x in xs]
    mpix = sum(H * W for H, W in sizes) / 1e6
    groups = {}
    for i, s in enumerate(shapes):
        groups.setdefault(s, []).append(i)
    grouped = {s: torch.cat([xs[i] for i in idx]) for s, idx in groups.items()}

    def per_image_enc():
        return [m.encode_device(x, lanes=0) for x in xs]

    def per_image_dec(encs):
        return lambda: [m.decode_device(o.streams, o.lens, 1, *s, lanes=0) for o, s in zip(encs, shapes)]

    def per_shape_enc():
        return {s: m.encode_device(x, lanes=0) for s, x in grouped.items()}

    def per_shape_dec(encs):
        return lambda: {s: m.decode_device(o.streams, o.lens, len(groups[s]), *s, lanes=0) for s, o in encs.items()}

    def mixed_enc():
        return m.encode_device_mixed(xs, lanes=0)

    def mixed_dec(o):
        return lambda: m.decode_device_mixed(o.streams, o.lens, shapes, lanes=0)

    res = {}
    for name, enc, dec in (("per_image", per_image_enc, per_image_dec), ("per_shape", per_shape_enc, per_shape_dec),
                           ("mixed", mixed_enc, mixed_dec)):
        e = enc()                      # warm-up (workspace growth, module loads)
        dec(e)()
        m.check_errors()
        t_enc, all_enc, e = timed(enc, args.reps)
        t_dec, all_dec, d = timed(dec(e), args.reps)
        m.check_errors()
        res[name] = dict(calls=len(xs) if name == "per_image" else len(groups) if name == "per_shape" else 1,
                         encode_ms=t_enc, decode_ms=t_dec, encode_ms_all=all_enc, decode_ms_all=all_dec,
                         encode_mpix_s=mpix / (t_enc / 1e3), decode_mpix_s=mpix / (t_dec / 1e3),
                         round_trip_mpix_s=mpix / ((t_enc + t_dec) / 1e3))
        res[name]["_out"] = (e, d)
    # the mixed call's outputs are the per-image calls' outputs
    pe, pd = res["per_image"].pop("_out")
    me, md = res["mixed"].pop("_out")
    res["per_shape"].pop("_out")
    lens_mixed = me.lens.cpu().tolist()
    identical = True
    for i, o in enumerate(pe):
        n = int(o.lens[0])
        identical &= lens_mixed[i] == n and torch.equal(me.streams[i, :n], o.streams[0, :n])
        identical &= torch.equal(me.zhat[i], o.zhat) and torch.equal(md[i], pd[i])
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    print(json.dumps(dict(set=args.set, config="B8_lowrate", container="lane", images=len(xs),
                          distinct_shapes=len(groups), mpixel=mpix, gpu=gpu, reps=args.reps,
                          timing="device-resident, CUDA events, best of reps after one warm-up pass",
                          mixed_equals_per_image=bool(identical),
                          mixed_vs_per_image_round_trip=res["mixed"]["round_trip_mpix_s"] /
                          res["per_image"]["round_trip_mpix_s"],
                          mixed_vs_per_shape_round_trip=res["mixed"]["round_trip_mpix_s"] /
                          res["per_shape"]["round_trip_mpix_s"], modes=res), indent=1))


if __name__ == "__main__":
    main()
