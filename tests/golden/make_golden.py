"""Generates the golden fixtures in this directory by running the UNMODIFIED reference model
(a checkout of it at $LBIC_REFERENCE_ROOT, imported through oracle/ref_shim) on seeded synthetic inputs.

Needs no GPU; the tests only read the committed .npz files.
    LBIC_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden.py

Each case_<name>.npz holds, for one (config, grid) pair with weights = synth_state_dict(cfg, seed):
    x         (1, 3B^2, Hb, Wb) fp32   input blocks in [-0.5, 0.5]
    zhat      same shape               reference compress() reconstruction (NET:319-361)
    zhat_dec  same shape               reference decompress() output (NET:400-452)
    stream    uint8                    reference bitstream
    symbols   (Hb, Wb, M) int16        quantised latents  (oracle loop; stream identity with the reference
    indexes   (Hb, Wb, M) uint8        CDF indexes         is asserted below, so these are the reference's)
tables.npz holds the reference's quantized_cdf / cdf_length / offset / scale_table after update().
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

import lbic_b200  # noqa: E402
from lbic_b200 import weights  # noqa: E402
from oracle import nets  # noqa: E402
from oracle.ref_shim import load_reference  # noqa: E402

CASES = [
    # name, config, Hb, Wb, seed, harsh, image kind
    ("B8_lowrate_6x9", "B8_lowrate", 6, 9, 1337, False, "smooth"),
    ("B8_lowrate_5x12_harsh", "B8_lowrate", 5, 12, 7, True, "noise"),
    ("B4_highrate_7x10", "B4_highrate", 7, 10, 1337, False, "smooth"),
    ("B8_highrate_4x7", "B8_highrate", 4, 7, 1337, False, "smooth"),
    ("B16_lowrate_3x5", "B16_lowrate", 3, 5, 1337, False, "smooth"),
]


def main():
    torch.set_num_threads(8)
    torch.use_deterministic_algorithms(True)
    ref = load_reference.load()
    tables_saved = False
    for name, cfgname, Hb, Wb, seed, harsh, kind in CASES:
        cfg = lbic_b200.load_config(cfgname)
        sd = weights.synth_state_dict(cfg, seed, harsh=harsh)
        m = ref.BlockBasedImgCompLossyNetv9(cfg).eval()
        m.load_state_dict(sd, strict=False)
        m.update(force=True)
        B = cfg.block_size
        img = weights.synth_images(1, Hb * B, Wb * B, seed0=1000 + seed, kind=kind)
        x = nets.arrange_block_pixels_to_channel_dim(img - 0.5, B)
        L = sum(int(k) // 2 for k in cfg.KS)
        with torch.no_grad():
            stream, zhat = m.compress(x, [L, L, L], cfg.M)
            zdec = m.decompress(stream, [L, L, L], x.shape, cfg.M, "cpu")
        g = m.conditional_gaussian_model
        tabs = (g.quantized_cdf, g.cdf_length, g.offset)
        P = nets.effective_params(sd, cfg)
        ostream, ozhat, syms, idxs = nets.compress(P, tabs, x)
        assert ostream == stream, f"{name}: oracle stream differs from the reference"
        assert torch.equal(ozhat, zhat), f"{name}: oracle zhat differs from the reference"
        assert syms.abs().max() < 2 ** 15
        np.savez_compressed(os.path.join(HERE, f"case_{name}.npz"),
                            config=cfgname, seed=seed, harsh=harsh,
                            x=x.numpy(), zhat=zhat.numpy(), zhat_dec=zdec.numpy(),
                            stream=np.frombuffer(stream, dtype=np.uint8),
                            symbols=syms.numpy().astype(np.int16), indexes=idxs.numpy().astype(np.uint8))
        print(f"{name}: {len(stream)} bytes, |sym|max {int(syms.abs().max())}, nonzero "
              f"{float((syms != 0).float().mean()):.2f}, enc/dec maxdiff {float((zhat - zdec).abs().max()):.1e}, "
              f"clamped {float((zhat.abs() >= 0.5).float().mean()):.2f}")
        if not tables_saved:
            np.savez_compressed(os.path.join(HERE, "tables.npz"), quantized_cdf=g.quantized_cdf.numpy(),
                                cdf_length=g.cdf_length.numpy(), offset=g.offset.numpy(),
                                scale_table=g.scale_table.numpy())
            tables_saved = True


if __name__ == "__main__":
    main()
