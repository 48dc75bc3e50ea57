"""Golden fixtures for the open-loop forward (the reference's model.forward(zhat, x), NET:90-106; SURVEY.md 8(f) rank 2).

Runs the UNMODIFIED reference model (imported through oracle/ref_shim) in eval mode on the inputs of the existing
closed-loop cases -- x, and as context the closed-loop reconstruction zhat of case_<name>.npz -- asserts that
oracle.nets.forward_open_loop reproduces it, and writes forward_<name>.npz:
    xhat       (1, 3B^2, Hb, Wb) fp32   reference forward output (not clamped)
    selfinfo   (1, M, Hb, Wb)    fp32   -log2 of the Gaussian-conditional likelihoods
    symbols    (Hb, Wb, M)       int16  round(y - means) of the oracle restatement
Run with a checkout of the reference: LBIC_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden_forward.py
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

CASES = ["B8_lowrate_6x9", "B8_lowrate_5x12_harsh", "B4_highrate_7x10", "B8_highrate_4x7", "B16_lowrate_3x5"]


def main():
    torch.set_num_threads(8)
    torch.use_deterministic_algorithms(True)
    ref = load_reference.load()
    for name in CASES:
        c = np.load(os.path.join(HERE, f"case_{name}.npz"))
        cfg = lbic_b200.load_config(str(c["config"]))
        sd = weights.synth_state_dict(cfg, int(c["seed"]), harsh=bool(c["harsh"]))
        m = ref.BlockBasedImgCompLossyNetv9(cfg).eval()
        m.load_state_dict(sd, strict=False)
        m.update(force=True)
        x, zhat = torch.from_numpy(c["x"]), torch.from_numpy(c["zhat"])
        with torch.no_grad():
            xhat, info = m(zhat, x)
        P = nets.effective_params(sd, cfg)
        oxhat, oinfo, osym = nets.forward_open_loop(P, zhat, x)
        dx = float((oxhat - xhat).abs().max())
        di = float((oinfo - info).abs().max())
        assert dx < 1e-5 and di < 1e-3, f"{name}: oracle forward differs from the reference (xhat {dx:.2e}, info {di:.2e})"
        np.savez_compressed(os.path.join(HERE, f"forward_{name}.npz"), xhat=xhat.numpy(), selfinfo=info.numpy(),
                            symbols=osym[0].numpy().astype(np.int16))
        print(f"{name}: oracle vs reference xhat maxdiff {dx:.2e}, selfinfo maxdiff {di:.2e}, bits {float(info.sum()):.1f}, "
              f"xhat range [{float(xhat.min()):.2f}, {float(xhat.max()):.2f}]")


if __name__ == "__main__":
    main()
