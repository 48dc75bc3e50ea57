import ctypes, sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import lbic_b200
from lbic_b200 import _lib
from lbic_b200.net import BlockBasedImgCompLossyNetv9
from lbic_b200.weights import synth_state_dict
cfg = lbic_b200.load_config("B8_lowrate")
m = BlockBasedImgCompLossyNetv9(cfg, device="cuda:0")
m.load_state_dict(synth_state_dict(cfg)); m.update()
L = _lib.lib()
def opt(o, v): _lib.check(L.lbic_set_option(m._need(), o, v))
names = ["RAW", "PREGDN", "GDN", "QUANT", "LRELU", "KSI", "RECON"]
def run(R, K, C, epi, pair, iters=30):
    opt(_lib.LBIC_OPT_WS, 2); opt(_lib.LBIC_OPT_PAIR, pair)
    ms = ctypes.c_double()
    _lib.check(L.lbic_debug_gemm_bench(m._need(), R, K, C, epi, iters, ctypes.byref(ms)))
    tf = 2.0 * R * K * C / (ms.value * 1e-3) / 1e12
    print(f"pair={pair} R={R:6d} K={K:5d} C={C:4d} {names[epi]:7s}: {ms.value*1e3:8.1f} us ({3*tf:7.1f} mma)", flush=True)
for pair in (1, 3):
    for (K, C, e) in [(768, 768, 0), (768, 768, 1), (768, 768, 2), (1152, 960, 4), (768, 1152, 4), (672, 672, 1), (672, 672, 2), (576, 576, 2), (960, 768, 1)]:
        run(24576, K, C, e, pair)
