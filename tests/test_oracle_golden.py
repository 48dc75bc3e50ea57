"""CPU tests (-m "not gpu"): the oracle against the golden vectors the reference itself produced
(tests/golden/make_golden.py), plus independent cross-checks of the restated native functions."""
import numpy as np
import pytest
import torch

import lbic_b200
from lbic_b200 import weights
from oracle import native, nets
from conftest import golden_cases, load_case, load_tables


def _setup(c):
    cfg = lbic_b200.load_config(str(c["config"]))
    sd = weights.synth_state_dict(cfg, int(c["seed"]), harsh=bool(c["harsh"]))
    return cfg, nets.effective_params(sd, cfg)


@pytest.fixture(scope="module")
def tables():
    t = nets.build_tables()
    return t


# The golden closed-loop vectors were produced with 8 intra-op threads, and MKL's fp32 GEMM splits its reduction by the
# thread count (1, 2, 4, 16 or 64 threads move zhat by 1e-7 .. 1e-5): bit-exact comparisons run the oracle on 8 threads
# whatever the host has.
GOLDEN_THREADS = 8


@pytest.fixture
def golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def test_tables_equal_reference(tables):
    ref = load_tables()
    assert np.array_equal(tables[0].numpy(), ref["quantized_cdf"])
    assert np.array_equal(tables[1].numpy(), ref["cdf_length"])
    assert np.array_equal(tables[2].numpy(), ref["offset"])
    assert tables[0].shape == (64, 3133)
    assert int(tables[1].min()) == 5 and int(tables[1].max()) == 3133


@pytest.mark.parametrize("case", golden_cases())
def test_oracle_reproduces_reference(case, tables, golden_threads):
    c = load_case(case)
    cfg, P = _setup(c)
    x = torch.from_numpy(c["x"])
    stream, zhat, syms, idxs = nets.compress(P, tables, x)
    assert np.array_equal(syms.numpy(), c["symbols"].astype(np.int32))
    assert np.array_equal(idxs.numpy(), c["indexes"].astype(np.int32))
    assert torch.equal(zhat, torch.from_numpy(c["zhat"]))
    assert stream == c["stream"].tobytes()
    zdec = nets.decompress_loop(P, tables, stream, x.shape)
    assert torch.equal(zdec, torch.from_numpy(c["zhat_dec"]))
    # fixed point (SURVEY.md A.6): one parallel evaluation on the final zhat reproduces the loop
    s2, i2, xh2, _, _ = nets.whole_image_eval(P, x, zhat)
    assert int((s2[0] != syms).sum()) == 0 and int((i2[0] != idxs).sum()) == 0
    assert float((xh2 - zhat).abs().max()) < 1e-4   # fp32 accumulation order (batched vs per-block conv)


def _py_pmf_to_cdf(pmf, precision=16):
    """Independent pure-Python transcription of SURVEY.md Appendix B.1."""
    import math
    cdf = [0] + [int(math.floor(np.float32(p) * np.float32(1 << precision) + np.float32(0.5))) for p in pmf]
    total = sum(cdf)
    cdf = [((1 << precision) * c) // total for c in cdf]
    for i in range(1, len(cdf)):
        cdf[i] += cdf[i - 1]
    cdf[-1] = 1 << precision
    n = len(cdf) - 1
    for i in range(n):
        if cdf[i] == cdf[i + 1]:
            best, steal = None, -1
            for j in range(n):
                f = cdf[j + 1] - cdf[j]
                if f > 1 and (best is None or f < best):
                    best, steal = f, j
            if steal < i:
                for j in range(steal + 1, i + 1):
                    cdf[j] -= 1
            else:
                for j in range(i + 1, steal + 1):
                    cdf[j] += 1
    return cdf


@pytest.mark.parametrize("case", golden_cases())
def test_oracle_forward_reproduces_reference_forward(case):
    """forward_<case>.npz = the UNMODIFIED reference's model.forward(zhat, x) (tests/golden/make_golden_forward.py)."""
    import os
    from conftest import GOLDEN
    c = load_case(case)
    f = np.load(os.path.join(GOLDEN, f"forward_{case}.npz"))
    cfg, P = _setup(c)
    xhat, info, sym = nets.forward_open_loop(P, torch.from_numpy(c["zhat"]), torch.from_numpy(c["x"]))
    assert np.array_equal(sym[0].numpy(), f["symbols"].astype(np.int32))
    assert float((xhat - torch.from_numpy(f["xhat"])).abs().max()) <= 1e-5 * max(1.0, float(np.abs(f["xhat"]).max()))
    assert float((info - torch.from_numpy(f["selfinfo"])).abs().max()) < 1e-3


def test_pmf_to_quantized_cdf_against_python_transcription():
    rng = np.random.default_rng(0)
    for n in (3, 17, 200):
        p = rng.random(n).astype(np.float32) ** 6
        p /= p.sum()
        p[rng.integers(0, n, size=max(1, n // 3))] = 0.0     # force zero-frequency fix-ups
        got = native.pmf_to_quantized_cdf(p)
        assert list(got) == _py_pmf_to_cdf(p.tolist())
        assert got[0] == 0 and got[-1] == 65536 and (np.diff(got) > 0).all()


class _PyRans:
    """Independent pure-Python transcription of SURVEY.md Appendix B.2 (encoder only)."""
    L = 1 << 31

    @classmethod
    def encode(cls, symbols, indexes, cdf, lens, offs):
        pushed = []
        for s, ci in zip(symbols, indexes):
            row, maxv = cdf[ci], int(lens[ci]) - 2
            v, raw = int(s) - int(offs[ci]), 0
            if v < 0:
                raw, v = -2 * v - 1, maxv
            elif v >= maxv:
                raw, v = 2 * (v - maxv), maxv
            pushed.append((int(row[v]), int(row[v + 1] - row[v]), False))
            if v == maxv:
                nb = 0
                while (raw >> (4 * nb)) != 0:
                    nb += 1
                val = nb
                while val >= 15:
                    pushed.append((15, 16, True))
                    val -= 15
                pushed.append((val, val + 1, True))
                for j in range(nb):
                    q = (raw >> (4 * j)) & 15
                    pushed.append((q, q + 1, True))
        x, words = cls.L, []
        for start, rng, bypass in reversed(pushed):
            freq = (1 << 12) if bypass else rng
            if x >= ((cls.L >> 16) << 32) * freq:
                words.append(x & 0xFFFFFFFF)
                x >>= 32
            x = ((x << 4) | start) if bypass else ((x // rng) << 16) + (x % rng) + start
        words.append(x >> 32)
        words.append(x & 0xFFFFFFFF)
        return np.array(words[::-1], dtype=np.uint32).tobytes()


def _rand_symbols(tabs, n, seed, n_escape):
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, 64, size=n).astype(np.int32)
    sym = np.rint(rng.normal(0, 1, size=n) * tabs["scale_table"][idx]).astype(np.int32)
    pos = rng.integers(0, n, size=n_escape)
    sym[pos] += rng.integers(-70000, 70000, size=n_escape).astype(np.int32)
    return sym, idx


def test_rans_c_against_python_transcription_and_roundtrip():
    tabs = load_tables()
    T = native.Tables(tabs["quantized_cdf"], tabs["cdf_length"], tabs["offset"])
    sym, idx = _rand_symbols(tabs, 4000, 3, 60)
    stream = native.rans_encode(sym, idx, T)
    assert len(stream) % 4 == 0 and len(stream) >= 8
    assert stream == _PyRans.encode(sym.tolist(), idx.tolist(), tabs["quantized_cdf"], tabs["cdf_length"],
                                    tabs["offset"])
    assert np.array_equal(native.rans_decode(stream, idx, T), sym)
    # stateful per-block decode (NET:439) consumes exactly the stream
    d = native.RansDecoder()
    d.set_stream(stream)
    out = np.concatenate([d.decode_stream(idx[i:i + 96], T) for i in range(0, 4000, 96)])
    assert np.array_equal(out, sym)
    assert d.consumed() == len(stream)


def test_rans_empty_and_single():
    tabs = load_tables()
    T = native.Tables(tabs["quantized_cdf"], tabs["cdf_length"], tabs["offset"])
    s = native.rans_encode(np.zeros(0, np.int32), np.zeros(0, np.int32), T)
    assert s == np.array([1 << 31, 0], dtype=np.uint32).tobytes()     # flush of the initial state only
    for v in (0, -1, 5, -2000, 2000):
        st = native.rans_encode(np.array([v], np.int32), np.array([0], np.int32), T)
        assert native.rans_decode(st, np.array([0], np.int32), T)[0] == v


def test_layout_definition_roundtrip():
    img = torch.rand(2, 3, 16, 24)
    y = nets.arrange_block_pixels_to_channel_dim(img, 8)
    assert y.shape == (2, 192, 2, 3)
    assert y[1, (3 * 8 + 5) * 3 + 2, 1, 2] == img[1, 2, 8 + 3, 16 + 5]      # channel = (v*B+h)*C + c
    assert torch.equal(nets.arrange_channel_dim_to_block_pixels(y, 8), img)


@pytest.mark.needs_reference
def test_oracle_equals_reference_live():
    """Runs the unmodified reference through the import shim on a fresh input (skipped where
    LBIC_REFERENCE_ROOT does not name a checkout of the reference)."""
    from oracle.ref_shim import load_reference
    if not load_reference.available():
        pytest.skip("reference tree not present (LBIC_REFERENCE_ROOT)")
    ref = load_reference.load()
    cfg = lbic_b200.load_config("B8_lowrate")
    sd = weights.synth_state_dict(cfg, 99)
    m = ref.BlockBasedImgCompLossyNetv9(cfg).eval()
    m.load_state_dict(sd, strict=False)
    m.update(force=True)
    img = weights.synth_images(1, 24, 32, seed0=5)
    x = nets.arrange_block_pixels_to_channel_dim(img - 0.5, 8)
    with torch.no_grad():
        stream, zhat = m.compress(x, [1, 1, 1], cfg.M)
    g = m.conditional_gaussian_model
    P = nets.effective_params(sd, cfg)
    ostream, ozhat, _, _ = nets.compress(P, (g.quantized_cdf, g.cdf_length, g.offset), x)
    assert ostream == stream and torch.equal(ozhat, zhat)
    # and the synthetic state_dict carries exactly the reference's key set / shapes
    ref_sd = m.state_dict()
    assert list(ref_sd.keys()) == list(sd.keys())
    for k in sd:
        if not k.startswith("conditional_gaussian_model._") and "scale_table" not in k:
            assert tuple(ref_sd[k].shape) == tuple(sd[k].shape), k


@pytest.mark.needs_reference
def test_validation_loop_equals_reference_forward_loop():
    """validate_recu_reco_fast (AGENT:491-549) run with the UNMODIFIED reference model vs the oracle's codec loop +
    self_information, KS3111 (for KS[1]=1 the forward() windows and the codec-path windows coincide, SURVEY.md A.6)."""
    from oracle.ref_shim import load_reference
    if not load_reference.available():
        pytest.skip("reference tree not present (LBIC_REFERENCE_ROOT)")
    ref = load_reference.load()
    cfg = lbic_b200.load_config("B8_lowrate")
    sd = weights.synth_state_dict(cfg, 5)
    m = ref.BlockBasedImgCompLossyNetv9(cfg).eval()
    m.load_state_dict(sd, strict=False)
    img = weights.synth_images(1, 32, 40, seed0=9)
    x = nets.arrange_block_pixels_to_channel_dim(img - 0.5, 8)
    bt, ch, hg, wd = x.shape
    L = R = U = 1                                                    # get_lru_(KS, 'validation') for [3,1,1,1]
    zhat = torch.zeros_like(x)
    infos = torch.zeros(bt, cfg.M, hg, wd)
    with torch.no_grad():
        for v in range(hg):
            for h in range(wd):
                LL, RR, UU = max(0, h - L), min(wd, h + R + 1), max(0, v - U)
                xh, si = m(zhat[:, :, UU:v + 1, LL:RR], x[:, :, UU:v + 1, LL:RR])
                infos[:, :, v, h] = si[:, :, v - UU, h - LL]
                zhat[:, :, v, h] = xh[:, :, v - UU, h - LL].clamp_(-0.5, 0.5)
    P = nets.effective_params(sd, cfg)
    syms, idxs, ozhat = nets.compress_loop(P, x)
    assert float((ozhat - zhat).abs().max()) < 1e-5
    _, _, _, _, ksi = nets.whole_image_eval(P, x, ozhat)
    want = nets.self_information(syms.permute(2, 0, 1)[None], ksi[:, :cfg.M])
    assert float((want - infos).abs().max()) < 1e-3 * float(infos.abs().max())
