"""GPU parity tests (run with -m gpu on a B200): the CUDA path through the C ABI against the oracle
and the committed golden vectors produced by the reference itself (tests/golden/make_golden.py).

Bar: integer work (symbols, indexes, rANS bytes, CDF tables given identical inputs) bit-exact;
floating point: symbols identical on >= 99.99 % of positions, zhat within 1e-4 (tolerances stated at
each assert)."""
import os

import numpy as np
import pytest
import torch

import lbic_b200
from lbic_b200 import weights
from lbic_b200.net import BlockBasedImgCompLossyNetv9, get_lru
from oracle import native as onative
from conftest import GOLDEN, golden_cases, load_case, load_tables

pytestmark = pytest.mark.gpu

KS3111_CASES = golden_cases()   # all four reference topologies (KS3111 and KS3311)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


_models = {}


def get_model(cfgname, seed, harsh, dev, core="tcgen05"):
    key = (cfgname, seed, harsh)
    if key not in _models:
        cfg = lbic_b200.load_config(cfgname)
        m = BlockBasedImgCompLossyNetv9(cfg, device=dev)
        m.load_state_dict(weights.synth_state_dict(cfg, seed, harsh=harsh))
        assert m.update(force=True) is True
        _models[key] = m
    m = _models[key]
    m.set_gemm_core(core)
    return m


# Worst distance of a teacher-forced mismatch from its rounding boundary.  The arithmetic noise of y - mean on the B200
# path is the tensor cores' truncating fp32 accumulation (profiles/r2_gemm_precision.md: 2-3.5e-6 relative at K = 576-960,
# 1.4e-5 at K = 3840, growing linearly with K; the hi/lo operand split itself contributes 6e-8).  Measured worst distances
# over 36 full-size images (profiles/r2_parity_sweep.jsonl): 8.8e-5 for the B8 / B4 topologies, 1.7e-4 for B16 (first
# layers with K = 3840).  The bars are ~2-3x those, an order of magnitude below a 1e-3 arithmetic bug.
TF_BOUNDARY_TOL = 2e-4
TF_BOUNDARY_TOL_BY_CONFIG = {"B16_lowrate": 5e-4}


def tf_tol(cfgname):
    return TF_BOUNDARY_TOL_BY_CONFIG.get(str(cfgname), TF_BOUNDARY_TOL)


def tf_boundary_report(s2, i2, y2, ksi2, sym_c, idx_c, scale_table):
    """EVERY teacher-forced mismatch (oracle evaluation on the GPU's own zhat vs the GPU's symbols / indexes) must be a
    rounding-boundary case: the oracle's y - mean within TF_BOUNDARY_TOL of a .5 boundary AND the two symbols adjacent
    integers; for an index, the oracle's scale within TF_BOUNDARY_TOL (relative) of a scale-table threshold.
    Returns the worst distances over all mismatching positions."""
    M = sym_c.shape[-1]
    d = (y2 - ksi2[:, M:]).permute(0, 2, 3, 1)                               # (n,Hb,Wb,M) like the symbols
    frac = (d - torch.floor(d) - 0.5).abs()
    smis = s2 != sym_c
    sc = torch.clamp(ksi2[:, :M], min=0.11).permute(0, 2, 3, 1)
    rel = ((sc[..., None] - scale_table) .abs() / scale_table).min(dim=-1).values
    imis = i2 != idx_c
    return dict(tf_worst_symbol_boundary_distance=float(frac[smis].max()) if bool(smis.any()) else 0.0,
                tf_worst_symbol_step=int((s2 - sym_c).abs().max()),
                tf_worst_index_boundary_distance=float(rel[imis].max()) if bool(imis.any()) else 0.0,
                tf_worst_index_step=int((i2 - idx_c).abs().max()))


def assert_tf_boundary(rep, tol=TF_BOUNDARY_TOL):
    assert rep["tf_worst_symbol_boundary_distance"] < tol and rep["tf_worst_symbol_step"] <= 1, rep
    assert rep["tf_worst_index_boundary_distance"] < tol and rep["tf_worst_index_step"] <= 1, rep


def closed_loop_report(cfgname, seed, harsh, x, sym, idx, zhat, ref_sym, ref_idx):
    """Compares a GPU closed-loop result with the reference's.

    The reference loop is a DPCM-style feedback system: ONE symbol that rounds the other way (y - mean within fp noise
    of a .5 boundary) changes that block's reconstruction by a quantisation step and every later block then sees
    different inputs, so two implementations that are not bit-identical in summation order agree exactly up to the
    first such flip and diverge afterwards (the reference's own fp32 ops in a different accumulation order show the
    same, tests/golden/make_golden_full.py).  The well-posed checks are therefore:
      * teacher-forced agreement: one oracle (torch CPU fp32) evaluation on the GPU's final zhat must reproduce the
        GPU's symbols / indexes on >= 99.99 % of positions (fixed point, SURVEY.md fact 10);
      * the FIRST closed-loop mismatch (raster order), if any, must be a rounding-boundary case."""
    from oracle import nets
    cfg = lbic_b200.load_config(cfgname)
    P = nets.effective_params(weights.synth_state_dict(cfg, seed, harsh=harsh), cfg)
    s2, i2, xh2, y2, ksi2 = nets.whole_image_eval(P, x.cpu(), zhat.cpu())
    sym_c, idx_c = sym.cpu(), idx.cpu().int()
    n = sym_c.numel()
    rep = dict(symbols=n, tf_symbol_mismatches=int((s2 != sym_c).sum()), tf_index_mismatches=int((i2 != idx_c).sum()),
               closed_loop_symbol_mismatches=int((sym_c != ref_sym).sum()),
               closed_loop_index_mismatches=int((idx_c != ref_idx).sum()), first_mismatch=None)
    rep.update(tf_boundary_report(s2, i2, y2, ksi2, sym_c, idx_c, P.scale_table))
    bad = ((sym_c != ref_sym) | (idx_c != ref_idx))
    if bool(bad.any()):
        M = sym_c.shape[-1]
        flat = bad.reshape(bad.shape[0], -1, M)
        img = int(flat.any(dim=-1).any(dim=-1).float().argmax())
        blk = int(flat[img].any(dim=-1).float().argmax())              # first block in raster order
        Hb, Wb = sym_c.shape[1], sym_c.shape[2]
        v, h = blk // Wb, blk % Wb
        ch = torch.nonzero(flat[img, blk]).flatten().tolist()
        d = (y2[img, :, v, h] - ksi2[img, M:, v, h])
        frac = (d - torch.floor(d) - 0.5).abs()                         # distance of y - mean from a .5 boundary
        sc = torch.clamp(ksi2[img, :M, v, h], min=0.11)
        tab = P.scale_table
        rel = ((sc[:, None] - tab[None, :]).abs() / tab[None, :]).min(dim=1).values   # distance from a scale threshold
        rep["first_mismatch"] = dict(image=img, block=[v, h], channels=ch[:8],
                                     boundary_distance=[float(min(frac[c], rel[c])) for c in ch[:8]])
    return rep


@pytest.mark.parametrize("core", ["simt", "tcgen05"])
@pytest.mark.parametrize("shape", [(128, 64, 256), (200, 960, 768), (77, 96, 96), (300, 864, 672), (129, 200, 48)])
def test_gemm_core_vs_fp64(dev, core, shape):
    """D = A W^T from bf16 hi/lo split operands; tolerance 3e-5 relative to |A||W| row norms
    (the dropped lo*lo term and fp32 accumulation; plain bf16 would be ~4e-3)."""
    R, K, C = shape
    m = get_model("B8_lowrate", 1337, False, dev, core)
    g = torch.Generator().manual_seed(R * 1000 + K)
    A = torch.randn(R, K, generator=g).to(dev)
    W = (torch.randn(C, K, generator=g) / K ** 0.5).to(dev)
    D = m.debug_gemm(A, W)
    ref = (A.double() @ W.double().T)
    scale = (A.double().abs() @ W.double().abs().T)
    err = ((D.double() - ref).abs() / scale).max().item()
    assert err < 3e-5, f"{core} gemm {shape}: scaled error {err:.3e}"


def test_tables_match_reference(dev):
    """K4: tables built on the GPU vs the reference's update() output (golden)."""
    m = get_model("B8_lowrate", 1337, False, dev)
    g, ref = m.conditional_gaussian_model, load_tables()
    assert np.array_equal(g.cdf_length.numpy(), ref["cdf_length"])
    assert np.array_equal(g.offset.numpy(), ref["offset"])
    cdf = g.quantized_cdf.numpy()
    assert cdf.shape == ref["quantized_cdf"].shape
    ndiff = int((cdf != ref["quantized_cdf"]).sum())
    # structural invariants regardless of erfc rounding: strictly increasing to 2^16
    for i in range(64):
        row = cdf[i, : g.cdf_length[i]]
        assert row[0] == 0 and row[-1] == 65536 and (np.diff(row) > 0).all()
    assert ndiff == 0, f"{ndiff} CDF entries differ from the reference table"


def _rand_symbols(tabs, n, seed, escapes=True):
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, 64, size=n).astype(np.uint8)
    scale = tabs["scale_table"][idx]
    sym = np.rint(rng.normal(0, 1, size=n) * scale).astype(np.int32)
    if escapes:
        pos = rng.integers(0, n, size=max(4, n // 50))
        sym[pos] += rng.integers(-40000, 40000, size=pos.size).astype(np.int32)
    return sym, idx


@pytest.mark.parametrize("n_streams,n_sym,thread_form", [(1, 5000, 0), (7, 1234, 0), (64, 96, 0), (7, 1236, 1),
                                                         (300, 96, 1)])
def test_rans_bit_exact_vs_oracle(dev, n_streams, n_sym, thread_form):
    """K5/K6: GPU rANS bytes == oracle bytes for identical symbols/indexes/tables; GPU decode inverts.
    thread_form forces the thread-per-stream encoder (the default for >= 4096 streams)."""
    m = get_model("B8_lowrate", 1337, False, dev)
    m.set_option("enc_thread_streams", 1 if thread_form else 1 << 30)
    tabs = load_tables()
    g = m.conditional_gaussian_model
    T = onative.Tables(g.quantized_cdf.numpy(), g.cdf_length.numpy(), g.offset.numpy())
    sym, idx = _rand_symbols(tabs, n_streams * n_sym, 11 + n_streams)
    sym_d = torch.from_numpy(sym).to(dev)
    idx_d = torch.from_numpy(idx).to(dev)
    cap = 8 * n_sym + 64
    out = torch.zeros(n_streams, cap, dtype=torch.uint8, device=dev)
    lens = torch.zeros(n_streams, dtype=torch.int32, device=dev)
    from lbic_b200 import _lib
    _lib.check(_lib.lib().lbic_rans_encode(m._need(), sym_d.data_ptr(), idx_d.data_ptr(), n_streams, n_sym,
                                           out.data_ptr(), cap, lens.data_ptr(), None))
    torch.cuda.synchronize()
    lens_h, out_h = lens.cpu().numpy(), out.cpu().numpy()
    for s in range(n_streams):
        want = onative.rans_encode(sym[s * n_sym:(s + 1) * n_sym], idx[s * n_sym:(s + 1) * n_sym], T)
        got = out_h[s, : lens_h[s]].tobytes()
        assert got == want, f"stream {s}: GPU rANS bytes differ from the oracle ({len(got)} vs {len(want)})"
    dec = torch.zeros(n_streams * n_sym, dtype=torch.int32, device=dev)
    _lib.check(_lib.lib().lbic_rans_decode(m._need(), out.data_ptr(), lens.data_ptr(), cap, idx_d.data_ptr(),
                                           n_streams, n_sym, dec.data_ptr(), None))
    torch.cuda.synchronize()
    m.set_option("enc_thread_streams", 4096)
    assert np.array_equal(dec.cpu().numpy(), sym)


@pytest.mark.parametrize("core", ["simt", "tcgen05"])
@pytest.mark.parametrize("case", KS3111_CASES)
def test_encode_matches_reference_golden(dev, case, core):
    """compress() vs the reference's own output: symbols/indexes >= 99.99 % identical (here: all of them,
    the grids are small), zhat within 1e-4, and - symbols being identical - the bitstream bit-exact."""
    c = load_case(case)
    m = get_model(str(c["config"]), int(c["seed"]), bool(c["harsh"]), dev, core)
    x = torch.from_numpy(c["x"]).to(dev)
    strings, zhat, sym, idx = m.compress_batch(x, lanes=1, return_symbols=True)
    ref_sym = torch.from_numpy(c["symbols"].astype(np.int32))[None]
    ref_idx = torch.from_numpy(c["indexes"].astype(np.int32))[None]
    rep = closed_loop_report(str(c["config"]), int(c["seed"]), bool(c["harsh"]), x, sym, idx, zhat, ref_sym, ref_idx)
    n = rep["symbols"]
    assert rep["tf_symbol_mismatches"] <= max(1, n // 10000) and rep["tf_index_mismatches"] <= max(1, n // 10000), rep
    tol = 1e-3 if bool(c["harsh"]) else tf_tol(c["config"])
    assert_tf_boundary(rep, tol)
    mism = rep["closed_loop_symbol_mismatches"] + rep["closed_loop_index_mismatches"]
    if mism:
        # accumulation-order noise is ~1e-5 here; anything that is not a boundary case is a real bug
        assert max(rep["first_mismatch"]["boundary_distance"]) < tol, rep
    zref = torch.from_numpy(c["zhat"])
    xh = torch.from_numpy(c["x"])
    psnr = lambda z: -10.0 * float(torch.log10(((xh - z) ** 2).mean()))
    assert abs(psnr(zhat.cpu()) - psnr(zref)) < 0.01, "PSNR delta vs reference exceeds 0.01 dB"
    assert abs(len(strings[0]) - c["stream"].size) <= max(8, c["stream"].size // 200), "bitstream size differs > 0.5 %"
    if mism == 0:
        zerr = float((zhat.cpu() - zref).abs().max())
        # fp32 accumulation-order noise: ~1e-5 normally; the "harsh" weights (decoder input at full scale, 86 % of
        # samples clamped) amplify it to ~3e-4 even for plain fp32 FFMA (the SIMT twin), hence 1e-3 there.
        assert zerr < (1e-3 if bool(c["harsh"]) else 1e-4), f"{case}/{core}: zhat max abs diff {zerr:.2e}"
    tabs_equal = np.array_equal(m.conditional_gaussian_model.quantized_cdf.numpy(), load_tables()["quantized_cdf"])
    if tabs_equal and mism == 0:
        assert strings[0] == c["stream"].tobytes(), "bitstream differs from the reference for identical symbols"
    # single-image reference-surface call
    L = list(get_lru(m.KS))
    s1, z1 = m.compress(x, L, m.M)
    assert s1 == strings[0] and torch.equal(z1, zhat)


@pytest.mark.parametrize("lanes", [1, 0])
@pytest.mark.parametrize("case", KS3111_CASES)
def test_decode_roundtrip(dev, case, lanes):
    """decompress(compress(x)) reproduces the encoder's zhat exactly (the reference's own check,
    AGENT:601-602: Enc-Dec.Mad/Max/Min == 0), for the reference container and the lane container."""
    c = load_case(case)
    m = get_model(str(c["config"]), int(c["seed"]), bool(c["harsh"]), dev)
    x = torch.from_numpy(c["x"]).to(dev)
    strings, zhat = m.compress_batch(x, lanes=lanes)
    zdec = m.decompress_batch(strings, x.shape, lanes=lanes)
    assert torch.equal(zdec, zhat), f"enc/dec mismatch {float((zdec - zhat).abs().max()):.3e}"
    if lanes == 1:
        # and the reference's bitstream decodes to the reference's reconstruction
        zref = m.decompress(c["stream"].tobytes(), list(get_lru(m.KS)), x.shape, m.M, dev)
        tol = 1e-3 if bool(c["harsh"]) else 1e-4   # see test_encode_matches_reference_golden
        assert float((zref.cpu() - torch.from_numpy(c["zhat_dec"])).abs().max()) < tol


@pytest.mark.parametrize("cfgname", ["B8_lowrate", "B4_highrate", "B16_lowrate", "B8_highrate"])
def test_thread_per_stream_decode_equals_warp_per_stream(dev, cfgname):
    """rans_dec_step_thread_kernel (one stream per thread, compact CDFs + bucket table in shared memory) must decode
    exactly what the warp-per-stream kernel decodes, for the lane container and the reference container; the harsh
    weights make escape (bypass) symbols occur."""
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    for harsh in (False, True):
        m = get_model(cfgname, 1337, harsh, dev)
        B = m.B
        img = weights.synth_images(40, 5 * B, 9 * B, seed0=311, kind="noise" if harsh else "smooth")
        x = arrange_block_pixels_to_channel_dim((img - 0.5).to(dev), B)
        try:
            m.set_option("wave", 0)
            for lanes in (0, 1):
                strings, zhat, sym, _ = m.compress_batch(x, lanes=lanes, return_symbols=True)
                out = {}
                # never / always the thread-per-stream kernels (decoder and encoder); the warp-per-row decode step on the
                # int32 tables in global memory (key 2) and on shared-memory copies of the compact rows (the default)
                for rows in (1 << 30, 1, 2):
                    m.set_option("dec_smem_warp", 0 if rows == 2 else 1)
                    rows = (1 << 30) if rows == 2 else rows
                    m.set_option("dec_thread_rows", rows)
                    m.set_option("enc_thread_streams", rows)
                    enc_dev = m.encode_device(x, lanes=lanes)
                    got = m._gather_streams(enc_dev)
                    assert got == strings, "bitstreams differ between the two encoder kernels"
                    z, s = m.decode_device(enc_dev.streams, enc_dev.lens, x.shape[0], x.shape[2], x.shape[3], lanes=lanes,
                                           want_symbols=True)
                    if rows == (1 << 30) and (1 << 30) in out:
                        assert torch.equal(out[rows][1], s) and torch.equal(out[rows][0], z), \
                            "warp-per-row decode differs between shared-memory and global-memory tables"
                    out[rows] = (z, s)
                assert torch.equal(out[1][1], out[1 << 30][1]), "symbols differ between the two decode kernels"
                assert torch.equal(out[1][0], out[1 << 30][0])
                assert torch.equal(out[1][1], sym) and torch.equal(out[1][0], zhat)
        finally:
            m.set_option("dec_thread_rows", 4096)
            m.set_option("enc_thread_streams", 4096)
            m.set_option("dec_smem_warp", 1)
            m.set_option("wave", 1)


def test_batch_invariance_and_ragged_grids(dev):
    """A block's result must not depend on batch size / tile placement: encode 5 images together and one
    by one; odd grids (1xW, Hx1, 1x1) exercise the wavefront edges."""
    m = get_model("B8_lowrate", 1337, False, dev)
    B = m.B
    for Hb, Wb, n in [(3, 5, 5), (1, 7, 2), (6, 1, 3), (1, 1, 1), (4, 4, 1)]:
        img = weights.synth_images(n, Hb * B, Wb * B, seed0=50 + Hb)
        from lbic_b200.layout import arrange_block_pixels_to_channel_dim
        x = arrange_block_pixels_to_channel_dim((img - 0.5).to(dev), B)
        strings, zhat, sym, idx = m.compress_batch(x, return_symbols=True)
        for i in range(n):
            s1, z1, sy1, id1 = m.compress_batch(x[i:i + 1], return_symbols=True)
            assert torch.equal(sy1[0], sym[i]) and torch.equal(id1[0], idx[i]) and torch.equal(z1[0], zhat[i])
            assert s1[0] == strings[i]
        zdec = m.decompress_batch(strings, x.shape)
        assert torch.equal(zdec, zhat)


@pytest.mark.parametrize("cfgname,n,Hb,Wb", [("B8_lowrate", 1, 7, 11), ("B8_lowrate", 1, 40, 70), ("B8_lowrate", 6, 9, 13),
                                             ("B8_lowrate", 5, 30, 64), ("B16_lowrate", 3, 5, 9), ("B8_lowrate", 2, 1, 5),
                                             ("B8_lowrate", 1, 6, 1),
                                             # KS3311 (five-tap second entropy layer): extended steps, g0 store, gather5 tiles
                                             ("B8_highrate", 1, 7, 11), ("B4_highrate", 1, 20, 33), ("B8_highrate", 3, 9, 13),
                                             ("B4_highrate", 1, 1, 6), ("B8_highrate", 1, 5, 1), ("B8_highrate", 1, 64, 96)])
def test_wave_kernel_equals_per_layer_launches(dev, cfgname, n, Hb, Wb):
    """gemm_wave_kernel (a whole encode / decode of small steps in ONE persistent cooperative launch: gather, every layer
    and the rANS decode step as tiles of an in-kernel list, 128 x 32 tiles, cross-step dependencies through monotonic
    counters) must be bit-identical to one launch per layer: symbols, indexes, reconstruction, bytes, for the lane and
    the reference container, one and several 128-row blocks per step (5 x 30 rows = 150), degenerate grids; and through
    the host calls, whose band hooks cut the launch into several."""
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    m = get_model(cfgname, 1337, False, dev)
    B = m.B
    img = weights.synth_images(n, Hb * B, Wb * B, seed0=131)
    x = arrange_block_pixels_to_channel_dim((img - 0.5).to(dev), B)
    try:
        m.set_option("wave_dec_max_rows", 4096)          # (default 64: beyond that the per-layer decode is faster)
        for lanes in (0, 1):
            m.set_option("wave", 0)
            ref = m.compress_batch(x, lanes=lanes, return_symbols=True)
            zref = m.decompress_batch(ref[0], x.shape, lanes=lanes)
            m.set_option("wave", 1)
            for bn in (0, 64, 128):                      # tile width: automatic (64 / 128 by rows), narrowest, widest
                m.set_option("wave_bn", bn)
                l0 = m.launch_count()
                got = m.compress_batch(x, lanes=lanes, return_symbols=True)
                if not (m.KS[1] == 3 and Wb < 2):         # (one-column KS3311 grids stay on the per-layer path)
                    assert m.launch_count() - l0 < 20, "the wave path should need a handful of launches per encode"
                assert torch.equal(got[2], ref[2]), f"symbols differ (lanes={lanes}, bn={bn})"
                assert torch.equal(got[3], ref[3]) and torch.equal(got[1], ref[1])
                assert got[0] == ref[0], f"bitstreams differ (lanes={lanes}, bn={bn})"
                o = m.encode_device(x, lanes=lanes)
                l0 = m.launch_count()
                zdec, sdec = m.decode_device(o.streams, o.lens, n, Hb, Wb, lanes=lanes, want_symbols=True)
                if not (m.KS[1] == 3 and (lanes == 1 or Wb < 2)):   # (KS3311 has no raster mode in the wave kernel)
                    assert m.launch_count() - l0 < 20, "the wave path should need a handful of launches per decode"
                assert torch.equal(sdec, ref[2]), f"decoded symbols differ (lanes={lanes}, bn={bn})"
                assert torch.equal(zdec, zref) and torch.equal(zdec, got[1])
            m.set_option("wave_bn", 0)
        # host calls: the band hooks cut the wave launch; 8-bit entry points on the same images
        imgs_u8 = (img * 255).round().to(torch.uint8).numpy()
        m.set_option("wave", 0)
        want_s, want_rec = m.compress_images_u8(imgs_u8, lanes=0, return_recon=True)
        m.set_option("wave", 1)
        for bands in (16, 3):
            m.set_option("host_bands", bands)
            got_s, got_rec = m.compress_images_u8(imgs_u8, lanes=0, return_recon=True)
            assert got_s == want_s and np.array_equal(got_rec, want_rec)
            assert np.array_equal(m.decompress_images_u8(got_s, Hb * B, Wb * B, lanes=0), want_rec)
    finally:
        m.set_option("wave", 1)
        m.set_option("wave_bn", 0)
        m.set_option("wave_dec_max_rows", 64)
        m.set_option("host_bands", 16)


@pytest.mark.parametrize("cfgname", ["B8_lowrate", "B4_highrate", "B16_lowrate", "B8_highrate"])
def test_warp_specialised_kernel_equals_per_tile_kernel(dev, cfgname):
    """gemm_ws_kernel (persistent, overlapped epilogue, 192-wide tiles), in its single-CTA and CTA-pair (cta_group::2,
    256-row tiles) forms, must be bit-identical to gemm_tc_kernel."""
    m = get_model(cfgname, 1337, False, dev)
    B = m.B
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    img = weights.synth_images(24, 6 * B, 13 * B, seed0=91)
    x = arrange_block_pixels_to_channel_dim((img - 0.5).to(dev), B)
    try:
        m.set_option("wave", 0)
        m.set_option("ws", 0)
        ref = m.compress_batch(x, lanes=0, return_symbols=True)
        for pair in (0, 1):
            m.set_option("ws", 2)
            m.set_option("pair", pair)
            got = m.compress_batch(x, lanes=0, return_symbols=True)
            assert got[0] == ref[0], f"bitstreams differ (pair={pair})"
            assert torch.equal(got[1], ref[1]) and torch.equal(got[2], ref[2]) and torch.equal(got[3], ref[3])
            zdec = m.decompress_batch(got[0], x.shape, lanes=0)
            assert torch.equal(zdec, got[1])
    finally:
        m.set_option("ws", 1)
        m.set_option("pair", 1)
        m.set_option("wave", 1)


@pytest.mark.parametrize("cfgname", ["B8_lowrate", "B4_highrate", "B16_lowrate", "B8_highrate"])
def test_dataflow_launch_equals_per_layer_launches(dev, cfgname):
    """gemm_flow_kernel (all layers of a step in one launch, row-block dependency counters instead of kernel boundaries)
    must be bit-identical to one launch per layer, encode and decode, including ragged last row blocks."""
    m = get_model(cfgname, 1337, False, dev)
    B = m.B
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    img = weights.synth_images(37, 7 * B, 12 * B, seed0=57)
    x = arrange_block_pixels_to_channel_dim((img - 0.5).to(dev), B)
    try:
        m.set_option("wave", 0)
        m.set_option("flow", 0)
        ref = m.compress_batch(x, lanes=0, return_symbols=True)
        zref = m.decompress_batch(ref[0], x.shape, lanes=0)
        m.set_option("flow", 2)
        for tma_store in (1, 0):     # TMA stores from swizzled staging planes / staged copy loops (the default)
            m.set_option("tma_store", tma_store)
            got = m.compress_batch(x, lanes=0, return_symbols=True)
            assert got[0] == ref[0], f"bitstreams differ (tma_store={tma_store})"
            assert torch.equal(got[1], ref[1]) and torch.equal(got[2], ref[2]) and torch.equal(got[3], ref[3])
            zdec = m.decompress_batch(got[0], x.shape, lanes=0)
            assert torch.equal(zdec, zref) and torch.equal(zdec, got[1])
        zv, iv = m.validate_recu_reco(x)
        assert torch.equal(zv, got[1])
        # the quad form: clusters of four CTAs, two pairs on adjacent column tiles sharing the activation operand by
        # TMA multicast (layers with an odd number of column tiles give the second pair a dummy tile)
        m.set_option("flow_quad", 1)
        l0 = m.launch_count()
        quad = m.compress_batch(x, lanes=0, return_symbols=True)
        assert quad[0] == ref[0], "bitstreams differ (quad form)"
        assert torch.equal(quad[1], ref[1]) and torch.equal(quad[2], ref[2]) and torch.equal(quad[3], ref[3])
        assert torch.equal(m.decompress_batch(quad[0], x.shape, lanes=0), zref)
        m.set_option("flow_quad", 0)
        # the single-CTA form for small steps (128 x 96 tiles, off by default)
        m.set_option("flow", 1)
        m.set_option("flow_small", 1)
        small = m.compress_batch(x, lanes=0, return_symbols=True)
        assert small[0] == ref[0] and torch.equal(small[1], ref[1]) and torch.equal(small[2], ref[2])
        assert torch.equal(m.decompress_batch(small[0], x.shape, lanes=0), zref)
    finally:
        m.set_option("flow", 1)
        m.set_option("flow_small", 0)
        m.set_option("flow_quad", 0)
        m.set_option("tma_store", 0)
        m.set_option("wave", 1)


# BASELINE.json configs at their own sizes: C1 (B8_lowrate 768x512), C2 (B4_highrate 768x512, batch of 24),
# C3 (B8_highrate 768x512, enough images that the persistent / CTA-pair / dataflow kernels engage: 96 images x 48 rows
# = 4608-row steps), C4 (B16_lowrate 2048x2048).  The oracle checks the first `n_chk` images; encode -> decode covers all.
@pytest.mark.parametrize("cfgname,H,W,n_img,n_chk", [("B8_lowrate", 512, 768, 2, 2), ("B4_highrate", 512, 768, 24, 2),
                                                     ("B8_highrate", 512, 768, 96, 2), ("B16_lowrate", 2048, 2048, 1, 1),
                                                     ("B4_highrate", 128, 192, 2, 2), ("B16_lowrate", 256, 256, 2, 2)])
def test_full_size_fixed_point_vs_oracle(dev, cfgname, H, W, n_img, n_chk):
    """BASELINE-size check through a size-independent property (SURVEY.md fact 10 / A.6): the closed-loop result is
    the unique fixed point of the open-loop network, so ONE parallel oracle evaluation (torch CPU fp32) on the GPU's
    final zhat must reproduce the GPU's symbols (>= 99.99 %), indexes and reconstruction; and decode(encode) == zhat."""
    import json, os
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    from oracle import nets
    cfg = lbic_b200.load_config(cfgname)
    m = get_model(cfgname, 1337, False, dev)
    B = m.B
    img = weights.synth_images(n_img, H, W, seed0=1000)
    x = arrange_block_pixels_to_channel_dim((img - 0.5).to(dev), B)
    lanes = 1 if n_img <= 2 else 0          # the raster-serial reference container on the small batches only
    strings, zhat, sym, idx = m.compress_batch(x, lanes=lanes, return_symbols=True)
    P = nets.effective_params(weights.synth_state_dict(cfg, 1337), cfg)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    xc, zc, sc, ic = x[:n_chk].cpu(), zhat[:n_chk].cpu(), sym[:n_chk].cpu(), idx[:n_chk].cpu().int()
    s2, i2, xh2, y2, ksi2 = nets.whole_image_eval(P, xc, zc)
    n = sc.numel()
    sym_mis = int((s2 != sc).sum())
    idx_mis = int((i2 != ic).sum())
    brep = tf_boundary_report(s2, i2, y2, ksi2, sc, ic, P.scale_table)
    # compare reconstructions only on blocks whose symbols agree (a +-1 symbol flip legitimately moves its block)
    same_blk = ((s2 == sc).all(dim=-1)).unsqueeze(1)                              # (n,1,Hb,Wb)
    zerr = float(((xh2 - zc).abs() * same_blk).max())
    print(json.dumps(dict(config=cfgname, H=H, W=W, images=n_img, images_checked=n_chk, symbols=n, symbol_mismatches=sym_mis,
                          index_mismatches=idx_mis, zhat_maxdiff=zerr, sym_std=float(sym.float().std()),
                          sym_absmax=int(sym.abs().max()), bytes=[len(s) for s in strings[:4]], **brep)))   # shown with -rP
    assert sym_mis <= n // 10000, f"{sym_mis} of {n} symbols differ from the oracle fixed point (> 0.01 %)"
    assert idx_mis <= n // 10000, f"{idx_mis} of {n} indexes differ"
    assert_tf_boundary(brep, tf_tol(cfgname))
    assert zerr < 5e-4, f"zhat differs from the oracle fixed point by {zerr:.2e}"
    zdec = m.decompress_batch(strings, x.shape, lanes=lanes)
    assert torch.equal(zdec, zhat)
    if lanes != 1:
        return
    # bit-exact entropy stage for the GPU's own symbols, against the oracle coder
    g = m.conditional_gaussian_model
    T = onative.Tables(g.quantized_cdf.numpy(), g.cdf_length.numpy(), g.offset.numpy())
    want = onative.rans_encode(sym[0].cpu().numpy().reshape(-1), idx[0].cpu().numpy().reshape(-1), T)
    assert strings[0] == want


@pytest.mark.parametrize("cfgname,gw,gh", [("B8_lowrate", 768, 512), ("B8_highrate", 768, 512), ("B4_highrate", 768, 512),
                                           ("B16_lowrate", 2048, 2048)])
def test_full_size_image_vs_reference_closed_loop(dev, cfgname, gw, gh):
    """The headline parity number: ONE full-size image per reference topology at the size BASELINE.json names for it
    (B8 KS3111 N768 M96 768x512: 589 824 symbols; B8 KS3311 N1152 M128: 786 432; B4 KS3311 N512 M96: 2 359 296;
    B16 KS3111 N1280 M192 2048x2048: 3 145 728) against the UNMODIFIED reference's closed loop
    (tests/golden/make_golden_full.py).

    north_star bar: symbols identical on >= 99.99 % of positions, bpp within 0.1 %, PSNR within 0.01 dB; if all symbols
    match, the bitstream must be byte-identical (sha256).  The symbol bar is only meaningful up to the first
    rounding-boundary flip: the UNMODIFIED reference itself, run with a permuted accumulation order or with ONE symbol
    forced the other way, differs from its own stock run on 0.1-1.2 % of the image
    (tests/golden/closed_loop_noise_B8_lowrate_768x512.json, make_closed_loop_noise.py).  So this test asserts
      * identity with the reference up to the first mismatch, which must be a boundary case (< TF_BOUNDARY_TOL);
      * EVERY teacher-forced mismatch over the whole image is a boundary case of one step (assert_tf_boundary) and
        there are <= 100 ppm of them;
      * after the first flip the fraction of differing symbols stays within what ONE forced flip produces in the
        reference itself (<= 3 %: the fixture's worst case is 1.2 %);
      * bpp / PSNR bars; decode(encode) exact."""
    import hashlib, json, os
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    path = os.path.join(os.path.dirname(__file__), "golden", f"full_{cfgname}_{gw}x{gh}.npz")
    if not os.path.exists(path):
        pytest.skip("full-size golden not generated")
    gold = np.load(path)
    m = get_model(cfgname, 1337, False, dev)
    H, W = int(gold["H"]), int(gold["W"])
    x_img = weights.u8_to_model_input(weights.synth_image_u8(H, W, int(gold["image_seed"])))
    x = arrange_block_pixels_to_channel_dim(x_img.to(dev), m.B)
    strings, zhat, sym, idx = m.compress_batch(x, lanes=1, return_symbols=True)
    ref_sym = torch.from_numpy(gold["symbols"].astype(np.int32))[None]
    ref_idx = torch.from_numpy(gold["indexes"].astype(np.int32))[None]
    rep = closed_loop_report(cfgname, 1337, False, x, sym, idx, zhat, ref_sym, ref_idx)
    n = rep["symbols"]
    psnr = -10.0 * float(torch.log10(((x - zhat) ** 2).mean()))
    bpp_rel = abs(len(strings[0]) - int(gold["stream_len"])) / int(gold["stream_len"])
    rep.update(bytes=len(strings[0]), ref_bytes=int(gold["stream_len"]), bpp_rel_diff=bpp_rel, psnr=psnr,
               ref_psnr=float(gold["psnr"]), reference_fp32_noise_floor_symbol_mismatches=int(gold["fp32_noise_symbol_mismatches"]),
               stream_identical=hashlib.sha256(strings[0]).hexdigest() == str(gold["stream_sha256"]))
    if rep["first_mismatch"]:
        v, h = rep["first_mismatch"]["block"]
        after = n - (v * sym.shape[2] + h) * sym.shape[3]
        rep["mismatches_after_first_fraction"] = rep["closed_loop_symbol_mismatches"] / max(1, after)
    print(json.dumps(rep))                                                      # shown with -rP
    assert rep["tf_symbol_mismatches"] <= n // 10000 and rep["tf_index_mismatches"] <= n // 10000, rep
    assert_tf_boundary(rep, tf_tol(cfgname))
    if rep["closed_loop_symbol_mismatches"] + rep["closed_loop_index_mismatches"]:
        assert max(rep["first_mismatch"]["boundary_distance"]) < tf_tol(cfgname), rep
        assert rep["mismatches_after_first_fraction"] < 0.03, rep
    else:
        assert rep["stream_identical"], "identical symbols but different bytes"
    assert bpp_rel < 1e-3, f"bpp differs by {100 * bpp_rel:.3f} %"
    assert abs(psnr - float(gold["psnr"])) < 0.01
    zdec = m.decompress_batch(strings, x.shape, lanes=1)
    assert torch.equal(zdec, zhat)


def test_eval_model_matches_reference_log_line(dev):
    """eval_model's per-image body (AGENT:578-637) on the image and weights of tests/golden/eval_model_*.json, which
    holds what the UNMODIFIED reference agent logged for them on the CPU (make_golden_eval_model.py): ToTensor, -0.5,
    padding, space-to-depth, compress, decompress, Enc-Dec check, bpp, MSE / PSNR.  Bars: bpp within 0.1 %, PSNR within
    0.01 dB, Enc-Dec.Mad/Max/Min = 0; the formatted log line must agree in every field but the timings."""
    import json, math
    from lbic_b200.codec import pad_to_blocks, ms_ssim
    gold = json.load(open(os.path.join(GOLDEN, "eval_model_B8_lowrate_208x176.json")))
    g = gold["record"]
    m = get_model(gold["config"], int(gold["weight_seed"]), False, dev)
    B, H, W = m.B, int(gold["H"]), int(gold["W"])
    img = weights.synth_image_u8(H, W, int(gold["image_seed"]))
    x = (torch.from_numpy(img).float().div(255)[None] - 0.5).to(dev)                       # ToTensor on the CPU, AGENT:581
    xp = lbic_b200.arrange_block_pixels_to_channel_dim(pad_to_blocks(x, B), B)              # AGENT:583-589
    L = list(get_lru(m.KS))
    bitstream, xhat_enc = m.compress(xp, L, m.M)                                            # AGENT:592
    xhat_dec = m.decompress(bitstream, L, xp.shape, m.M, dev)                               # AGENT:598
    dif = (xhat_enc - xhat_dec).abs()
    bpp = len(bitstream) * 8.0 / (H * W)                                                    # AGENT:608-609
    xhat_img = lbic_b200.arrange_channel_dim_to_block_pixels(xhat_enc, B)
    mse = float(torch.nn.functional.mse_loss(x, xhat_img))                                  # AGENT:611
    psnr = -10 * math.log10(mse)
    msssim = float(ms_ssim(x + 0.5, xhat_img + 0.5, data_range=1.0))
    assert float(dif.max()) == 0.0                                                          # Enc-Dec.Mad/Max/Min 0.00/0.00/0.00
    assert abs(len(bitstream) - g["bytes"]) <= g["bytes"] * 1e-3, (len(bitstream), g["bytes"])
    assert abs(psnr - (-10 * math.log10(g["mse_padded"]))) < 0.01
    line = ('RDLoss:{:.3f} MSE/PSNR:{:.5f}/{:.2f} Rate:{:.3f} MS-SSIM/dB:{:.6f}/{:.2f} Enc-Dec.Mad/Max/Min:{:.2f}/{:.2f}/{:.2f}'
            .format(bpp + 117.045 * mse, mse, psnr, bpp, msssim, -10 * math.log10(1.0 - msssim), float(dif.mean()) * 255,
                    float(dif.max()) * 255, float(dif.min()) * 255))
    import re
    want = re.sub(r"Enc/DecTime:[\d.]+/[\d.]+ ", "", gold["log_line"].split("--> ")[1].rsplit(" (", 1)[0])
    if len(bitstream) == g["bytes"]:
        # every field of the reference's line; MS-SSIM (a stand-in for pytorch_msssim on both sides, torch CPU there and
        # torch CUDA here) to 1e-5 instead of its sixth printed digit
        drop = lambda s: re.sub(r"MS-SSIM/dB:[\d.]+/", "MS-SSIM/dB:*/", s)
        assert drop(line) == drop(want), (line, want)
        assert abs(msssim - g["msssim"]) < 1e-5


@pytest.mark.parametrize("case", ["B8_lowrate_6x9", "B4_highrate_7x10", "B16_lowrate_3x5"])
def test_postprocessing_module_matches_reference_golden(dev, case):
    """SURVEY.md 8(f) rank 4: BlkBasedPostProcessing (NET:455-476).  tests/golden/postpm_<case>.npz holds the UNMODIFIED
    reference module's output on the case's closed-loop reconstruction (make_golden_postpm.py).  No feedback here, so the
    bar is plain fp32-grade accuracy: 2e-5 of the output range (8e-5 for B16, whose 3x3 layer contracts 6912 values); border blocks must be returned bit-exactly; the in-kernel
    clamp equals clamp_ of the unclamped result; larger batches / several raster chunks give the same numbers."""
    c = load_case(case)
    f = np.load(os.path.join(GOLDEN, f"postpm_{case}.npz"))
    cfg = lbic_b200.load_config(str(c["config"]))
    m = get_model(str(c["config"]), int(c["seed"]), bool(c["harsh"]), dev)
    pm = lbic_b200.BlkBasedPostProcessing(m)
    if (str(c["config"]), "pp") not in _models:
        with pytest.raises((RuntimeError, ValueError)):
            pm(torch.zeros(1, m.Cin, 3, 3, device=dev))                  # weights not loaded yet
        _models[(str(c["config"]), "pp")] = True
    pm.load_state_dict(weights.synth_postpm_state_dict(cfg, int(f["seed"])))
    z = torch.from_numpy(c["zhat"]).to(dev)
    out = pm(z)
    want = torch.from_numpy(f["out"])
    # the tensor cores' truncating accumulation grows with the contraction length (profiles/r2_closed_loop_parity.md):
    # 2e-5 at K = 9 * 192 (B8), four times that at K = 9 * 768 (B16)
    tol = 2e-5 * max(1.0, 9 * m.Cin / 1728.0)
    err = float((out.cpu() - want).abs().max())
    assert err < tol * max(1.0, float(want.abs().max())), f"post-processing output differs by {err:.3e} (tolerance {tol:.1e})"
    border = torch.ones(z.shape[2], z.shape[3], dtype=torch.bool)
    border[1:-1, 1:-1] = False
    assert torch.equal(out.cpu()[:, :, border], z.cpu()[:, :, border])
    assert float((out - z).abs().max()) > 0.05                            # the residual is really there
    assert torch.equal(pm(z, clamp=True), out.clamp(-0.5, 0.5))
    big = pm(z.repeat(70, 1, 1, 1))
    assert torch.equal(big[0], out[0]) and torch.equal(big[69], out[0])
    # degenerate grids: nothing but border
    thin = z[:, :, :2].contiguous()
    assert torch.equal(pm(thin), thin)


@pytest.mark.parametrize("n,H,W", [(2, 176, 208), (1, 512, 768), (3, 161, 333)])
def test_gpu_metrics_match_torch_definitions(dev, n, H, W):
    """SURVEY.md 8(f) rank 4: the figures of AGENT:611-619 from lbic_image_metrics: MSE / PSNR against F.mse_loss
    (1e-6 relative: fp64 accumulation here, fp32 there) and MS-SSIM against the torch restatement of pytorch_msssim
    in lbic_b200.codec (1e-5; odd sizes exercise the zero-padded average pooling)."""
    from lbic_b200 import codec
    m = get_model("B8_lowrate", 1337, False, dev)
    g = torch.Generator().manual_seed(n * 1000 + H)
    x = (weights.synth_images(n, H, W, seed0=70) - 0.5).to(dev)
    y = (x + 0.08 * torch.randn(x.shape, generator=g).to(dev) * torch.rand(n, 1, 1, 1, generator=g).to(dev)).clamp(-0.5, 0.5)
    got = m.image_metrics(x, y)
    for i in range(n):
        mse = float(torch.nn.functional.mse_loss(x[i:i + 1], y[i:i + 1]))
        assert abs(got["mse"][i] - mse) <= 1e-6 * mse
        assert abs(got["psnr"][i] - (-10 * np.log10(mse))) < 1e-4
        want = float(codec.ms_ssim(x[i:i + 1] + 0.5, y[i:i + 1] + 0.5, data_range=1.0))
        assert abs(got["msssim"][i] - want) < 1e-5, (got["msssim"][i], want)
    only = m.image_metrics(x, y, msssim=False)
    assert only["msssim"] is None and np.array_equal(only["mse"], got["mse"])
    with pytest.raises(RuntimeError):
        m.image_metrics(x[:, :, :100], y[:, :, :100])                     # too small for five scales


def test_validation_rate_estimate(dev):
    """validate_recu_reco_fast (AGENT:491-549): closed loop without entropy coding + -log2 pmf.  The reconstruction
    must equal compress()'s; the self-information must match the oracle's on the same symbols/scales (1e-3 relative:
    erfc differs by a few ulp between CUDA and torch); the estimated rate is of the order of the coded rate (with
    random-init weights the predicted scales are poor, so the two need not be close)."""
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    from oracle import nets
    cfg = lbic_b200.load_config("B8_lowrate")
    m = get_model("B8_lowrate", 1337, False, dev)
    img = weights.synth_images(3, 5 * 8, 9 * 8, seed0=300)
    x = arrange_block_pixels_to_channel_dim((img - 0.5).to(dev), 8)
    zhat, info = m.validate_recu_reco(x)
    strings, zhat2, sym, idx = m.compress_batch(x, lanes=1, return_symbols=True)
    assert torch.equal(zhat, zhat2)
    P = nets.effective_params(weights.synth_state_dict(cfg, 1337), cfg)
    s2, i2, _, _, ksi = nets.whole_image_eval(P, x.cpu(), zhat.cpu())
    want = nets.self_information(sym.cpu().permute(0, 3, 1, 2), ksi[:, :m.M])
    got = info.cpu()
    same = (s2 == sym.cpu()).permute(0, 3, 1, 2)
    rel = ((got - want).abs() / want.clamp(min=1e-3))[same]
    assert float(rel.max()) < 1e-3, f"self-information differs by {float(rel.max()):.2e}"
    est_bits, coded_bits = float(got.sum()), 8.0 * sum(len(s) for s in strings)
    assert 0.5 * coded_bits < est_bits < 2.0 * coded_bits, (est_bits, coded_bits)


@pytest.mark.parametrize("case", KS3111_CASES)
def test_open_loop_forward_matches_reference_golden(dev, case):
    """SURVEY.md 8(f) rank 2: model.forward(zhat, x) (NET:90-106).  tests/golden/forward_<case>.npz holds the UNMODIFIED
    reference's output on the case's x with the case's closed-loop zhat as context (make_golden_forward.py).  No closed
    loop here, so a rounding-boundary flip stays local: symbols must agree to 100 ppm, and the reconstruction and the
    self-informations must match wherever the block's symbols agree."""
    c = load_case(case)
    f = np.load(os.path.join(GOLDEN, f"forward_{case}.npz"))
    m = get_model(str(c["config"]), int(c["seed"]), bool(c["harsh"]), dev)
    x = torch.from_numpy(c["x"]).to(dev)
    zhat = torch.from_numpy(c["zhat"]).to(dev)
    xhat, info, sym = m.forward(zhat, x, return_symbols=True)
    sym_ref = torch.from_numpy(f["symbols"].astype(np.int32))
    diff = (sym[0].cpu() != sym_ref)
    # 100 ppm on a full image; the small fixtures (5-7 k symbols) are allowed two rounding-boundary flips (|d| = 1)
    assert int(diff.sum()) <= max(2, int(1e-4 * diff.numel())), f"{int(diff.sum())} of {diff.numel()} symbols differ"
    assert int((sym[0].cpu() - sym_ref).abs().max()) <= 1
    same_blk = ~diff.any(dim=2)                                        # (Hb, Wb)
    xref, iref = torch.from_numpy(f["xhat"]), torch.from_numpy(f["selfinfo"])
    scale = float(xref.abs().max())
    dx = ((xhat.cpu() - xref)[0].abs().amax(dim=0) * same_blk).max()
    # the harsh weights drive the unclamped output to +-43 through three IGDN stages: relative 1e-4 there (as for the
    # closed-loop harsh case), 2e-5 otherwise
    tol = (1e-4 if bool(c["harsh"]) else 2e-5) * max(1.0, scale)
    assert float(dx) < tol, f"xhat differs by {float(dx):.3e} on blocks with identical symbols"
    di = ((info.cpu() - iref)[0].abs().amax(dim=0) * same_blk).max()
    assert float(di) < 2e-3, f"self-information differs by {float(di):.3e}"
    bits, bits_ref = float(info.sum()), float(iref.sum())
    assert abs(bits - bits_ref) <= 1e-3 * bits_ref
    # the clamp the callers apply (AGENT:667) is available in-kernel, and a second chunking gives the same result
    xc, _ = m.forward(zhat, x, clamp=True)
    assert torch.equal(xc, xhat.clamp(-0.5, 0.5))
    xb, ib = m.forward(zhat.repeat(3, 1, 1, 1), x.repeat(3, 1, 1, 1))
    assert torch.equal(xb[2], xhat[0]) and torch.equal(ib[1], info[0])


@pytest.mark.parametrize("lanes", [1, 0])
def test_image_codec_roundtrip_on_ragged_size(dev, lanes, tmp_path):
    """SURVEY.md 8(f) rank 3: whole-image encode / decode through the self-describing container on an image whose size is
    not a multiple of the block size (replicate padding AGENT:583-586, crop after depth->space), plus PNG in / out."""
    from lbic_b200.codec import ImageCodec, unpack_container
    m = get_model("B8_lowrate", 1337, False, dev)
    codec = ImageCodec(m, lanes=lanes)
    H, W = 203, 261                                             # 26 x 33 blocks after padding to 208 x 264
    img = weights.synth_images(1, H, W, seed0=5)[0]
    blob = codec.encode(img)
    meta, payload = unpack_container(blob)
    assert (meta["H"], meta["W"], meta["B"], meta["lanes"]) == (H, W, 8, lanes)
    rec = codec.decode(blob)
    assert rec.shape == (1, 3, H, W) and float(rec.min()) >= 0.0 and float(rec.max()) <= 1.0
    # the same numbers as driving the model by hand the way eval_model does
    from lbic_b200.codec import pad_to_blocks
    x = lbic_b200.arrange_block_pixels_to_channel_dim(pad_to_blocks(img[None].to(dev) - 0.5, 8), 8)
    if lanes == 1:
        stream, zhat = m.compress(x, [1, 1, 1], m.M)
        assert stream == payload
    else:
        zhat = m.compress_batch(x, lanes=0)[1]
    want = (lbic_b200.arrange_channel_dim_to_block_pixels(zhat, 8)[:, :, :H, :W] + 0.5).clamp(0, 1)
    assert torch.equal(rec, want)
    ev = codec.evaluate(img)
    assert ev["bytes"] == len(payload) and abs(ev["bpp"] - 8.0 * len(payload) / (H * W)) < 1e-12
    assert "msssim" in ev and 0.0 < ev["msssim"] <= 1.0
    # files
    from PIL import Image
    src = tmp_path / "in.png"
    Image.fromarray((img * 255).round().to(torch.uint8).permute(1, 2, 0).numpy(), "RGB").save(src)
    blob2 = codec.encode_file(str(src))
    codec.decode_to_file(blob2, str(tmp_path / "out.png"))
    with Image.open(tmp_path / "out.png") as im:
        assert im.size == (W, H)
    with pytest.raises(ValueError):
        ImageCodec(get_model("B16_lowrate", 1337, False, dev)).decode(blob)


def test_two_devices_in_one_process(dev):
    """One model per device inside ONE process (function attributes, tensor maps and workspaces are per device)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    cfg = lbic_b200.load_config("B8_lowrate")
    sd = weights.synth_state_dict(cfg, 1337)
    img = weights.synth_images(70, 64, 96, seed0=3)
    outs = []
    for d in (1, 0):                                   # the second device first: nothing may be cached from device 0
        devd = torch.device("cuda", d)
        m = BlockBasedImgCompLossyNetv9(cfg, device=devd)
        m.load_state_dict(sd)
        m.update(force=True)
        m.set_option("flow", 2)
        m.set_option("wave", 0)
        m.set_option("enc_thread_streams", 1)
        m.set_option("dec_thread_rows", 1)
        x = arrange_block_pixels_to_channel_dim((img - 0.5).to(devd), 8)
        strings, zhat = m.compress_batch(x, lanes=0)
        zdec = m.decompress_batch(strings, x.shape, lanes=0)
        assert torch.equal(zdec, zhat)
        outs.append((strings, zhat.cpu()))
        m.set_option("enc_thread_streams", 4096)
        m.set_option("dec_thread_rows", 4096)
    assert outs[0][0] == outs[1][0] and torch.equal(outs[0][1], outs[1][1])


@pytest.mark.parametrize("Hb,Wb,ranks", [(12, 17, 1), (12, 17, 3), (5, 40, 2), (9, 4, 4)])
def test_band_steps_with_halo_exchange_equal_single_pass(dev, Hb, Wb, ranks):
    """BASELINE config 5 (one large image in block-row bands over several GPUs, lbic_b200/band.py) on ONE GPU: `ranks`
    model instances on the same device play the ranks, every wavefront step runs per band (lbic_band_step) and the halo
    block of lbic_b200.band.halo_columns is copied from the upper instance's reconstruction to the lower one's -- the
    only thing torch.distributed moves in the real thing.  Streams (lane container) and reconstruction must be
    bit-identical to compress_batch / decompress_batch of the whole image."""
    from lbic_b200 import band
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    cfg = lbic_b200.load_config("B8_lowrate")
    sd = weights.synth_state_dict(cfg, 1337)
    ref_m = get_model("B8_lowrate", 1337, False, dev)
    img = weights.synth_images(1, Hb * 8, Wb * 8, seed0=909)
    x = arrange_block_pixels_to_channel_dim((img - 0.5).to(dev), 8)
    want_s, want_z = ref_m.compress_batch(x, lanes=0)
    models = []
    for _ in range(ranks):
        mm = BlockBasedImgCompLossyNetv9(cfg, device=dev)
        mm.load_state_dict(sd)
        mm.update(force=True)
        models.append(mm)
    bands = [band.band_rows(Hb, ranks, r) for r in range(ranks)]

    def run(decode_blob=None):
        engs = [band.LibEngine(mm) for mm in models]
        if decode_blob is None:
            zts = [e.begin(x, 1, Hb, Wb) for e in engs]
        else:
            cap = (len(decode_blob) + 3) // 4 * 4
            host = np.zeros((1, cap), np.uint8)
            host[0, :len(decode_blob)] = np.frombuffer(decode_blob, np.uint8)
            st = torch.from_numpy(host).to(dev)
            ln = torch.tensor([len(decode_blob)], dtype=torch.int32, device=dev)
            zts = [e.begin(None, 1, Hb, Wb, st, ln) for e in engs]
        for t in range(Wb + 2 * (Hb - 1)):
            for r, (v0, v1) in enumerate(bands):
                recv_h, _ = band.halo_columns(t, v0, v1, Hb, Wb)
                if recv_h is not None and r > 0:
                    zts[r][:, v0 - 1, recv_h] = zts[r - 1][:, v0 - 1, recv_h]
            for r, (v0, v1) in enumerate(bands):
                engs[r].step(t, v0, v1)
        outs = [e.end(v0, v1, decode_blob is None) for e, (v0, v1) in zip(engs, bands)]
        z = torch.cat([o[0][0] for o in outs], dim=0).permute(2, 0, 1).unsqueeze(0)
        lanes = [l for o in outs for l in (o[1] or [])]
        return z, lanes

    z, lanes = run()
    blob = band.pack_lane_container(lanes)
    assert blob == want_s[0], "band-encoded lane container differs from the single-pass one"
    assert torch.equal(z, want_z)
    zd, _ = run(blob)
    assert torch.equal(zd, want_z)
    assert torch.equal(ref_m.decompress_batch([blob], x.shape, lanes=0), want_z)


def test_host_calls_banded_pipeline_equals_device_calls(dev):
    """lbic_encode_host / lbic_decode_host move the batch over PCIe in bands of block rows overlapped with the wavefront
    (LBIC_OPT_HOST_BANDS); any band count must return exactly what the device-resident calls return; odd batch size,
    a grid whose rows do not divide by the band count, both containers, both topologies' first layers."""
    from lbic_b200 import _lib
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    L = _lib.lib()
    for cfgname, n, Hb, Wb in (("B8_lowrate", 11, 5, 9), ("B4_highrate", 3, 19, 7)):
        m = get_model(cfgname, 1337, False, dev)
        B = m.B
        img = weights.synth_images(n, Hb * B, Wb * B, seed0=77)
        x = arrange_block_pixels_to_channel_dim((img - 0.5).to(dev), B)
        xh = x.cpu().contiguous()
        try:
            for lanes in (0, 1):
                want_s, want_z = m.compress_batch(x, lanes=lanes)
                cap = (m.stream_bound(Hb, Wb, lanes) + 3) // 4 * 4
                for bands in (1, 3, 16):
                    m.set_option("host_bands", bands)
                    zenc, zdec = torch.full_like(xh, 7.0), torch.full_like(xh, 9.0)
                    streams = np.zeros((n, cap), np.uint8)
                    lens = np.zeros(n, np.uint32)
                    _lib.check(L.lbic_encode_host(m._need(), xh.data_ptr(), n, Hb, Wb, zenc.data_ptr(), streams.ctypes.data,
                                                  cap, lens.ctypes.data, lanes))
                    _lib.check(L.lbic_decode_host(m._need(), streams.ctypes.data, lens.ctypes.data, cap, n, Hb, Wb,
                                                  zdec.data_ptr(), lanes))
                    got = [streams[i, :lens[i]].tobytes() for i in range(n)]
                    assert got == want_s, f"bitstreams differ ({cfgname}, lanes={lanes}, bands={bands})"
                    assert torch.equal(zenc, want_z.cpu()) and torch.equal(zdec, zenc)
        finally:
            m.set_option("host_bands", 16)


@pytest.mark.parametrize("cfgname,H,W", [("B8_lowrate", 203, 261), ("B8_lowrate", 64, 96), ("B4_highrate", 50, 37),
                                         ("B16_lowrate", 40, 72)])
def test_u8_image_entry_points_match_eval_model_steps(dev, cfgname, H, W):
    """lbic_encode_images_u8_host / lbic_decode_images_u8_host = eval_model's per-image body (AGENT:581-599, 610-628)
    for a batch: the streams must equal those of compress() on the float tensor eval_model builds (ToTensor, -0.5,
    replicate padding, space-to-depth: done here with torch ops exactly as the reference does), and the 8-bit images
    must equal depth-to-space + crop + save_image's quantisation of the reconstruction.  Ragged sizes included."""
    import torch.nn.functional as F
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim, arrange_channel_dim_to_block_pixels
    m = get_model(cfgname, 1337, False, dev)
    B = m.B
    n = 5
    imgs = np.stack([weights.synth_image_u8(H, W, seed=40 + i) for i in range(n)])
    # ToTensor on the CPU as the reference's loader does (a TRUE division: torch's CUDA kernel for `x / scalar` multiplies
    # by the reciprocal and differs in the last bit for some pixel values), then AGENT:581
    x = (torch.from_numpy(imgs).float().div(255) - 0.5).to(dev)
    Hp, Wp = (H + B - 1) // B * B, (W + B - 1) // B * B
    xp = F.pad(x, (0, Wp - W, 0, Hp - H), mode="replicate")                           # AGENT:583-586
    xb = arrange_block_pixels_to_channel_dim(xp, B)                                   # AGENT:588-589
    for lanes in (1, 0):
        want_s, zhat = m.compress_batch(xb, lanes=lanes)
        rec = arrange_channel_dim_to_block_pixels(zhat, B)[:, :, :H, :W] + 0.5         # AGENT:610, 628
        want_u8 = rec.mul(255).add_(0.5).clamp_(0, 255).to(torch.uint8).cpu().numpy()  # torchvision.utils.save_image
        for bands in (16, 2):
            m.set_option("host_bands", bands)
            got_s, got_rec = m.compress_images_u8(imgs, lanes=lanes, return_recon=True)
            assert got_s == want_s, f"streams differ (lanes={lanes}, bands={bands})"
            assert np.array_equal(got_rec, want_u8)
            dec = m.decompress_images_u8(got_s, H, W, lanes=lanes)
            assert np.array_equal(dec, want_u8)
        m.set_option("host_bands", 16)
        got_s2, none = m.compress_images_u8(torch.from_numpy(imgs), lanes=lanes)
        assert got_s2 == want_s and none is None


def test_layout_kernels_match_reference_definition(dev):
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim, arrange_channel_dim_to_block_pixels
    from oracle import nets
    for B, H, W in [(8, 48, 72), (4, 20, 12), (16, 32, 64)]:
        img = torch.rand(2, 3, H, W)
        want = nets.arrange_block_pixels_to_channel_dim(img, B)
        got = arrange_block_pixels_to_channel_dim(img.to(dev), B)
        assert torch.equal(got.cpu(), want)
        back = arrange_channel_dim_to_block_pixels(got, B)
        assert torch.equal(back.cpu(), img)


def test_saturation_counter(dev):
    """The fp16 operand planes clip at +-65504 silently; with check_saturation set every layer's hi plane is scanned and
    the clipped elements are counted: none for the conditioned synthetic weights, many when the last encoder layer is
    scaled far out of range; results do not depend on the option."""
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    cfg = lbic_b200.load_config("B8_lowrate")
    img = weights.synth_images(3, 5 * 8, 7 * 8, seed0=9)
    x = arrange_block_pixels_to_channel_dim((img - 0.5).to(dev), 8)
    m = get_model("B8_lowrate", 1337, False, dev)
    ref = m.compress_batch(x, lanes=0, return_symbols=True)
    try:
        m.set_option("check_saturation", 1)
        m.saturation_count(reset=True)
        got = m.compress_batch(x, lanes=0, return_symbols=True)
        assert m.saturation_count() == 0
        assert got[0] == ref[0] and torch.equal(got[1], ref[1]) and torch.equal(got[2], ref[2])
    finally:
        m.set_option("check_saturation", 0)
    big = BlockBasedImgCompLossyNetv9(cfg, device=dev)
    big.load_state_dict(weights.synth_state_dict(cfg, 1337, latent_gain=3e6))
    big.update(force=True)
    big.set_option("check_saturation", 1)
    o = big.encode_device(x, lanes=0, stream_cap=1 << 20)
    n = big.saturation_count()
    assert n > 0, "y_qnt of ~1e5 must clip its fp16 hi plane"
    assert big.saturation_count() == 0      # reset by the previous call


def test_error_behaviour(dev):
    cfg = lbic_b200.load_config("B8_lowrate")
    m = BlockBasedImgCompLossyNetv9(cfg, device=dev)
    x = torch.zeros(1, m.Cin, 2, 2, device=dev)
    with pytest.raises(ValueError):          # reference: ValueError("Uninitialized CDFs. Run update() first")
        m.compress(x, [1, 1, 1], m.M)
    m.load_state_dict(weights.synth_state_dict(cfg, 1))
    with pytest.raises(ValueError):
        m.compress(x, [1, 1, 1], m.M)        # tables still missing
    m.update(force=True)
    with pytest.raises(ValueError):
        m.compress(x, [2, 2, 2], m.M)        # LRU inconsistent with KS
    m.compress(x, [1, 1, 1], m.M)


def test_stream_capacity_and_corrupt_streams(dev):
    """Error behaviour of the entropy stage: a too-small caller buffer is reported (never written past), a damaged
    lane container is rejected, a damaged reference stream decodes to something finite (the coder reads zeros past the
    end, like a corrupt CompressAI stream yields garbage symbols, never a crash), and the model stays usable."""
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim
    m = get_model("B8_lowrate", 1337, False, dev)
    img = weights.synth_images(2, 4 * 8, 6 * 8, seed0=12)
    x = arrange_block_pixels_to_channel_dim((img - 0.5).to(dev), 8)
    good, zhat = m.compress_batch(x, lanes=1)
    o = m.encode_device(x, lanes=1, stream_cap=64)                 # real streams are ~2 kB
    with pytest.raises(RuntimeError):
        m._gather_streams(o)
    lane_strings, _ = m.compress_batch(x, lanes=0)
    bad = bytearray(lane_strings[0]); bad[0] ^= 0xFF               # break the 'LBML' magic
    with pytest.raises(RuntimeError, match="malformed"):           # rejected, not silently decoded to garbage
        m.decompress_batch([bytes(bad), lane_strings[1]], x.shape, lanes=0)
    # a lane length that wraps 32-bit offset arithmetic (ADVICE r1): offset + 0xFFFFFFF0 overflows to a small number
    wrap = bytearray(lane_strings[0])
    wrap[8 + 4:8 + 8] = (0xFFFFFFF0).to_bytes(4, "little")         # length of lane 1
    with pytest.raises(RuntimeError, match="malformed"):
        m.decompress_batch([bytes(wrap), lane_strings[1]], x.shape, lanes=0)
    odd = bytearray(lane_strings[0])
    odd[8:12] = (int.from_bytes(odd[8:12], "little") + 2).to_bytes(4, "little")   # lane 0 length not a multiple of 4
    with pytest.raises(RuntimeError, match="malformed"):
        m.decompress_batch([bytes(odd), lane_strings[1]], x.shape, lanes=0)
    # the device API flags the error without raising and leaves the intact image of the batch untouched
    cap = (max(len(bad), len(lane_strings[1])) + 3) // 4 * 4
    host = np.zeros((2, cap), np.uint8)
    host[0, :len(bad)] = np.frombuffer(bytes(bad), np.uint8)
    host[1, :len(lane_strings[1])] = np.frombuffer(lane_strings[1], np.uint8)
    lens = torch.tensor([len(bad), len(lane_strings[1])], dtype=torch.int32, device=dev)
    zb = m.decode_device(torch.from_numpy(host).to(dev), lens, 2, x.shape[2], x.shape[3], lanes=0)
    with pytest.raises(RuntimeError):
        m.check_errors()
    assert torch.equal(zb[1], zhat[1])                             # the intact image is unaffected
    m.check_errors()                                               # the flag is cleared by reading it
    # lane container of a one-block-row image (lanes == 1 row): header must still be parsed as a container
    x1 = x[:, :, :1].contiguous()
    s1, z1 = m.compress_batch(x1, lanes=0)
    assert s1[0][:4] == b"LBML" and torch.equal(m.decompress_batch(s1, x1.shape, lanes=0), z1)
    assert m.stream_bound(1, 6, 0) >= m.stream_bound(1, 6, 1) + 12
    cut = good[0][: len(good[0]) // 2 // 4 * 4]
    zc = m.decompress_batch([cut, good[1]], x.shape, lanes=1)
    assert bool(torch.isfinite(zc).all()) and torch.equal(zc[1], zhat[1])
    again, zhat2 = m.compress_batch(x, lanes=1)
    assert again == good and torch.equal(zhat2, zhat)
    with pytest.raises((RuntimeError, ValueError)):
        m.compress_batch(x[:0], lanes=1)
