"""The entropy stage bit for bit: every rANS encoder and decoder form and the CDF tables they read, against the
CompressAI coder restated in oracle/ (native.rans_encode / RansDecoder) and a NumPy restatement of the table builder.

The closed-loop tests elsewhere only see the symbols the network happens to produce and compare the kernel forms with each
other.  Here each form is chosen explicitly through the test hooks (lbic_debug_rans_encode, lbic_debug_rans_decode_steps,
lbic_debug_compact_tables), on crafted symbols that reach the edges closed-loop data almost never reaches: escapes at
every nibble count up to the largest raw value below 2^31, the escape bin itself, frequencies 1, 2, 3, 2^k and 2^k + 1,
the ends of the decoders' 32-entry search windows, rows shorter than a window, stream lengths around the CTA encoder's
1024-symbol chunks; on four scale tables: the reference's, a non-geometric one that fits the compact 16-bit form, one
whose rows (4037 entries) nearly fill the table builder's capacity, and one too large for the compact form.  JSON lines
(pytest -rP) list the forms and tables exercised."""
import ctypes
import json
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import lbic_b200
from lbic_b200 import _lib, weights
from lbic_b200.net import BlockBasedImgCompLossyNetv9, get_scale_table
from oracle import native as onative
from oracle import nets
from conftest import golden_cases, load_case

TAIL_MASS = 1e-9
COMPACT_MAX = 60000                 # tables_compact: 16-bit rows of at most this many entries fit shared memory
LENGTHS = (0, 1, 3, 4, 5, 255, 256, 257, 1023, 1024, 1025, 4099)
RAWS = [r for k in range(1, 8) for r in (16 ** k - 2, 16 ** k - 1, 16 ** k, 16 ** k + 1)] + [2 ** 31 - 2, 2 ** 31 - 1]


def geometric(hi):
    return torch.exp(torch.linspace(np.log(0.11), np.log(hi), 64))


def quadratic(hi):
    i = torch.arange(64, dtype=torch.float64)
    return (0.11 + (hi - 0.11) * (i / 63) ** 2).float()


# name -> scale table; entries of the compact rows: 27 192, 52 776, 33 972 (rows of 4037), 67 512 (no compact form)
TABLES = {"geometric_256": get_scale_table(), "quadratic_200": quadratic(200.0), "geometric_330": geometric(330.0),
          "quadratic_256": quadratic(256.0)}


def report(**kw):
    print(json.dumps(kw))


@pytest.fixture(scope="module")
def model():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    cfg = lbic_b200.load_config("B8_lowrate")
    m = BlockBasedImgCompLossyNetv9(cfg, device=torch.device("cuda", 0))
    m.load_state_dict(weights.synth_state_dict(cfg, 1337))
    m.update(force=True)
    yield m
    m.update(force=True)


def build(m, tab):
    """lbic_build_tables for scale table tab -> (cdf [64, stride], cdf_length, offset) as installed; raises on failure."""
    st = np.ascontiguousarray(tab.numpy().astype(np.float32))
    h = m._need()
    _lib.check(_lib.lib().lbic_build_tables(h, st.ctypes.data, 64, TAIL_MASS, None))
    n, stride = ctypes.c_int(), ctypes.c_int()
    _lib.check(_lib.lib().lbic_get_tables(h, ctypes.byref(n), ctypes.byref(stride), None, None, None))
    cdf = np.empty((64, stride.value), dtype=np.int32)
    ln, off = np.empty(64, dtype=np.int32), np.empty(64, dtype=np.int32)
    _lib.check(_lib.lib().lbic_get_tables(h, None, None, cdf.ctypes.data, ln.ctypes.data, off.ctypes.data))
    return cdf, ln, off


# ---- A. tables ---------------------------------------------------------------------------------------------------------
def numpy_tables(tab):
    """build_cdf_kernel's stated definition: the pmf of GaussianConditional.update in fp32 with each erfc evaluated in
    float64 and rounded once to fp32, quantised by CompressAI's pmf_to_quantized_cdf (oracle restatement)."""
    from scipy.special import erfc
    from scipy.stats import norm
    f32 = np.float32
    mult = f32(-norm.ppf(TAIL_MASS / 2))
    c = f32(-0.70710678118654752440)

    def cum(v):
        return f32(0.5) * erfc((c * v).astype(np.float64)).astype(f32)

    scales = tab.numpy().astype(f32)
    centers = np.ceil(scales * mult).astype(np.int64)
    stride = int(2 * centers.max() + 3)
    cdf = np.zeros((64, stride), dtype=np.int32)
    for i, (s, ctr) in enumerate(zip(scales, centers)):
        samp = np.abs(np.arange(2 * ctr + 1) - ctr).astype(f32)
        pmf = cum((f32(0.5) - samp) / s) - cum((f32(-0.5) - samp) / s)
        tail = f32(2.0) * cum(np.array([(f32(-0.5) - f32(ctr)) / s], dtype=f32))
        q = onative.pmf_to_quantized_cdf(np.concatenate([pmf, tail]).astype(f32))
        cdf[i, :q.size] = q
    return cdf, (2 * centers + 3).astype(np.int32), (-centers).astype(np.int32)


def compact_reference(cdf, ln):
    """Tables::cdf16 restated: rows without their final 65536 back to back, total rounded up to even, lut[l][b] = first k
    with row[k] > 256 b (lut[l][256] = len - 1)."""
    off = np.concatenate([[0], np.cumsum(ln - 1)]).astype(np.int32)
    rows = np.concatenate([cdf[l, :ln[l] - 1] for l in range(64)]).astype(np.uint16)
    lut = np.array([[np.searchsorted(cdf[l, :ln[l]], 256 * b, side="right") for b in range(256)] + [ln[l] - 1]
                    for l in range(64)], dtype=np.uint16)
    return (int(off[64]) + 1) & ~1, rows, off, lut


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TABLES))
def test_tables_bit_exact_vs_numpy_restatement(model, name):
    """CDF rows, lengths and offsets equal the float64-erfc restatement bit for bit; the compact rows and bucket tables equal
    their restatement; they exist exactly when the rows fit (<= 60 000 entries).  Entries that differ from oracle.nets'
    build_tables (torch's fp32 erfc) are counted and reported, not asserted (0 for these four tables on the host)."""
    tab = TABLES[name]
    cdf, ln, off = build(model, tab)
    want, wln, woff = numpy_tables(tab)
    assert np.array_equal(ln, wln) and np.array_equal(off, woff)
    assert cdf.shape == want.shape, f"{name}: stride {cdf.shape[1]}, expected {want.shape[1]}"
    diff = int((cdf != want).sum())
    assert diff == 0, f"{name}: {diff} CDF entries differ from the float64-erfc restatement"
    ocdf, oln, ooff = (t.numpy() for t in nets.build_tables(tab))
    assert np.array_equal(oln, ln) and np.array_equal(ooff, off)
    vs_torch = int((ocdf != cdf).sum())
    total, rows, offs, lut = model.debug_compact_tables()
    wtotal, wrows, woffs, wlut = compact_reference(cdf, ln)
    assert (total > 0) == (wtotal <= COMPACT_MAX), f"{name}: compact total {total}, rows hold {wtotal} entries"
    if total:
        assert total == wtotal and np.array_equal(offs, woffs)
        assert np.array_equal(rows[:wrows.size], wrows), f"{name}: compact rows differ"
        assert np.array_equal(lut, wlut), f"{name}: {int((lut != wlut).sum())} bucket-table entries differ"
    report(test="tables", table=name, stride=int(cdf.shape[1]), entries=int((ln - 1).sum()), compact_total=total,
           differ_from_torch_fp32_erfc=vs_torch)


@pytest.mark.gpu
def test_table_beyond_capacity_fails_cleanly(model):
    """0.11 ... 336 needs rows of 4109 entries, beyond the builder's 4096: LBIC_ERR_INVALID, the installed tables stay."""
    build(model, TABLES["geometric_256"])
    with pytest.raises(RuntimeError, match="lbic error -1"):
        build(model, geometric(336.0))
    total, _, _, _ = model.debug_compact_tables()
    assert total == 27192


# ---- crafted symbols ---------------------------------------------------------------------------------------------------
def window_start(center, ln):
    """Start g of the decoders' 32-entry window (dec_symbol_warp / rans_decode_row_warp)."""
    return max(0, min(center - 15, max(ln - 32, 0)))


def value_of_raw(r, maxv):
    return maxv + r // 2 if r % 2 == 0 else -(r + 1) // 2


def symbol_pool(cdf, ln, off, seed=0):
    """(symbols int32, indexes uint8): for every index the values 0, 1, the window edges, the escape bin and its neighbours,
    escapes with raw values at every nibble count, one or two values of each frequency 1, 2, 3, 2^k, 2^k + 1 in random
    order, then a run of 300 escapes and a run of 300 frequency-1 symbols."""
    syms, idxs, f1 = [], [], []
    for ci in range(64):
        L, o = int(ln[ci]), int(off[ci])
        c, maxv = -o, L - 2
        g = window_start(c, L)
        vs = [0, 1] + list(range(c - 16, c + 18)) + [g - 1, g, g + 30, g + 31, maxv - 1, maxv, maxv + 1, -1]
        vs += [value_of_raw(r, maxv) for r in RAWS]
        freq = np.diff(cdf[ci, :L].astype(np.int64))[:maxv]
        for f in [1, 2, 3] + [2 ** k + d for k in range(2, 16) for d in (0, 1)]:
            vs += [int(v) for v in np.nonzero(freq == f)[0][:2]]
        f1 += [(ci, int(v)) for v in np.nonzero(freq == 1)[0][:8]]
        syms += [v + o for v in vs]
        idxs += [ci] * len(vs)
    rng = np.random.default_rng(seed)
    perm = rng.permutation(len(syms))
    syms, idxs = np.array(syms, dtype=np.int64)[perm], np.array(idxs, dtype=np.int64)[perm]
    esc_ci = rng.integers(0, 64, 300)
    esc_raw = rng.integers(0, 2 ** 31, 300)
    esc = np.array([value_of_raw(int(r), int(ln[ci]) - 2) + int(off[ci]) for ci, r in zip(esc_ci, esc_raw)])
    assert f1, "no frequency-1 entries in the table"
    run = [f1[j % len(f1)] for j in range(300)]
    one = np.array([v + int(off[ci]) for ci, v in run])
    half = syms.size // 2
    syms = np.concatenate([syms[:half], esc, syms[half:], one])
    idxs = np.concatenate([idxs[:half], esc_ci, idxs[half:], [ci for ci, _ in run]])
    assert syms.min() >= -2 ** 31 and syms.max() < 2 ** 31
    return syms.astype(np.int32), idxs.astype(np.uint8)


def streams_from_pool(pool, lengths):
    """Stream s of the given lengths: the pool from an offset of its own, wrapping around."""
    sym, idx = pool
    P = sym.size
    take = [(np.arange(L) + (s * 7919 + L * 131)) % P for s, L in enumerate(lengths)]
    flat = np.concatenate(take) if take else np.zeros(0, np.int64)
    return sym[flat], idx[flat]


def encode_cases():
    cases = [(f"{n}x{L}", [L] * n) for L in LENGTHS for n in (1, 33)]
    cases += [("592x257", [257] * 592), ("593x1024", [1024] * 593), ("4096x12", [12] * 4096)]
    cases += [("mixed", [LENGTHS[s % len(LENGTHS)] for s in range(37)]),
              ("mixed_x4", [(0, 4, 8, 256, 1024, 4100, 12)[s % 7] for s in range(41)])]
    return cases


# ---- B. encoders -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TABLES))
def test_encoders_bit_exact_vs_oracle(model, name):
    """Every encoder form whose preconditions hold (warp per stream: always; CTA per stream: equal lengths; thread per
    stream: compact tables, lengths and starts multiples of 4) writes the oracle's bytes for every stream; where they do
    not hold the hook refuses with LBIC_ERR_INVALID."""
    cdf, ln, off = build(model, TABLES[name])
    compact = model.debug_compact_tables()[0] > 0
    T = onative.Tables(cdf, ln, off)
    pool = symbol_pool(cdf, ln, off)
    dev = torch.device("cuda", 0)
    ran = {1: 0, 2: 0, 3: 0}
    for case, lengths in encode_cases():
        sym, idx = streams_from_pool(pool, lengths)
        seg = np.concatenate([[0], np.cumsum(lengths)])
        want = [onative.rans_encode(sym[a:b], idx[a:b], T) for a, b in zip(seg[:-1], seg[1:])]
        sym_d, idx_d = torch.from_numpy(sym).to(dev), torch.from_numpy(idx).to(dev)
        cap = 8 * max(lengths) + 64
        for form in (1, 2, 3):
            ok = form == 1 or (form == 2 and len(set(lengths)) == 1) or \
                (form == 3 and compact and all(L % 4 == 0 for L in lengths))
            if not ok:
                with pytest.raises(RuntimeError, match="lbic error -1"):
                    model.debug_rans_encode(sym_d, idx_d, seg, form, cap)
                continue
            got = model.debug_rans_encode(sym_d, idx_d, seg, form, cap)
            bad = [s for s in range(len(lengths)) if got[s] != want[s]]
            assert not bad, f"{name} {case} form {form}: streams {bad[:5]} differ from the oracle (length {lengths[bad[0]]})"
            ran[form] += len(lengths)
    report(test="encoders", table=name, compact=compact, pool=int(pool[0].size),
           streams_checked={"warp": ran[1], "block": ran[2], "thread": ran[3]})


# ---- C. decoders on bytes produced elsewhere -----------------------------------------------------------------------------
def level_scales(tab):
    """A scale per level whose CDF index (build_indexes) is that level: the level itself."""
    s = tab.clone()
    assert torch.equal(nets.build_indexes(SimpleNamespace(scale_table=tab), s), torch.arange(64, dtype=torch.int32))
    return s


def h16_split(v):
    v = v.clamp(-65504.0, 65504.0)
    hi = v.half()
    return hi, (v - hi.float()).half()


def check_decode_forms(model, streams, sym, idx, n_steps, M, tab, compact, what, seed):
    """Decodes the streams (stream s = steps of M symbols, sym / idx (n_streams, n_steps * M)) with every form; symbols,
    yq = split_h16(sym + mean) and the words consumed must be exact.  Returns the forms that ran."""
    dev = torch.device("cuda", 0)
    n = len(streams)
    sc = level_scales(tab)[torch.from_numpy(idx.astype(np.int64))].reshape(n, n_steps, M)
    g = torch.Generator().manual_seed(seed)
    mu = (torch.randn(n, n_steps, M, generator=g) * 3).float()
    ksi = torch.cat([sc, mu], dim=2).permute(1, 0, 2).reshape(n_steps * n, 2 * M).contiguous().to(dev)
    want = torch.from_numpy(sym.astype(np.int32)).reshape(n, n_steps, M).permute(1, 0, 2)
    hi_w, lo_w = h16_split(want.float() + mu.permute(1, 0, 2))
    words = torch.tensor([len(s) // 4 for s in streams], dtype=torch.int32)
    ran = []
    for form in (0, 1, 2, 3):
        if (form == 2 and not compact) or (form == 3 and (not compact or M % 4)):
            with pytest.raises(RuntimeError, match="lbic error -1"):
                model.debug_rans_decode_steps(streams, ksi, M, n_steps, form)
            continue
        s, hi, lo, pos = model.debug_rans_decode_steps(streams, ksi, M, n_steps, form)
        bad = int((s.cpu() != want).sum())
        assert bad == 0, f"{what} form {form}: {bad} symbols differ"
        if form:
            assert torch.equal(hi.cpu().view(torch.int16), hi_w.view(torch.int16)), f"{what} form {form}: yq hi plane"
            assert torch.equal(lo.cpu().view(torch.int16), lo_w.view(torch.int16)), f"{what} form {form}: yq lo plane"
            assert torch.equal(pos.cpu(), words), f"{what} form {form}: words consumed differ from the stream lengths"
        ran.append(form)
    return ran


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TABLES))
def test_decoders_on_oracle_streams(model, name):
    """Every decode form (whole stream, warp step on int32 tables, warp step on shared-memory tables, thread step) on the
    oracle's streams of crafted symbols; the CompressAI decoder consumes every word of them, and so must the steps."""
    tab = TABLES[name]
    cdf, ln, off = build(model, tab)
    compact = model.debug_compact_tables()[0] > 0
    T = onative.Tables(cdf, ln, off)
    pool = symbol_pool(cdf, ln, off, seed=1)
    ran = set()
    for n, n_steps, M in ((1, 1, 16), (1, 300, 16), (33, 64, 16), (7, 257, 16), (300, 4, 16), (5, 40, 6)):
        sym, idx = streams_from_pool(pool, [n_steps * M] * n)
        sym, idx = sym.reshape(n, -1), idx.reshape(n, -1)
        streams = [onative.rans_encode(sym[s], idx[s], T) for s in range(n)]
        d = onative.RansDecoder()
        d.set_stream(streams[0])
        assert np.array_equal(d.decode_stream(idx[0], T), sym[0]) and d.consumed() == len(streams[0])
        ran.update(check_decode_forms(model, streams, sym, idx, n_steps, M, tab, compact, f"{name} {n}x{n_steps}x{M}",
                                      seed=n_steps))
    report(test="decoders_oracle_streams", table=name, compact=compact, forms=sorted(ran))


@pytest.mark.gpu
@pytest.mark.parametrize("case", golden_cases())
def test_decoders_on_reference_streams(model, case):
    """Every decode form on the unmodified reference's stream of a golden case, with that case's indexes."""
    c = load_case(case)
    tab = TABLES["geometric_256"]
    build(model, tab)
    sym = c["symbols"].astype(np.int32).reshape(1, -1)
    idx = c["indexes"].astype(np.uint8).reshape(1, -1)
    M = int(c["symbols"].shape[-1])
    n_steps = sym.size // M
    ran = check_decode_forms(model, [c["stream"].tobytes()], sym, idx, n_steps, M, tab, True, case, seed=7)
    report(test="decoders_reference_streams", case=case, symbols=int(sym.size), forms=ran)


# ---- D. the encoder's reciprocal, restated on the host ---------------------------------------------------------------------
def test_reciprocal_division_host_restatement():
    """rans_encode_kernel / rans_encode_block_kernel divide by the range with rcp = ceil(2^(63+s) / range), s =
    ceil(log2 range), computed as two 64-bit divides: for every range 2 ... 65535, floor(x / range) = mulhi64(x, rcp) >>
    (s - 1) at the state bounds x = RANS_L and x_max - 1 (x_max = range << 47) and at multiples of the range near x_max."""
    RANS_L, MASK = 1 << 31, (1 << 64) - 1
    for rng in range(2, 65536):
        shift = 0
        while rng > (1 << shift):
            shift += 1
        x0, x1 = rng - 1, 1 << (shift + 31)
        t1 = x1 // rng
        x0 = (x0 + ((x1 % rng) << 32)) & MASK
        rcp = (x0 // rng + (t1 << 32)) & MASK
        assert rcp == -(-(1 << (63 + shift)) // rng), rng
        x_max = rng << 47
        k = (x_max - 1) // rng
        for x in (RANS_L, RANS_L + 1, x_max - 1, rng * k - 1, rng * k, rng * (k - 1) - 1, rng * (k - 1), rng * 65536):
            if RANS_L <= x < x_max:
                assert ((x * rcp) >> 64) >> (shift - 1) == x // rng, (rng, x)
