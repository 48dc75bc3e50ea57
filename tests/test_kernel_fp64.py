"""One fused GEMM layer at a time against a plain float64 (or fp32 restatement) reference.

The parity tests of test_gpu_parity.py compare kernel forms with each other, and whole networks with the oracle at bars
sized for closed-loop noise; an arithmetic error that every form shares, in one layer, can hide behind those.  Here each
core form (SIMT twin, per-tile tcgen05 kernel at every split-factor tile width, persistent kernel, its CTA-pair forms)
and each epilogue mode is compared, through lbic_debug_layer, with a reference of the same single operation, at the
(K segments, cout) of every GEMM layer the codec packs, on the operands the codec feeds them.  Worst errors are printed
as JSON (pytest -rP shows them)."""
import json
import math
from types import SimpleNamespace

import pytest
import torch

import lbic_b200
from lbic_b200 import weights
from lbic_b200.net import BlockBasedImgCompLossyNetv9, get_scale_table
from oracle import nets

pytestmark = pytest.mark.gpu

CONFIGS = ["B8_lowrate", "B4_highrate", "B8_highrate", "B16_lowrate"]
R_LIST = (1, 16, 17, 63, 64, 65, 127, 128, 129, 255, 256, 257, 1000, 4097)
TC_FORMS = ("tc", "ws", "pair", "pair_wide")          # the tensor-core forms: one MMA order, identical bits
H16_MAX = 65504.0

# GEMM error bar, per output element (r, c), relative to |A||W|_rc = sum_k |a_rk||w_ck|:
#   C0 = 2^-20: the hi/lo representation of each operand (<= 2^-22 relative each) and the dropped lo*lo term (2^-24),
#        2^-21 in all, with a 2x margin;
#   C1 = 2.7e-8 per unit of K: the tensor core's truncating fp32 accumulation, linear in K.  The steepest slope in
#        profiles/r2_gemm_precision.jsonl is the non-negative (GDN-like, no cancellation) operand set at K = 576:
#        max error 7.57e-6 of |D| = |A||W|, i.e. 1.31e-8 per unit of K; C1 is twice that;
#   FLOOR = 2^-24 absolute per unit of ||W_c||_1 + ||A_r||_1: a lo plane below fp16's normal range (|v| < 2^-3, e.g. the
#        reconstruction of flat grey regions) is rounded to the subnormal spacing 2^-24, an error of up to 2^-25 per
#        operand element; twice that.
C0, C1, FLOOR = 2.0 ** -20, 2.7e-8, 2.0 ** -24


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def model(dev):
    cfg = lbic_b200.load_config("B8_lowrate")
    m = BlockBasedImgCompLossyNetv9(cfg, device=dev)
    m.load_state_dict(weights.synth_state_dict(cfg, 1337))
    m.update(force=True)
    return m


def report(**kw):
    print(json.dumps(kw))


def f32(x, dev):
    return torch.tensor(x, dtype=torch.float32, device=dev)


def h16_split(v):
    """split_h16 (csrc/epilogue.cuh) restated: clamp to +-65504, hi = fp16(v), lo = fp16(v - hi), round to nearest even."""
    v = v.clamp(-H16_MAX, H16_MAX)
    hi = v.half()
    return hi, (v - hi.float()).half()


def bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == torch.float16 else torch.int32)


def assert_planes(out, v, what):
    hi, lo = h16_split(v)
    assert torch.equal(bits(out["hi"]), bits(hi)), f"{what}: hi plane is not split_h16 of the result"
    assert torch.equal(bits(out["lo"]), bits(lo)), f"{what}: lo plane is not split_h16 of the result"


# ---- the codec's GEMM layers ---------------------------------------------------------------------------------------
def gemm_layers(cfgname):
    """(name, K per segment, cout, kind) of every GEMM layer the codec packs for a config (csrc/api.cu pack_dual /
    pack_linear / pack_gdn), from weights.layer_specs; a masked 3x3 conv keeps 4 ('A') or 5 ('B') taps."""
    cfg = lbic_b200.load_config(cfgname)
    specs = {p: a for p, kind, a in weights.layer_specs(cfg)}
    kinds = {p: kind for p, kind, a in weights.layer_specs(cfg)}

    def k_of(p):
        mtype, cout, cin, k = specs[p]
        return cin * (1 if k == 1 else (4 if mtype == "A" else 5))

    out = [("F0", [k_of("prtr_forward1"), k_of("prtr_forward2")], specs["prtr_forward1"][1], "conv"),
           ("D0", [k_of("prtr_inverse1"), k_of("prtr_inverse2")], specs["prtr_inverse1"][1], "conv")]
    for p, kind in kinds.items():
        if p in ("prtr_forward1", "prtr_forward2", "prtr_inverse1", "prtr_inverse2"):
            continue
        if kind == "gdn":
            out.append((p, [specs[p][0]], specs[p][0], "gdn"))
        else:
            out.append((p, [k_of(p)], specs[p][1], "conv"))
    seen, uniq = set(), []
    for name, K, cout, kind in out:
        if (tuple(K), cout, kind) not in seen:
            seen.add((tuple(K), cout, kind))
            uniq.append((name, K, cout, kind))
    return uniq


def postpm_layers():
    """The post-processing net of B16 (the largest): a 3x3 conv over all nine taps (K = 9 * 768 = 6912) and a 1x1."""
    C = 3 * 16 * 16
    return [("postpm.0", [9 * C], 4 * C, "conv"), ("postpm.2", [4 * C], C, "conv")]


def operands(family, R, Ks, cout, kind, dev, seed):
    """A segments (R, K_s), W segments (cout, K_s) as the codec feeds a layer:
    randn   - activations and weights of order 1 / 1/sqrt(K);
    zhat    - the reconstruction: integers / 255 - 0.5, every third row flat grey (|a| <= 2/255: subnormal lo planes);
    scaled  - weights packed the way finish_layer packs them (max |w| in [2^9, 2^10)); for GDN layers the operands of
              the gamma product: squares of pre-GDN activations of order 10-100 times non-negative gamma."""
    g = torch.Generator(device=dev).manual_seed(seed)
    Ktot = sum(Ks)
    A, W = [], []
    for K in Ks:
        if family == "zhat":
            a = torch.randint(0, 256, (R, K), generator=g, device=dev).float() / 255.0 - 0.5
            flat = torch.randint(126, 131, (R, K), generator=g, device=dev).float() / 255.0 - 0.5
            a[::3] = flat[::3]
        elif family == "scaled" and kind == "gdn":
            a = (torch.randn(R, K, generator=g, device=dev) * 30.0) ** 2
        else:
            a = torch.randn(R, K, generator=g, device=dev) * (4.0 if family == "scaled" else 1.0)
        w = (torch.rand(cout, K, generator=g, device=dev) * 2 - 1) / math.sqrt(Ktot)
        if family == "scaled" and kind == "gdn":
            w = w.abs()
        A.append(a)
        W.append(w)
    k = 0
    if family == "scaled":
        k = 9 - int(math.floor(math.log2(max(float(w.abs().max()) for w in W))))
        W = [w * 2.0 ** k for w in W]
    return A, W, 2.0 ** -k


def fp64_ref(A, W):
    ref = sum(a.double() @ w.double().T for a, w in zip(A, W))
    aw = sum(a.double().abs() @ w.double().abs().T for a, w in zip(A, W))
    l1 = sum(a.double().abs().sum(1, keepdim=True) + w.double().abs().sum(1)[None, :] for a, w in zip(A, W))
    return ref, aw, l1


def gemm_check(D, A, W, what):
    """Asserts the bar above; returns (worst error / bar, worst error / |A||W|)."""
    ref, aw, l1 = fp64_ref(A, W)
    Ktot = sum(a.shape[1] for a in A)
    err = (D.double() - ref).abs()
    bar = (C0 + C1 * Ktot) * aw + FLOOR * l1
    assert bool(torch.isfinite(D).all()), f"{what}: non-finite output"
    ratio = float((err / bar).max())
    assert ratio <= 1.0, f"{what}: error {ratio:.3f} x the bar ((C0 + C1 K) |A||W| + 2^-24 (|W_c|_1 + |A_r|_1), K = {Ktot})"
    rel = float((err / aw.clamp_min(1e-300)).max())
    return ratio, rel


def split_widths(cout):
    """The tile widths of the six split factors (csrc/api.cu bn_variants, lbic_split)."""
    out = []
    for f in (1, 2, 3, 4, 6, 8):
        nt = f * ((cout + 256 * f - 1) // (256 * f))
        out.append(max(16, ((cout + nt - 1) // nt + 15) // 16 * 16))
    return sorted(set(out))


# ---- A. GEMM cores against float64 at the codec's layer shapes -----------------------------------------------------
@pytest.mark.parametrize("family", ["randn", "zhat", "scaled"])
@pytest.mark.parametrize("net", CONFIGS + ["postpm"])
def test_gemm_cores_vs_fp64_at_layer_shapes(model, dev, net, family):
    layers = postpm_layers() if net == "postpm" else gemm_layers(net)
    fi = ["randn", "zhat", "scaled"].index(family)
    worst = {}
    for li, (name, Ks, cout, kind) in enumerate(layers):
        R = R_LIST[(li + 5 * fi + 3 * len(net)) % len(R_LIST)]
        A, W, _ = operands(family, R, Ks, cout, kind, dev, seed=1000 * li + fi)
        outs = {}
        for core in ("simt",) + TC_FORMS:
            D = model.debug_layer("raw", A, W, core=core)["f32"]
            ratio, rel = gemm_check(D, A, W, f"{net} {name} K={Ks} cout={cout} R={R} {family} {core}")
            outs[core] = D
            w = worst.setdefault(core, dict(ratio=0.0, rel=0.0, at=None))
            if ratio > w["ratio"]:
                w.update(ratio=round(ratio, 4), rel=float(f"{rel:.3e}"), at=f"{name} K={Ks} cout={cout} R={R}")
        for core in TC_FORMS[1:]:
            assert torch.equal(bits(outs[core]), bits(outs["tc"])), f"{net} {name} R={R}: {core} differs from tc in bits"
    report(test="gemm_vs_fp64", net=net, family=family, worst=worst)


@pytest.mark.parametrize("net", CONFIGS + ["postpm"])
def test_every_split_factor_tile_width_is_bit_identical(model, dev, net):
    """The per-tile kernel at each split-factor width of pick_bn / bn_variants (LBIC_OPT_FORCE_BN) against float64 and
    bit for bit against the automatic width, on the two-segment first layer and the widest-K layer."""
    layers = postpm_layers() if net == "postpm" else gemm_layers(net)
    pick = [layers[0], max(layers, key=lambda l: sum(l[1]))]
    worst = 0.0
    for li, (name, Ks, cout, kind) in enumerate(pick):
        A, W, _ = operands("zhat", 257, Ks, cout, kind, dev, seed=77 + li)
        D0 = model.debug_layer("raw", A, W, core="tc")["f32"]
        for bn in split_widths(cout):
            D = model.debug_layer("raw", A, W, core="tc", force_bn=bn)["f32"]
            ratio, _ = gemm_check(D, A, W, f"{net} {name} bn={bn}")
            worst = max(worst, ratio)
            assert torch.equal(bits(D), bits(D0)), f"{net} {name}: tile width {bn} differs from the automatic width in bits"
    report(test="tile_widths", net=net, widths={l[0]: split_widths(l[2]) for l in pick}, worst_ratio=round(worst, 4))


# ---- B. the operand split ------------------------------------------------------------------------------------------
def split_values(dev):
    mags = torch.logspace(-7, 6, 400, dtype=torch.float64)
    pows = torch.tensor([2.0 ** e for e in range(-24, 20)], dtype=torch.float64)
    edge = torch.tensor([H16_MAX, 65519.0, 65520.0, 65536.0, 2.0 ** -14, 2.0 ** -24, 2.0 ** -25], dtype=torch.float64)
    v = torch.cat([mags, pows, edge]).float()
    big = f32([H16_MAX], "cpu")
    v = torch.cat([v, torch.nextafter(big, f32([0.0], "cpu")), torch.nextafter(big, f32([1e9], "cpu"))])
    v = torch.cat([v, -v])
    n = (v.numel() + 47) // 48 * 48
    return torch.cat([v, torch.zeros(n - v.numel())]).to(dev)


def split_err_ok(s, v):
    """s = hi + lo of v: within max(2^-22 |v|, 2^-25) for |v| <= 65504, exactly +-65504 beyond."""
    s, v64 = s.double(), v.double()
    inside = v64.abs() <= H16_MAX
    err = (s - v64).abs()
    bound = torch.maximum(2.0 ** -22 * v64.abs(), torch.full_like(v64, 2.0 ** -25))
    assert bool(torch.isfinite(s).all()), "a split plane holds inf / NaN"
    assert bool((err[inside] <= bound[inside]).all()), f"split error {float((err / bound)[inside].max()):.3f} x the bound"
    assert bool((s[~inside] == torch.sign(v64[~inside]) * H16_MAX).all()), "values beyond 65504 do not saturate at +-65504"
    return float((err / bound)[inside].max())


@pytest.mark.parametrize("core", ["simt", "tc", "pair_wide"])
def test_operand_split_hi_plus_lo(model, dev, core):
    """Activation split (launch_split_f32) and output split (the epilogue's hi/lo planes) over |v| in [1e-7, 1e6]: with an
    identity weight matrix D = hi + lo of each activation exactly; the LRELU planes split D * 2^4 (values up to 1.6e7)."""
    v = split_values(dev)
    n = v.numel()
    A = [v.reshape(-1, 48)]
    Wt = [torch.eye(48, device=dev)]
    D = model.debug_layer("raw", A, Wt, core=core)["f32"].reshape(-1)
    hi_a, lo_a = h16_split(v)
    # values (not bits): the accumulator starts at +0, so a -0 + -0 split reads back as +0
    assert torch.equal(D, hi_a.float() + lo_a.float()), "D = A I^T is not hi + lo of the activations"
    in_ratio = split_err_ok(D, v)
    s = 16.0
    out = model.debug_layer("lrelu", A, Wt, core=core, acc_scale=s)
    y = D * f32(s, dev)
    y = torch.where(y > 0, y, y * f32(0.01, dev))
    assert_planes({"hi": out["hi"].reshape(-1), "lo": out["lo"].reshape(-1)}, y, "lrelu split")
    out_ratio = split_err_ok(out["hi"].reshape(-1).float() + out["lo"].reshape(-1).float(), y)
    report(test="operand_split", core=core, values=n, worst_in=round(in_ratio, 4), worst_out=round(out_ratio, 4))


def test_saturation_count_matches_fp64(model, dev):
    """With check_saturation set, lbic_debug_layer scans its hi plane as run_gemm_layer does; the count must equal the
    outputs beyond 65504 in the float64 reference.  (The scan reads hi = +-65504 as clipped, so the values stay clear
    of [65488, 65504], which rounds to that hi.)"""
    g = torch.Generator(device=dev).manual_seed(5)
    R, K, C = 300, 64, 48
    A = torch.randn(R, K, generator=g, device=dev)
    W = torch.randn(C, K, generator=g, device=dev) * 300.0 / math.sqrt(K)
    ref = A.double() @ W.double().T
    keep = ((ref ** 2 - 65496.0).abs() > 700.0).all(dim=1)     # whole rows away from the rounding band
    A = A[keep]
    ref = ref[keep]
    model.set_option("check_saturation", 1)
    try:
        model.saturation_count(reset=True)
        out = model.debug_layer("pregdn", [A], [W], core="tc")
        n = model.saturation_count(reset=True)
    finally:
        model.set_option("check_saturation", 0)
    want = int((ref.abs() ** 2 > H16_MAX).sum())
    assert want > 0 and n == want, f"saturation count {n}, float64 reference {want}"
    assert bool(torch.isfinite(out["hi"].float()).all())
    report(test="saturation_count", count=n, rows=int(A.shape[0]))


# ---- C. each epilogue mode, isolated from GEMM noise ----------------------------------------------------------------
def nongeometric_table():
    """An increasing scale table that is not geometric (quadratic in the level), as a checkpoint may carry."""
    i = torch.arange(64, dtype=torch.float64)
    return (0.11 + (256.0 - 0.11) * (i / 63) ** 2).float()


def crafted_scales(tab):
    """Every level, one ulp either side of it, below / at / above the 0.11 floor, above the last level, +inf."""
    up, down = torch.nextafter(tab, f32([1e30], "cpu")), torch.nextafter(tab, f32([-1e30], "cpu"))
    floor = f32([0.11], "cpu")
    extra = torch.cat([floor, torch.nextafter(floor, f32([1.0], "cpu")), torch.nextafter(floor, f32([0.0], "cpu")),
                       f32([0.0, -1.0, 0.05, 300.0, 1e30, float("inf")], "cpu"), tab[-1:] * 2])
    return torch.cat([tab, up, down, extra])


def ref_index(scales, tab):
    return nets.build_indexes(SimpleNamespace(scale_table=tab.cpu()), scales.cpu())


def epi_operands(dev, R=300, cout=96):
    """Two K segments as the first encoder layer of B4 has them (x: 48 = less than one 64-wide k-block, zhat taps: 192),
    zhat-like x, weights packed with a power-of-two scale undone by acc_scale."""
    A, W, s = operands("scaled", R, [48, 192], cout, "conv", dev, seed=11)
    A[0] = operands("zhat", R, [48], cout, "conv", dev, seed=12)[0][0]
    return A, W, s


@pytest.mark.parametrize("core", ["simt"] + list(TC_FORMS))
def test_epilogue_modes_exact(model, dev, core):
    """Every mode X against its formula applied to the same core's RAW accumulator D: with acc_scale a power of two,
    D * s + b in fp32 is the kernel's fmaf, so LRELU, PREGDN, KSI, RECON, RESID and QUANT must match bit for bit."""
    A, W, s = epi_operands(dev)
    R, cout = A[0].shape[0], W[0].shape[0]
    g = torch.Generator(device=dev).manual_seed(3)
    bias = (torch.rand(cout, generator=g, device=dev) - 0.5)
    D = model.debug_layer("raw", A, W, core=core)["f32"]
    v = D * f32(s, dev) + bias
    assert float(v.abs().max()) > 1.0 and float(v.abs().median()) > 0.05
    kw = dict(core=core, bias=bias, acc_scale=s)
    o = model.debug_layer("lrelu", A, W, **kw)
    assert_planes(o, torch.where(v > 0, v, v * f32(0.01, dev)), "lrelu")
    o = model.debug_layer("pregdn", A, W, **kw)
    assert torch.equal(bits(o["f32"]), bits(v)), "pregdn f32 plane"
    assert_planes(o, v * v, "pregdn")
    o = model.debug_layer("ksi", A, W, **kw)
    assert torch.equal(bits(o["f32"]), bits(v)), "ksi"
    for nc in (False, True):
        o = model.debug_layer("recon", A, W, no_clamp=nc, **kw)
        assert torch.equal(bits(o["f32"]), bits(v if nc else v.clamp(-0.5, 0.5))), f"recon no_clamp={nc}"
        res = torch.randn(R, cout, generator=g, device=dev) * 0.3
        o = model.debug_layer("resid", A, W, aux=res, no_clamp=nc, **kw)
        want = res + v
        assert torch.equal(bits(o["f32"]), bits(want if nc else want.clamp(-0.5, 0.5))), f"resid no_clamp={nc}"
    report(test="epilogue_exact", core=core, modes=["lrelu", "pregdn", "ksi", "recon", "resid"], R=R, K=[48, 192])


@pytest.mark.parametrize("table", ["geometric", "nongeometric"])
@pytest.mark.parametrize("core", ["simt", "tc", "pair_wide"])
def test_quant_ties_and_indexes(model, dev, core, table):
    """QUANT: symbols round half to even (ties of y - mean crafted exactly at k + 0.5 and one ulp either side), y_qnt =
    sym + mean in the hi/lo planes, and indexes equal to build_indexes at every table level, one ulp either side, the
    0.11 floor and beyond the last level; the non-geometric table (passed explicitly) forces the bisection fallback."""
    tab = get_scale_table() if table == "geometric" else nongeometric_table()
    A, W, s = epi_operands(dev)
    R, M = A[0].shape[0], W[0].shape[0]
    nz = 120                                     # rows [0, nz) of A are zero: y = 0 exactly there (bias 0)
    A = [a.clone() for a in A]
    for a in A:
        a[:nz] = 0
    D = model.debug_layer("raw", A, W, core=core)["f32"]
    y = D * f32(s, dev)
    g = torch.Generator(device=dev).manual_seed(21)
    means = torch.randn(R, M, generator=g, device=dev) * 3
    ties = torch.tensor([k + 0.5 for k in range(-4, 4)] + [1000.5, -1000.5], dtype=torch.float32)
    cand = torch.cat([ties, torch.nextafter(ties, f32([1e9], "cpu")), torch.nextafter(ties, f32([-1e9], "cpu"))])
    means[:nz] = -cand[torch.arange(nz * M) % cand.numel()].reshape(nz, M).to(dev)
    sc = crafted_scales(tab)
    scales = sc[torch.arange(R * M) % sc.numel()].reshape(R, M).to(dev)
    ksi = torch.cat([scales, means], dim=1)
    o = model.debug_layer("quant", A, W, core=core, aux=ksi, acc_scale=s,
                          scale_table=tab.to(dev) if table == "nongeometric" else None)
    d = y - means
    assert bool((d[:nz] - torch.floor(d[:nz]) == 0.5).sum() >= 8 * M // 2), "no exact ties were produced"
    sym = torch.round(d)
    assert torch.equal(o["sym"], sym.int()), f"symbols: {int((o['sym'] != sym.int()).sum())} differ from round-half-even"
    assert_planes(o, sym + means, "quant y_qnt")
    want = ref_index(scales, tab).to(dev)
    bad = int((o["idx"].int() != want).sum())
    assert bad == 0, f"{bad} QUANT indexes differ from build_indexes"
    ib, ih = model.debug_scale_index(sc.to(dev), tab.to(dev))
    want_sc = ref_index(sc, tab).to(dev)
    assert torch.equal(ib, want_sc), "decoder bisection (scale_to_index) differs from build_indexes"
    assert torch.equal(ih, want_sc), "decoder hinted lookup differs from build_indexes"
    report(test="quant", core=core, table=table, ties=int((d[:nz] - torch.floor(d[:nz]) == 0.5).sum()),
           crafted_scales=int(sc.numel()))


@pytest.mark.parametrize("core", ["simt", "tc", "ws", "pair_wide"])
def test_gdn_igdn_vs_fp64(model, dev, core):
    """GDN / IGDN: a * (beta + gamma a^2)^(-+1/2) in float64 from the core's own accumulator.  Bar 3 * 2^-22 |ref| + 2^-25:
    rsqrt.approx.ftz (2 ulp = 2^-22), the fmaf and the products (2^-24 each), the hi/lo output split (2^-22; 2^-25 when lo
    is subnormal).  |lo| must not exceed half an ulp of hi, as split_h16 leaves it (hi + lo itself may re-round the other way at a tie)."""
    g = torch.Generator(device=dev).manual_seed(8)
    R, C = 257, 192
    a = torch.randn(R, C, generator=g, device=dev) * 5
    gamma = 0.1 * torch.eye(C, device=dev) + (0.6 / C) * torch.rand(C, C, generator=g, device=dev)
    k = 9 - int(math.floor(math.log2(float(gamma.max()))))
    Wg, s = gamma * 2.0 ** k, 2.0 ** -k
    beta = 0.5 + torch.rand(C, generator=g, device=dev)
    sq = a * a
    D = model.debug_layer("raw", [sq], [Wg], core=core)["f32"]
    norm = D.double() * s + beta.double()
    worst = {}
    for mode, p in (("gdn", -0.5), ("igdn", 0.5)):
        o = model.debug_layer(mode, [sq], [Wg], core=core, bias=beta, aux=a, acc_scale=s)
        ref = a.double() * norm ** p
        got = o["hi"].double() + o["lo"].double()
        err = (got - ref).abs()
        bar = 3 * 2.0 ** -22 * ref.abs() + 2.0 ** -25
        ratio = float((err / bar).max())
        assert ratio <= 1.0, f"{mode}: error {ratio:.3f} x the bar"
        hi, lo = o["hi"].float(), o["lo"].float()
        ulp = torch.where(hi.abs() < 2.0 ** -14, torch.full_like(hi, 2.0 ** -24),
                          torch.exp2(torch.floor(torch.log2(hi.abs().clamp_min(2.0 ** -14))) - 10))
        assert bool((lo.abs() <= ulp / 2).all()), f"{mode}: lo exceeds half an ulp of hi (not a split_h16 pair)"
        worst[mode] = dict(ratio=round(ratio, 4), rel=float(f"{float((err / ref.abs().clamp_min(1e-30)).max()):.3e}"))
    report(test="gdn_igdn", core=core, worst=worst)


# ---- D. self-information -------------------------------------------------------------------------------------------
def test_selfinfo_vs_reference_formula(model, dev):
    """selfinfo_step_kernel against oracle.nets.self_information (the reference's fp32 formula) over |sym| 0..1e4 and
    scales 0.05..300: relative where the likelihood is well above the 1e-9 floor, the clamp value -log2(1e-9) (fp32,
    one ulp) where it is well below.  The float64 (scipy) error is reported alongside."""
    from scipy.special import erfc
    syms = torch.tensor([0, 1, -1, 2, 3, -5, 8, 13, 30, -100, 300, 1000, -3000, 10000], dtype=torch.int32)
    scales = torch.cat([torch.logspace(math.log10(0.05), math.log10(300), 60), torch.tensor([0.11, 0.1100001, 0.1099999])]).float()
    i, j = torch.meshgrid(torch.arange(scales.numel()), torch.arange(syms.numel()), indexing="ij")
    S, Y = scales[i.reshape(-1)], syms[j.reshape(-1)]
    n = (S.numel() + 15) // 16 * 16
    S = torch.cat([S, torch.ones(n - S.numel())]).reshape(-1, 16)
    Y = torch.cat([Y, torch.zeros(n - Y.numel(), dtype=torch.int32)]).reshape(-1, 16)
    ksi = torch.cat([S, torch.zeros_like(S)], dim=1)
    got = model.debug_selfinfo(ksi.to(dev), Y.to(dev)).cpu()
    ref = nets.self_information(Y, S)
    s64 = torch.clamp(S, min=0.11).double().numpy()        # max(s, 0.11f) as the kernel takes it
    v64 = Y.abs().double().numpy()
    up = 0.5 * erfc(-(0.5 - v64) / (s64 * math.sqrt(2)))
    lo = 0.5 * erfc(-(-0.5 - v64) / (s64 * math.sqrt(2)))
    lik = torch.from_numpy(up - lo)
    info64 = -torch.log2(torch.clamp(lik, min=1e-9))
    well = lik >= 1e-7
    clamped = lik <= 0.5e-9
    assert int(well.sum()) > 300 and int(clamped.sum()) > 50
    # erfcf / torch.erfc: a few ulp of upper and lower each; the subtraction scales it by upper / likelihood
    tol = 2.0 ** -20 * ref.abs().double() + 16 * 2.0 ** -24 * torch.from_numpy(up) / (lik.clamp(min=1e-300) * math.log(2))
    err = (got.double() - ref.double()).abs()
    assert bool((err[well] <= tol[well]).all()), f"self-information error {float((err / tol)[well].max()):.3f} x the bar"
    cap = -torch.log2(torch.tensor(1e-9, dtype=torch.float32))
    ulp = float(torch.nextafter(cap, torch.tensor(100.0)) - cap)
    assert bool(((got[clamped] - cap).abs() <= ulp).all()), "clamped likelihoods do not give -log2(1e-9)"
    assert bool(torch.isfinite(got).all())
    report(test="selfinfo", points=int(S.numel()), worst_vs_fp32_ratio=round(float((err / tol)[well].max()), 4),
           worst_abs_vs_fp64_bits=float(f"{float((got.double() - info64)[well].abs().max()):.3e}"),
           worst_rel_vs_fp64=float(f"{float(((got.double() - info64).abs() / info64.clamp(min=1e-6))[well].max()):.3e}"),
           clamped=int(clamped.sum()))


# ---- E. end to end with a non-geometric installed table ------------------------------------------------------------
def test_nongeometric_table_end_to_end(dev):
    """A checkpoint whose conditional_gaussian_model buffers carry a non-geometric scale table (CDFs built by the
    oracle's restatement of update_scale_table / pmf_to_quantized_cdf): encode / decode are exact for both containers,
    with the wave kernel on and off and with both decoder forms, and the indexes are build_indexes of the oracle's
    teacher-forced ksi except at rounding boundaries (scale within 2e-4 of a level, one step)."""
    cfgname = "B8_lowrate"
    cfg = lbic_b200.load_config(cfgname)
    tab = nongeometric_table()
    cdf, ln, off = nets.build_tables(tab)
    sd = weights.synth_state_dict(cfg, 1337)
    sd["conditional_gaussian_model._quantized_cdf"] = cdf
    sd["conditional_gaussian_model._cdf_length"] = ln
    sd["conditional_gaussian_model._offset"] = off
    sd["conditional_gaussian_model.scale_table"] = tab
    m = BlockBasedImgCompLossyNetv9(cfg, device=dev)
    m.load_state_dict(sd)
    img = weights.synth_images(2, 48, 72)
    x = nets.arrange_block_pixels_to_channel_dim(img - 0.5, 8).contiguous().to(dev)
    P = nets.effective_params(sd, cfg)
    P.scale_table = tab
    runs = {}
    try:
        for wave in (1, 0):
            m.set_option("wave", wave)
            for lanes in (1, 0):
                strings, zhat, sym, idx = m.compress_batch(x, lanes=lanes, return_symbols=True)
                for rows in (1, 1 << 30):
                    m.set_option("dec_thread_rows", rows)
                    zdec = m.decompress_batch(strings, x.shape, lanes=lanes)
                    assert torch.equal(zdec, zhat), f"wave={wave} lanes={lanes} dec_thread_rows={rows}: decode differs"
                runs[(wave, lanes)] = (sym, idx, zhat)
    finally:
        m.set_option("dec_thread_rows", 4096)
        m.set_option("wave", 1)
    sym, idx, zhat = runs[(1, 1)]
    for k, (s2, i2, z2) in runs.items():
        assert torch.equal(s2, sym) and torch.equal(i2, idx) and torch.equal(z2, zhat), f"{k} differs from wave=1 lanes=1"
    _, i_or, _, _, ksi = nets.whole_image_eval(P, x.cpu(), zhat.cpu())
    M = cfg.M
    sc = torch.clamp(ksi[:, :M], min=0.11).permute(0, 2, 3, 1)
    mis = i_or != idx.cpu().int()
    dist = ((sc[..., None] - tab).abs() / tab).min(dim=-1).values
    assert int((i_or - idx.cpu().int()).abs().max()) <= 1
    assert bool((dist[mis] < 2e-4).all()), f"index mismatches away from a table level: {float(dist[mis].max()):.2e}"
    assert int(mis.sum()) <= max(1, mis.numel() // 10000)
    assert len(set(idx.unique().tolist())) > 10
    report(test="nongeometric_e2e", symbols=int(idx.numel()), index_mismatches=int(mis.sum()),
           levels_used=len(set(idx.unique().tolist())), stream_bytes=len(m.compress_batch(x, lanes=1)[0][0]))
