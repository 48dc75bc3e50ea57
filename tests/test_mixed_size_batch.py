"""One encode / decode call over images of different sizes (lbic_encode_mixed / lbic_decode_mixed): every image must
come out exactly as the single-image calls code it, in every launch form, with both containers and both topology
families."""
import ctypes

import pytest
import torch

import lbic_b200
from lbic_b200 import _lib, weights
from lbic_b200.net import BlockBasedImgCompLossyNetv9

pytestmark = pytest.mark.gpu

TOPOLOGIES = ["B8_lowrate", "B16_lowrate", "B8_highrate", "B4_highrate"]
# degenerate grids (1x1, 1xW, Hx1), portrait next to landscape, and one grid far larger than the rest
MIX = [(1, 1), (1, 7), (6, 1), (5, 9), (9, 4), (2, 3), (14, 21)]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


_models = {}


def model(cfgname, dev):
    if cfgname not in _models:
        cfg = lbic_b200.load_config(cfgname)
        m = BlockBasedImgCompLossyNetv9(cfg, device=dev)
        m.load_state_dict(weights.synth_state_dict(cfg, 1337, harsh=False))
        m.update(force=True)
        _models[cfgname] = m
    return _models[cfgname]


def block_images(m, shapes, dev, seed=11):
    B = m.B
    xs = []
    for i, (hb, wb) in enumerate(shapes):
        img = weights.synth_images(1, hb * B, wb * B, seed0=seed + i)
        xs.append(lbic_b200.arrange_block_pixels_to_channel_dim((img - 0.5).to(dev), B).contiguous())
    return xs


def singles(m, xs, lanes):
    """(streams, zhat, sym, idx) of each image coded alone."""
    out = []
    for x in xs:
        s, z, sy, ix = m.compress_batch(x, lanes=lanes, return_symbols=True)
        out.append((s[0], z, sy, ix))
    return out


def assert_mixed_equals_singles(m, xs, lanes, ref=None):
    ref = ref if ref is not None else singles(m, xs, lanes)
    streams, zs, sy, ix = m.compress_batch(xs, lanes=lanes, return_symbols=True)
    shapes = [tuple(x.shape[2:]) for x in xs]
    for i in range(len(xs)):
        assert streams[i] == ref[i][0], f"image {i} {shapes[i]}: stream differs"
        assert torch.equal(zs[i], ref[i][1]) and torch.equal(sy[i], ref[i][2]) and torch.equal(ix[i], ref[i][3])
    o = m.encode_device_mixed(xs, lanes=lanes)
    dz, dsym = m.decode_device_mixed(o.streams, o.lens, shapes, lanes=lanes, want_symbols=True)
    m.check_errors()
    for i in range(len(xs)):
        alone = m.decompress_batch([ref[i][0]], xs[i].shape, lanes=lanes)
        assert torch.equal(dz[i], alone) and torch.equal(dz[i], ref[i][1]), f"image {i}: decode differs"
        assert torch.equal(dsym[i], ref[i][2])
    return ref


@pytest.mark.parametrize("cfgname", TOPOLOGIES)
@pytest.mark.parametrize("lanes", [1, 0])
def test_each_image_as_if_alone(dev, cfgname, lanes):
    m = model(cfgname, dev)
    shapes = MIX + ([(7, 1)] if lbic_b200.load_config(cfgname).KS[1] == 3 else [])
    assert_mixed_equals_singles(m, block_images(m, shapes, dev), lanes)


def test_every_launch_form(dev):
    """Each form against the single-image calls under the same options (the contract of the mixed calls)."""
    m = model("B8_lowrate", dev)
    xs = block_images(m, MIX, dev, seed=3)
    forms = [("flow", dict(flow=0)), ("single_cta", dict(flow=1, flow_min_rows=1, flow_pair_min_rows=1 << 30)),
             ("pair", dict(flow=2)), ("ws0", dict(ws=0, flow=0))]
    launches = {}
    try:
        for name, opts in forms:
            for k, v in opts.items():
                m.set_option(k, v)
            for lanes in (0, 1):
                ref = singles(m, xs, lanes)           # the single-image calls with the same options
                l0 = m.launch_count()
                assert_mixed_equals_singles(m, xs, lanes, ref)
                launches[name] = launches.get(name, 0) + m.launch_count() - l0
            m.set_option("flow", 1); m.set_option("flow_min_rows", 2560); m.set_option("flow_pair_min_rows", 8192)
            m.set_option("ws", 1)
        assert launches["single_cta"] < launches["flow"] and launches["pair"] < launches["flow"], launches
        small = block_images(m, [(1, 1), (3, 5), (4, 2)], dev, seed=9)
        m.set_gemm_core("simt")
        for lanes in (0, 1):
            assert_mixed_equals_singles(m, small, lanes)
    finally:
        m.set_gemm_core("tcgen05")
        m.set_option("flow", 1); m.set_option("flow_min_rows", 2560); m.set_option("flow_pair_min_rows", 8192)
        m.set_option("ws", 1)


def test_throughput_regime(dev):
    """64 images of three shapes: steps of more than flow_min_rows rows, default options."""
    m = model("B8_lowrate", dev)
    shapes = [(64, 96), (96, 64), (48, 80)] * 21 + [(64, 96)]
    xs = block_images(m, shapes, dev, seed=21)
    streams, zs, sy, ix = m.compress_batch(xs, lanes=0, return_symbols=True)
    o = m.encode_device_mixed(xs, lanes=0)
    dz = m.decode_device_mixed(o.streams, o.lens, [s for s in shapes], lanes=0)
    m.check_errors()
    for i in (0, 1, 2, 31, 63):
        s, z, a, b = m.compress_batch(xs[i], lanes=0, return_symbols=True)
        assert streams[i] == s[0] and torch.equal(zs[i], z) and torch.equal(sy[i], a) and torch.equal(ix[i], b)
        assert torch.equal(dz[i], z)


def test_wave_kernel_not_taken(dev):
    m = model("B8_lowrate", dev)
    shapes = [(3, 5), (4, 4)]
    xs = block_images(m, shapes, dev, seed=31)
    m.set_option("wave", 1)
    ref = singles(m, xs, 0)
    l0 = m.launch_count()
    got = m.compress_batch(xs, lanes=0, return_symbols=True)
    n_steps = max(w + 2 * (h - 1) for h, w in shapes)
    assert m.launch_count() - l0 >= n_steps           # the wave path would need fewer than 20 launches
    assert all(got[0][i] == ref[i][0] and torch.equal(got[1][i], ref[i][1]) for i in range(2))
    # an equal-size list gives what the equal-size tensor call gives
    eq = block_images(m, [(4, 6)] * 3, dev, seed=41)
    s_list, z_list = m.compress_batch(eq, lanes=1)
    s_t, z_t = m.compress_batch(torch.cat(eq), lanes=1)
    assert s_list == s_t and torch.equal(torch.cat(z_list), z_t)


def test_errors(dev):
    m = model("B8_lowrate", dev)
    L = _lib.lib()
    h = m._need()
    shapes = [(2, 3), (6, 9), (1, 1)]
    xs = block_images(m, shapes, dev, seed=51)
    x = torch.cat([t.reshape(-1) for t in xs])
    z = torch.empty_like(x)
    cap = 4 * 1024
    out = torch.empty(3, cap, dtype=torch.uint8, device=dev)
    lens = torch.zeros(3, dtype=torch.int32, device=dev)

    def enc(n, hb, wb, lanes=1, c=cap):
        H = (ctypes.c_int * 3)(*hb) if hb is not None else None
        W = (ctypes.c_int * 3)(*wb) if wb is not None else None
        return L.lbic_encode_mixed(h, x.data_ptr(), n, H, W, z.data_ptr(), None, None, out.data_ptr(), c,
                                   lens.data_ptr(), lanes, m._stream())
    hb, wb = [s[0] for s in shapes], [s[1] for s in shapes]
    INVALID = -1
    assert enc(0, hb, wb) == INVALID
    assert enc(3, [2, 0, 1], wb) == INVALID and enc(3, hb, [3, 9, -1]) == INVALID
    assert enc(3, None, wb) == INVALID and enc(3, hb, None) == INVALID
    assert enc(3, hb, wb, lanes=2) == INVALID
    # a stream_cap that holds the streams of images 0 and 2 but not that of image 1: only image 1's length is
    # 0xFFFFFFFF, the other two are coded as if alone
    alone = [s[0] for s in singles(m, xs, 1)]
    small = (max(len(alone[0]), len(alone[2])) + 3) // 4 * 4
    assert small < len(alone[1])
    assert enc(3, hb, wb, lanes=1, c=small) == 0
    with pytest.raises(RuntimeError, match="stream_cap"):
        m.check_errors()
    got = lens.cpu().numpy().astype("uint32")
    assert got[1] == 0xFFFFFFFF and got[0] == len(alone[0]) and got[2] == len(alone[2])
    host = out.reshape(-1).cpu().numpy()                # slot i starts at i * stream_cap
    assert host[: got[0]].tobytes() == alone[0] and host[2 * small: 2 * small + got[2]].tobytes() == alone[2]
    # one corrupted lane container among valid ones
    o = m.encode_device_mixed(xs, lanes=0)
    m.check_errors()
    o.streams[1, 0] ^= 0xFF
    m.decode_device_mixed(o.streams, o.lens, shapes, lanes=0)
    with pytest.raises(RuntimeError, match="malformed"):
        m.check_errors()


def test_image_codec_encode_many_decode_many(dev):
    from lbic_b200.codec import ImageCodec
    m = model("B8_lowrate", dev)
    sizes = [(203, 261), (161, 333), (64, 96)]
    imgs = [weights.synth_images(1, H, W, seed0=61 + i)[0] for i, (H, W) in enumerate(sizes)]
    for lanes in (1, 0):
        codec = ImageCodec(m, lanes=lanes)
        blobs = codec.encode_many(imgs)
        recs = codec.decode_many(blobs)
        for img, blob, rec in zip(imgs, blobs, recs):
            assert blob == codec.encode(img)
            assert torch.equal(rec, codec.decode(blob))
    b1 = ImageCodec(m, lanes=1).encode(imgs[0])
    b0 = ImageCodec(m, lanes=0).encode(imgs[1])
    with pytest.raises(ValueError):
        ImageCodec(m).decode_many([b1, b0])
    other = model("B8_highrate", dev)
    with pytest.raises(ValueError):
        ImageCodec(m).decode_many([b1, ImageCodec(other).encode(imgs[2])])
