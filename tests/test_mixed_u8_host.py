"""One call over 8-bit host images of different sizes (lbic_encode_images_u8_host_mixed /
lbic_decode_images_u8_host_mixed): every image must come out exactly as the equal-size 8-bit calls code it alone, with
both containers, both topology families and any number of copy bands."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import lbic_b200
from lbic_b200 import _lib, weights
from lbic_b200.net import BlockBasedImgCompLossyNetv9

pytestmark = pytest.mark.gpu

TOPOLOGIES = ["B8_lowrate", "B16_lowrate", "B8_highrate", "B4_highrate"]
# smaller than one block, portrait next to landscape, one far larger than the rest; no size a multiple of B
SIZES = [(1, 1), (3, 70), (70, 3), (45, 29), (29, 45), (13, 21), (203, 171)]


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


def u8_images(sizes, seed=5):
    return [weights.synth_image_u8(H, W, seed=seed + i) for i, (H, W) in enumerate(sizes)]


def singles(m, imgs, lanes):
    out = []
    for a in imgs:
        s, r = m.compress_images_u8(a[None], lanes=lanes, return_recon=True)
        out.append((s[0], r[0]))
    return out


def assert_mixed_equals_singles(m, imgs, lanes, ref=None):
    ref = ref if ref is not None else singles(m, imgs, lanes)
    streams, recs = m.compress_images_u8_mixed(imgs, lanes=lanes, return_recon=True)
    for i, (s, r) in enumerate(ref):
        assert streams[i] == s, f"image {i} {imgs[i].shape}: stream differs"
        assert np.array_equal(recs[i], r), f"image {i}: reconstruction differs"
    dec = m.decompress_images_u8_mixed(streams, [a.shape[1:] for a in imgs], lanes=lanes)
    for i, (s, r) in enumerate(ref):
        alone = m.decompress_images_u8([s], *imgs[i].shape[1:], lanes=lanes)[0]
        assert np.array_equal(dec[i], alone) and np.array_equal(dec[i], r), f"image {i}: decode differs"
    return ref


@pytest.mark.parametrize("cfgname", TOPOLOGIES)
@pytest.mark.parametrize("lanes", [1, 0])
def test_each_image_as_if_alone(dev, cfgname, lanes):
    m = model(cfgname, dev)
    assert_mixed_equals_singles(m, u8_images(SIZES), lanes)


def test_matches_compress_batch_on_reference_tensors(dev):
    """The streams equal compress_batch(list) of the fp32 block tensors built as eval_model builds them (ToTensor as a
    true division on the CPU, -0.5, replicate padding, space-to-depth), and the 8-bit images save_image's quantisation."""
    from lbic_b200.layout import arrange_block_pixels_to_channel_dim, arrange_channel_dim_to_block_pixels
    m = model("B8_lowrate", dev)
    B = m.B
    imgs = u8_images(SIZES, seed=17)
    xs = []
    for a in imgs:
        x = (torch.from_numpy(a[None]).float().div(255) - 0.5).to(dev)
        H, W = a.shape[1:]
        xp = F.pad(x, (0, (-W) % B, 0, (-H) % B), mode="replicate")
        xs.append(arrange_block_pixels_to_channel_dim(xp, B).contiguous())
    for lanes in (1, 0):
        want_s, zs = m.compress_batch(xs, lanes=lanes)
        got_s, recs = m.compress_images_u8_mixed(imgs, lanes=lanes, return_recon=True)
        assert got_s == want_s
        for a, z, r in zip(imgs, zs, recs):
            H, W = a.shape[1:]
            rec = arrange_channel_dim_to_block_pixels(z, B)[:, :, :H, :W] + 0.5
            assert np.array_equal(r, rec.mul(255).add_(0.5).clamp_(0, 255).to(torch.uint8).cpu().numpy()[0])


def test_band_counts(dev):
    m = model("B8_highrate", dev)
    imgs = u8_images(SIZES, seed=23)
    tallest = max(-(-H // m.B) for H, _ in SIZES)
    try:
        for lanes in (0, 1):
            ref = None
            for bands in (1, 2, 16, tallest + 5):
                m.set_option("host_bands", bands)
                got = m.compress_images_u8_mixed(imgs, lanes=lanes, return_recon=True)
                dec = m.decompress_images_u8_mixed(got[0], [a.shape[1:] for a in imgs], lanes=lanes)
                if ref is None:
                    ref = (got, dec)
                    assert_mixed_equals_singles(m, imgs, lanes)
                assert got[0] == ref[0][0], f"bands={bands}"
                assert all(np.array_equal(a, b) for a, b in zip(got[1], ref[0][1]))
                assert all(np.array_equal(a, b) for a, b in zip(dec, ref[1]))
    finally:
        m.set_option("host_bands", 16)


def test_throughput_regime(dev):
    """64 images of three shapes: steps of more than flow_min_rows rows, default options."""
    m = model("B8_lowrate", dev)
    sizes = [(509, 765), (765, 509), (381, 637)] * 21 + [(509, 765)]
    imgs = u8_images(sizes, seed=31)
    streams, recs = m.compress_images_u8_mixed(imgs, lanes=0, return_recon=True)
    dec = m.decompress_images_u8_mixed(streams, sizes, lanes=0)
    for i in (0, 1, 2, 31, 63):
        s, r = m.compress_images_u8(imgs[i][None], lanes=0, return_recon=True)
        assert streams[i] == s[0] and np.array_equal(recs[i], r[0]) and np.array_equal(dec[i], r[0])


def test_equal_size_list(dev):
    m = model("B8_lowrate", dev)
    imgs = u8_images([(61, 83)] * 4, seed=41)
    for lanes in (1, 0):
        s_eq, r_eq = m.compress_images_u8(np.stack(imgs), lanes=lanes, return_recon=True)
        s_mx, r_mx = m.compress_images_u8_mixed(imgs, lanes=lanes, return_recon=True)
        assert s_mx == s_eq and all(np.array_equal(a, b) for a, b in zip(r_mx, r_eq))
        d_mx = m.decompress_images_u8_mixed(s_mx, [(61, 83)] * 4, lanes=lanes)
        assert np.array_equal(np.stack(d_mx), m.decompress_images_u8(s_eq, 61, 83, lanes=lanes))


def test_errors(dev):
    m = model("B8_lowrate", dev)
    L = _lib.lib()
    h = m._need()
    sizes = [(13, 21), (45, 70), (5, 5)]
    imgs = u8_images(sizes, seed=51)
    packed = np.concatenate([a.reshape(-1) for a in imgs])
    cap = (max(m.stream_bound(-(-H // m.B), -(-W // m.B), 1) for H, W in sizes) + 3) // 4 * 4
    out = np.zeros((3, cap), dtype=np.uint8)
    lens = np.zeros(3, dtype=np.uint32)
    INVALID, OVERFLOW = -1, -6

    def arr(v):
        return (ctypes.c_int * len(v))(*v) if v is not None else None

    def enc(n, H, W, lanes=1, c=cap):
        return L.lbic_encode_images_u8_host_mixed(h, packed.ctypes.data, n, arr(H), arr(W), None, out.ctypes.data, c,
                                                  lens.ctypes.data, lanes)

    def dec(n, H, W, ln, lanes=1, c=cap):
        img = np.empty(packed.size, dtype=np.uint8)
        return L.lbic_decode_images_u8_host_mixed(h, out.ctypes.data, ln.ctypes.data, c, n, arr(H), arr(W),
                                                  img.ctypes.data, lanes)
    Hs, Ws = [s[0] for s in sizes], [s[1] for s in sizes]
    assert enc(0, Hs, Ws) == INVALID
    assert enc(3, None, Ws) == INVALID and enc(3, Hs, None) == INVALID
    assert enc(3, [13, 0, 5], Ws) == INVALID and enc(3, Hs, [21, 70, -1]) == INVALID
    assert enc(3, Hs, Ws, lanes=2) == INVALID
    assert enc(3, Hs, Ws, c=cap - 2) == INVALID
    big = 1 << 30                                      # beyond the block limit of the mixed calls
    assert enc(3, [big, big, 5], [big, big, 5]) == INVALID
    assert b"too large" in L.lbic_last_error()
    top = 2 ** 31 - 1                                  # 3 * sum H W of two such images exceeds 2^64 bytes
    assert enc(3, [top, top, 5], [top, top, 5]) == INVALID
    assert b"address space" in L.lbic_last_error()
    assert enc(3, Hs, Ws) == 0
    good = lens.copy()
    assert dec(3, Hs, Ws, good) == 0
    assert dec(3, Hs, Ws, good, lanes=2) == INVALID and dec(0, Hs, Ws, good) == INVALID
    assert dec(3, None, Ws, good) == INVALID and dec(3, Hs, Ws, good, c=cap - 2) == INVALID
    too_long = good.copy()
    too_long[1] = cap + 4
    assert dec(3, Hs, Ws, too_long) == INVALID
    # a stream_cap that fits every image but one: LBIC_ERR_OVERFLOW, and the others' lengths are their own
    alone = [s for s, _ in singles(m, imgs, 1)]
    small = (max(len(alone[0]), len(alone[2])) + 3) // 4 * 4
    assert small < len(alone[1])
    assert enc(3, Hs, Ws, c=small) == OVERFLOW
    assert lens[0] == len(alone[0]) and lens[2] == len(alone[2]) and lens[1] == 0xFFFFFFFF
    # one corrupted lane container among valid ones
    streams, _ = m.compress_images_u8_mixed(imgs, lanes=0)
    bad = [streams[0], bytes([streams[1][0] ^ 0xFF]) + streams[1][1:], streams[2]]
    with pytest.raises(RuntimeError, match="malformed"):
        m.decompress_images_u8_mixed(bad, sizes, lanes=0)


@pytest.mark.parametrize("lanes", [1, 0])
def test_word_rows_after_unaligned_offsets(dev, lanes):
    """Images whose width is a multiple of 4 placed at packed byte offsets that are not (3 * sum H_j W_j after odd
    sizes): their 8-bit rows are written byte by byte where a 4-byte store would be misaligned."""
    m = model("B8_lowrate", dev)
    sizes = [(1, 1), (64, 96), (3, 5), (333, 501), (40, 768), (7, 9), (24, 32)]
    offs = np.cumsum([0] + [3 * H * W for H, W in sizes])[:-1]
    assert any(o % 4 and W % 4 == 0 for o, (H, W) in zip(offs, sizes))
    assert_mixed_equals_singles(m, u8_images(sizes, seed=71), lanes)


def test_image_codec_files(dev, tmp_path):
    from PIL import Image
    from lbic_b200.codec import ImageCodec
    m = model("B8_lowrate", dev)
    sizes = [(203, 261), (161, 333), (64, 96), (7, 5)]
    paths = []
    for i, (H, W) in enumerate(sizes):
        p = str(tmp_path / f"in{i}.png")
        Image.fromarray(np.ascontiguousarray(weights.synth_image_u8(H, W, seed=61 + i).transpose(1, 2, 0)), "RGB").save(p)
        paths.append(p)
    for lanes in (1, 0):
        codec = ImageCodec(m, lanes=lanes)
        blobs = codec.encode_files(paths)
        assert blobs == [codec.encode_file(p) for p in paths]
        outs = [str(tmp_path / f"out{lanes}_{i}.png") for i in range(len(paths))]
        codec.decode_to_files(blobs, outs)
        for blob, o, rec in zip(blobs, outs, codec.decode_many(blobs)):
            want = rec[0].mul(255).add_(0.5).clamp_(0, 255).to(torch.uint8).permute(1, 2, 0).cpu().numpy()
            with Image.open(o) as im:
                assert np.array_equal(np.asarray(im.convert("RGB")), want)
    b1 = ImageCodec(m, lanes=1).encode_files(paths[:1])[0]
    b0 = ImageCodec(m, lanes=0).encode_files(paths[1:2])[0]
    with pytest.raises(ValueError):
        ImageCodec(m).decode_to_files([b1, b0], [str(tmp_path / "x.png"), str(tmp_path / "y.png")])
    other = ImageCodec(model("B8_highrate", dev)).encode_files(paths[2:3])[0]
    with pytest.raises(ValueError):
        ImageCodec(m).decode_to_files([b1, other], [str(tmp_path / "x.png"), str(tmp_path / "y.png")])
