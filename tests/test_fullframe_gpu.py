"""Partial pixel blocks on the device (BitSwapCodec.encode/decode(extents=...)) and full-frame containers
(compress_images(crop=False)): parity with the masked oracle recursion, invariance over every coder path, exact round
trips, and the bits the mask saves."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as O                      # noqa: E402  (checker only)
from fullframe_oracle import MaskedBitSwapOracle, fill_block   # noqa: E402
from bitswap_b200 import synthetic                   # noqa: E402
from bitswap_b200.config import preset               # noqa: E402
from bitswap_b200.model import Model                 # noqa: E402
from bitswap_b200.codec import BitSwapCodec, PipelinedCodec, Bins, BITSWAP, BBANS   # noqa: E402
from bitswap_b200.streams import StreamSet           # noqa: E402
from bitswap_b200._lib import lib, check             # noqa: E402

EXTENTS = [(32, 32), (1, 1), (32, 1), (1, 32), (17, 29)]


def _setup(name, B, cap, tc=False, varied=True):
    cfg = preset(name)
    sd = synthetic.synthetic_state_dict(cfg, seed=50, varied=varied)
    m = Model.from_config(cfg, max_batch=B, use_tensor_cores=tc).load_state_dict(sd)
    m.compress()
    zend, zcen = synthetic.synthetic_bins(cfg, seed=0)
    codec = BitSwapCodec(cfg, m, Bins(cfg, zend, zcen), B)
    return cfg, m, sd, zend, zcen, codec, StreamSet(B, cap)


def _states(B, seed):
    out = []
    for b in range(B):
        w, head = synthetic.initial_words(3000 + 11 * b, seed=seed + b)
        out.append([int(v) for v in w] + [head])
    return out


def _ext(extents):
    return torch.tensor(extents, dtype=torch.int32).cuda().contiguous()


def _oracle(cfg, m, sd, zend, zcen):
    orc = MaskedBitSwapOracle(cfg, O.ModelOracle(cfg, sd), zend, zcen, coder="c", pmf="cuda")

    def gpu_net(kind, level, given):
        f = m.infer(level) if kind == "infer" else m.generate(level)
        mu, sc = f(given.cuda())
        return mu.cpu(), sc.cpu()
    orc._net = gpu_net
    return orc


@pytest.mark.parametrize("name,scheme", [("tiny3", BITSWAP), ("tiny3", BBANS), ("tiny", BITSWAP)])
def test_masked_recursion_vs_oracle_and_roundtrip(name, scheme):
    """Device masked recursion against the masked oracle recursion (GPU nets injected, the reference's float64 table
    expression on torch-CUDA): EVERY stream's full state list bit-identical after each image of a 2-image chain, with the
    extents (32,32), (1,1), (32,1), (1,32), (17,29) in one batch.  Then decode: valid pixels exact, the fill in the masked
    ones, initial states restored."""
    B, nimg = len(EXTENTS), 2
    cfg, m, sd, zend, zcen, codec, ss = _setup(name, B, 1 << 14)
    imgs = synthetic.synthetic_images(cfg, B * nimg, seed=11).reshape(nimg, B, *cfg.xs)
    exts = [EXTENTS, EXTENTS[1:] + EXTENTS[:1]]                 # the second image of each chain gets another extent
    states = _states(B, 100)
    ss.import_lists(states)
    orc = _oracle(cfg, m, sd, zend, zcen)
    want = [O.CState.from_list(s) for s in states]
    enc = orc.encode_image if scheme == BITSWAP else orc.encode_image_bbans
    for xi in range(nimg):
        codec.encode(ss, torch.from_numpy(imgs[xi]).cuda(), scheme=scheme, extents=_ext(exts[xi]))
        ss.raise_on_error()
        got = ss.export_lists()
        for b in range(B):
            want[b] = enc(want[b], imgs[xi, b], extent=exts[xi][b])
            assert got[b] == want[b].to_list(), f"image {xi}, stream {b} (extent {exts[xi][b]}) differs from the oracle"
    for xi in reversed(range(nimg)):
        out = codec.decode(ss, B, scheme=scheme, extents=_ext(exts[xi])).cpu().numpy()
        for b in range(B):
            vr, vc = exts[xi][b]
            assert np.array_equal(out[b, :, :vr, :vc], imgs[xi, b, :, :vr, :vc])
            assert np.array_equal(out[b], fill_block(imgs[xi, b], (vr, vc)))
    ss.raise_on_error()
    assert ss.export_lists() == states


@pytest.mark.parametrize("scheme", [BITSWAP, BBANS])
def test_neutral_extents_are_the_unmasked_call(scheme):
    B = 4
    cfg, m, sd, zend, zcen, codec, ss = _setup("tiny3", B, 1 << 14)
    imgs = synthetic.synthetic_images(cfg, B, seed=13)
    states = _states(B, 200)
    res = []
    for ext in (None, _ext([(32, 32)] * B)):
        ss.import_lists(states)
        codec.encode(ss, torch.from_numpy(imgs).cuda(), scheme=scheme, extents=ext)
        ss.raise_on_error()
        res.append(ss.export_lists())
    assert res[0] == res[1]


def test_masked_batch_is_identical_on_every_coder_path():
    """Default two-phase affine kernels, generic rows (bsw_set_rows_mode(0)), fused kernels (set_two_phase(False)), overlap
    mode (set_dual_stream(True)) and a 3-lane free-running PipelinedCodec leave identical streams for the same masked
    batch, and each path decodes them back."""
    B = len(EXTENTS)
    cfg, m, sd, zend, zcen, codec, ss = _setup("tiny3", B, 1 << 14)
    pc = PipelinedCodec(cfg, sd, Bins(cfg, zend, zcen), B, lanes=3, use_tensor_cores=False, free_running=True)
    imgs = synthetic.synthetic_images(cfg, 2 * B, seed=17).reshape(2, B, *cfg.xs)
    ext = _ext(EXTENTS)
    states = _states(B, 300)
    paths = {
        "affine": (codec, lambda: None, lambda: None),
        "rows_mode0": (codec, lambda: check(lib().bsw_set_rows_mode(0)), lambda: check(lib().bsw_set_rows_mode(-1))),
        "fused": (codec, lambda: codec.set_two_phase(False), lambda: codec.set_two_phase(True)),
        "overlap": (codec, lambda: codec.set_dual_stream(True), lambda: codec.set_dual_stream(False)),
        "lanes3": (pc, lambda: None, lambda: None),
    }
    res = {}
    for name, (c, on, off) in paths.items():
        on()
        try:
            ss.import_lists(states)
            for xi in range(2):
                c.encode(ss, torch.from_numpy(imgs[xi]).cuda(), extents=ext)
            if hasattr(c, "join"):
                c.join()
            torch.cuda.synchronize()
            ss.raise_on_error()
            res[name] = ss.export_lists()
            for xi in (1, 0):
                out = c.decode(ss, B, extents=ext)
                if hasattr(c, "join"):
                    c.join()
                torch.cuda.synchronize()
                want = np.stack([fill_block(imgs[xi, b], EXTENTS[b]) for b in range(B)])
                assert np.array_equal(out.cpu().numpy(), want), name
            ss.raise_on_error()
            assert ss.export_lists() == states, name
        finally:
            off()
    for name in paths:
        assert res[name] == res["affine"], f"{name} differs from the default path"


def test_full_frame_containers_vs_oracle_demo_procedure():
    """compress_images(crop=False): exact round trip of the full images; every container equals the reference demo
    procedure run by the masked oracle over the ceil-tiled blocks (partial blocks masked); a 64x96 image gives the same
    container as with crop=True; a free-running multi-lane codec gives identical containers."""
    from bitswap_b200.container import compress_images, decompress_images, extract_blocks_full
    sizes = [(1, 1), (31, 45), (100, 70), (64, 96), (40, 129)]
    rs = np.random.RandomState(5)
    images = [rs.randint(0, 256, (h, w, 3)).astype(np.uint8) for h, w in sizes]
    cfg, m, sd, zend, zcen, codec, _ = _setup("tiny3", len(images), 64)
    conts = compress_images(codec, images, excess_state_len=3000, crop=False)
    orc = _oracle(cfg, m, sd, zend, zcen)
    for img, cont in zip(images, conts):
        blocks, ext = extract_blocks_full(img)
        wds, head = synthetic.initial_words(3000, seed=100)
        st = O.CState(wds, head)
        low = st.n
        pops = []
        orc.trace = pops
        for b, e in zip(blocks, ext):
            st = orc.encode_image(st, b.transpose(2, 0, 1), extent=tuple(int(v) for v in e))
        low = min([ln - 1 for tag, ln, _ in pops if tag.startswith("pop")] + [low])
        h, w = img.shape[:2]
        want = np.concatenate([st.words[low:st.n], np.array([st.head & 0xffffffff, st.head >> 32, len(blocks), h, w],
                                                            dtype=np.uint64)]).astype(np.uint32)
        assert np.array_equal(cont, want), f"{h}x{w}"
    back = decompress_images(codec, conts)
    for img, rec in zip(images, back):
        assert np.array_equal(rec, img)
    i64 = sizes.index((64, 96))
    assert np.array_equal(compress_images(codec, [images[i64]], excess_state_len=3000, crop=True)[0], conts[i64])
    pc = PipelinedCodec(cfg, sd, Bins(cfg, zend, zcen), len(images), lanes=3, use_tensor_cores=False, free_running=True)
    conts_pc = compress_images(pc, images, excess_state_len=3000, crop=False)
    assert all(np.array_equal(a, b) for a, b in zip(conts, conts_pc))
    back_pc = decompress_images(pc, conts_pc)
    assert all(np.array_equal(a, b) for a, b in zip(images, back_pc))


def test_masked_pixels_cost_nothing():
    """A 40x40 image coded full-frame against its edge-padded 64x64 version coded with crop=True.  Both arms feed the nets
    identical blocks (per-block clamping equals image-level clamping at the right and bottom edges); the padded arm also
    codes the 64*64*3 - 40*40*3 = 7488 padded subpixels.  With the random-init weights of the bench preset the pixel level
    costs about 8 bits/dim, so the masked container must be shorter by at least half of that: 7488 * 4 bits."""
    from bitswap_b200.container import compress_images, decompress_images
    cfg, m, sd, zend, zcen, codec, _ = _setup("imagenetcrop4", 1, 64, varied=False)
    img = np.random.RandomState(23).randint(0, 256, (40, 40, 3)).astype(np.uint8)
    padded = np.pad(img, ((0, 24), (0, 24), (0, 0)), mode="edge")
    masked = compress_images(codec, [img], excess_state_len=3000, crop=False)[0]
    naive = compress_images(codec, [padded], excess_state_len=3000, crop=True)[0]
    gap = 32 * (len(naive) - len(masked))
    print(f"40x40 full-frame: {32 * (len(masked) - 5)} bits; edge-padded 64x64 crop=True: {32 * (len(naive) - 5)} bits; "
          f"saved {gap} bits = {gap / 7488:.2f} bits per padded subpixel")
    assert gap >= 7488 * 4
    assert np.array_equal(decompress_images(codec, [masked])[0], img)


def test_bad_extents_flag_only_their_stream():
    """An extent of 0 or 33 flags that stream (raise_on_error raises); the other streams of the batch code and round-trip
    normally."""
    B = 4
    cfg, m, sd, zend, zcen, codec, ss = _setup("tiny3", B, 1 << 14)
    imgs = synthetic.synthetic_images(cfg, B, seed=29)
    extents = [(17, 29), (0, 5), (33, 32), (32, 32)]
    states = _states(B, 400)
    ss.import_lists(states)
    codec.encode(ss, torch.from_numpy(imgs).cuda(), extents=_ext(extents))
    with pytest.raises(IndexError):
        ss.raise_on_error()
    _, _, flags = ss.sizes()
    assert flags.tolist() == [0, 4, 4, 0]
    got = ss.export_lists()
    assert got[1] == states[1] and got[2] == states[2]               # flagged streams were not touched
    # the good streams are exactly what a batch of only good streams gives
    ss2 = StreamSet(2, 1 << 14)
    ss2.import_lists([states[0], states[3]])
    codec.encode(ss2, torch.from_numpy(imgs[[0, 3]]).cuda(), extents=_ext([extents[0], extents[3]]))
    ss2.raise_on_error()
    assert ss2.export_lists() == [got[0], got[3]]
    out = codec.decode(ss, B, extents=_ext(extents)).cpu().numpy()
    for b in (0, 3):
        assert np.array_equal(out[b], fill_block(imgs[b], extents[b]))
    _, _, flags = ss.sizes()
    assert flags.tolist() == [0, 4, 4, 0]
    back = ss.export_lists()
    assert back[0] == states[0] and back[3] == states[3]
