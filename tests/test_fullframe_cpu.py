"""Full-frame containers without a GPU: the ceil tiling and its inverse, the header rule, and the masked oracle recursion
(partial pixel blocks) on the CPU tiny model."""
import numpy as np
import pytest

from bitswap_b200 import synthetic
from bitswap_b200.config import preset
from bitswap_b200.container import extract_blocks_full, unextract_blocks_full, parse_container
from oracle import oracle as O
from fullframe_oracle import MaskedBitSwapOracle, fill_block


@pytest.mark.parametrize("h,w", [(1, 1), (31, 33), (100, 70), (64, 96), (224, 225)])
def test_full_tiling_roundtrip_and_extents(h, w):
    rs = np.random.RandomState(h * 1000 + w)
    img = rs.randint(0, 256, (h, w, 3)).astype(np.uint8)
    blocks, ext = extract_blocks_full(img)
    nh, nw = -(-h // 32), -(-w // 32)
    assert blocks.shape == (nh * nw, 32, 32, 3) and ext.shape == (nh * nw, 2) and ext.dtype == np.int32
    assert np.array_equal(unextract_blocks_full(blocks, h, w), img)
    for k, (vr, vc) in enumerate(ext):
        by, bx = divmod(k, nw)                                             # row-major over the block grid
        assert (vr, vc) == (min(32, h - 32 * by), min(32, w - 32 * bx))
        assert np.array_equal(blocks[k, :vr, :vc], img[32 * by:32 * by + vr, 32 * bx:32 * bx + vc])
        # the host padding is the codec's fill: x[min(y, vr-1)][min(x, vc-1)]
        chw = blocks[k].transpose(2, 0, 1)
        assert np.array_equal(fill_block(chw, (vr, vc)), chw)


def test_header_rule_for_partial_blocks():
    words = [7, 7]
    ok = [(1, 1, 1), (2, 31, 33), (12, 100, 70), (6, 64, 96), (56, 224, 225)]
    for nb, h, w in ok:
        _, head, nblocks, hh, ww = parse_container(np.array(words + [5, 0, nb, h, w], np.uint32))
        assert (head, nblocks, hh, ww) == (5, nb, h, w)
    for nb, h, w in [(1, 31, 33), (3, 31, 33), (0, 1, 1), (11, 100, 70), (1, 0, 5)]:
        with pytest.raises(ValueError):
            parse_container(np.array(words + [5, 0, nb, h, w], np.uint32))
    # hwc_quirk: whole blocks only
    parse_container(np.array(words + [5, 0, 6, 64, 96], np.uint32), hwc_quirk=True)
    with pytest.raises(ValueError):
        parse_container(np.array(words + [5, 0, 2, 31, 33], np.uint32), hwc_quirk=True)


def test_hwc_quirk_with_partial_blocks_is_refused_before_device_work():
    from bitswap_b200.container import compress_images, decompress_images
    with pytest.raises(ValueError):
        compress_images(None, [np.zeros((40, 64, 3), np.uint8)], crop=False, hwc_quirk=True)
    with pytest.raises(ValueError):
        decompress_images(None, [np.array([7, 7, 5, 0, 2, 40, 32], np.uint32)], hwc_quirk=True)


def _oracle():
    cfg = preset("tiny")
    sd = synthetic.synthetic_state_dict(cfg, seed=50, varied=True)
    zend, zcen = synthetic.synthetic_bins(cfg, seed=0)
    return cfg, MaskedBitSwapOracle(cfg, O.ModelOracle(cfg, sd), zend, zcen, coder="c", pmf="torch")


@pytest.mark.parametrize("scheme", ["bitswap", "bbans"])
def test_masked_oracle_roundtrip_and_neutral_extent(scheme):
    cfg, orc = _oracle()
    enc = orc.encode_image if scheme == "bitswap" else orc.encode_image_bbans
    dec = orc.decode_image if scheme == "bitswap" else orc.decode_image_bbans
    imgs = synthetic.synthetic_images(cfg, 2, seed=9)
    w, head = synthetic.initial_words(2000, seed=100)
    init = O.CState(w, head).to_list()
    extents = [(17, 29), (1, 1)]
    st = O.CState(w, head)
    for x, e in zip(imgs, extents):
        st = enc(st, x, extent=e)
    for x, e in reversed(list(zip(imgs, extents))):
        st, got = dec(st, extent=e)
        got = got.reshape(cfg.xs)
        vr, vc = e
        assert np.array_equal(got[:, :vr, :vc], x[:, :vr, :vc])          # valid pixels restored
        assert np.array_equal(got, fill_block(x, e))                       # masked pixels hold the fill
    assert st.to_list() == init
    # (32, 32) is the unmasked call, state for state
    a = enc(O.CState(w, head), imgs[0], extent=(32, 32)).to_list()
    b = enc(O.CState(w, head), imgs[0]).to_list()
    assert a == b
