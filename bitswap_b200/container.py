"""Variable-size images as chained 32x32 block streams + the reference's demo container format.

Reference: block tiling `extract_blocks` / `unextract_blocks` (benchmark_compress.py:20-39), the demo codec
(demo_compress.py:72-162 compress, :268-284 file format; demo_decompress.py:69-148, :216-227).  One image =
ONE ANS chain over its blocks (imagenetcrop_compress.py:127-210); different images are independent chains, so
a set of images is coded as a StreamSet with one stream per image: step t codes block t of every image that
has more than t blocks (images are ordered by block count so the active streams are always a prefix).

Container (np.uint32 array, what demo_compress.py saves with np.save):
    [ words that were actually borrowed or produced ..., head_lo, head_hi, nblocks, h, w ]
Blocks are fed CHW like the demo path does (demo_compress.py:120).  `hwc_quirk=True` reproduces
imagenetcrop_compress.py:130 instead, which flattens each [32,32,3] HWC block straight into the CHW model's input
(`torch.from_numpy(x).view(xdim)`) -- the layout behind the README's ImageNet-crop numbers.

Full-frame containers (`compress_images(..., crop=False)`) are an extension of that format.  The reference crops h and w
down to multiples of 32; with crop=False the image is tiled into ceil(h/32) x ceil(w/32) blocks instead, and the blocks
on the right and bottom edges are PARTIAL: only their valid (valid_rows x valid_cols) pixels are coded, the rest is the
edge-replicate fill both sides rebuild (BitSwapCodec.encode(extents=...)).  The header is unchanged in shape -- h and w
are the true sizes, nblocks = ceil(h/32) * ceil(w/32) -- so for sizes that are multiples of 32 the two formats are the
same container word for word, and decompress_images reads both.  A container with partial blocks cannot be read by the
reference's demo_decompress.py.  Partial blocks are not supported with `hwc_quirk=True`: that layout has no
rectangular valid region.
"""
import numpy as np
import torch

from .codec import BITSWAP
from .streams import StreamSet
from .synthetic import initial_words


def extract_blocks(arr, block_size=(32, 32)):
    """HWC uint8 image -> (blocks [n, 32, 32, C] row-major over the block grid, h, w) with h, w cropped down to
    multiples of the block size (benchmark_compress.py:20-31)."""
    bh, bw = block_size
    h, w, c = arr.shape
    h -= h % bh
    w -= w % bw
    arr = arr[:h, :w]
    blocks = arr.reshape(h // bh, bh, w // bw, bw, c).swapaxes(1, 2).reshape(-1, bh, bw, c)
    return blocks, h, w


def unextract_blocks(blocks, h, w):
    """Inverse of extract_blocks (benchmark_compress.py:35-39)."""
    n, bh, bw, c = blocks.shape
    return blocks.reshape(h // bh, w // bw, bh, bw, c).swapaxes(1, 2).reshape(h, w, c)


def extract_blocks_full(arr, block_size=(32, 32)):
    """HWC uint8 image -> (blocks [n, 32, 32, C] row-major over the ceil(h/32) x ceil(w/32) grid, extents int32 [n, 2]).
    Partial blocks are padded by edge replication (the fill the codec applies to their masked pixels anyway); extents
    holds each block's (valid_rows, valid_cols)."""
    bh, bw = block_size
    h, w, c = arr.shape
    nh, nw = -(-h // bh), -(-w // bw)
    arr = np.pad(arr, ((0, nh * bh - h), (0, nw * bw - w), (0, 0)), mode="edge")
    blocks = arr.reshape(nh, bh, nw, bw, c).swapaxes(1, 2).reshape(-1, bh, bw, c)
    return blocks, block_extents(h, w, block_size)


def unextract_blocks_full(blocks, h, w):
    """Inverse of extract_blocks_full: the blocks' valid pixels as the [h, w, C] image."""
    n, bh, bw, c = blocks.shape
    nh, nw = -(-h // bh), -(-w // bw)
    return blocks.reshape(nh, nw, bh, bw, c).swapaxes(1, 2).reshape(nh * bh, nw * bw, c)[:h, :w]


def block_extents(h, w, block_size=(32, 32)):
    """(valid_rows, valid_cols) of every block of an h x w image, row-major over the ceil grid: int32 [n, 2]."""
    bh, bw = block_size
    nh, nw = -(-h // bh), -(-w // bw)
    rows = np.minimum(h - bh * np.arange(nh), bh)
    cols = np.minimum(w - bw * np.arange(nw), bw)
    return np.stack(np.broadcast_arrays(rows[:, None], cols[None, :]), axis=-1).reshape(-1, 2).astype(np.int32)


def parse_container(c, hwc_quirk=False):
    """Container array -> (words, head, nblocks, h, w), validated before any device work (demo_decompress.py:216-222
    trusts its input file).  h, w >= 1 and nblocks = ceil(h/32) * ceil(w/32): for multiples of 32 this is the reference's
    rule, otherwise a full-frame container with partial edge blocks (not readable with hwc_quirk)."""
    c = np.asarray(c, dtype=np.uint32)
    if c.ndim != 1 or c.size < 5:
        raise ValueError(f"container too short ({c.size} words): needs at least head_lo, head_hi, nblocks, h, w")
    nblocks, h, w = int(c[-3]), int(c[-2]), int(c[-1])                                          # demo_decompress.py:216-219
    if h <= 0 or w <= 0 or nblocks != (-(-h // 32)) * (-(-w // 32)) or nblocks > (1 << 20):
        raise ValueError(f"inconsistent container header: nblocks={nblocks}, h={h}, w={w}")
    if hwc_quirk and (h % 32 or w % 32):
        raise ValueError(f"a {h}x{w} container has partial blocks, which hwc_quirk=True does not support")
    head = (int(c[-4]) << 32) | int(c[-5])                                                      # :222
    return c[:-5], head, nblocks, h, w


def _blocks_to_model(blocks, hwc_quirk):
    """[n,32,32,C] HWC blocks -> [n,C,32,32] model input."""
    n, bh, bw, c = blocks.shape
    return blocks.reshape(n, c, bh, bw) if hwc_quirk else blocks.transpose(0, 3, 1, 2)


def _model_to_blocks(x, hwc_quirk):
    n, c, bh, bw = x.shape
    return np.ascontiguousarray(x).reshape(n, bh, bw, c) if hwc_quirk else np.ascontiguousarray(x.transpose(0, 2, 3, 1))


def _tile(im, crop, hwc_quirk):
    """-> (blocks, h, w, extents or None) of one image; h, w are what the header records."""
    im = np.asarray(im)
    if crop:
        blocks, h, w = extract_blocks(im)
        return blocks, h, w, None
    h, w = im.shape[:2]
    if h < 1 or w < 1:
        raise ValueError("empty image")
    if hwc_quirk and (h % 32 or w % 32):
        raise ValueError(f"a {h}x{w} image has partial blocks, which hwc_quirk=True does not support")
    blocks, ext = extract_blocks_full(im)
    return blocks, h, w, ext


def _extents_dev(exts, order, nblk, device):
    """Per-step extents of the chains, [step, stream, 2] on the device, or None if every block is whole."""
    if all(e is None or bool(np.all(e == 32)) for e in exts):
        return None
    host = np.full((max(nblk), len(order), 2), 32, dtype=np.int32)
    for j, i in enumerate(order):
        if exts[i] is not None:
            host[:nblk[j], j] = exts[i]
    return torch.from_numpy(host).to(torch.device("cuda", device))


def compress_images(codec, images, excess_state_len=10000, seed=100, scheme=BITSWAP, hwc_quirk=False, words_per_block=1400,
                    crop=True):
    """images: list of HWC uint8 arrays.  Returns one container array per image.
    Every chain starts from the reference's initial state: `excess_state_len` random words drawn with
    np.random.seed(100) (demo_compress.py:113-115, :202).
    crop=True (default): the reference's demo format -- h and w are cropped down to multiples of 32 (images need at least
    one whole block).  crop=False: the whole image, any size >= 1x1, losslessly (partial edge blocks, module docstring)."""
    tiled = [_tile(im, crop, hwc_quirk) for im in images]
    order = sorted(range(len(images)), key=lambda i: (-tiled[i][0].shape[0], i))
    nblk = [tiled[i][0].shape[0] for i in order]
    n = len(images)
    w, head = initial_words(excess_state_len, seed=seed)
    # capacity: `words_per_block` words per 32x32 block (1400 = 14.6 bits/dim; 8 bits/dim of raw pixels is 768).  A chain
    # that still overflows is retried with twice the room instead of failing after the whole chain was coded.
    for attempt in range(4):
        ss = StreamSet(n, excess_state_len + (words_per_block << attempt) * max(nblk) + 64, device=codec.device)
        ss.fill(w, head)
        try:
            return _compress_chains(codec, ss, tiled, order, nblk, scheme, hwc_quirk)
        except OverflowError:
            if attempt == 3:
                raise
    raise AssertionError("unreachable")


def _compress_chains(codec, ss, tiled, order, nblk, scheme, hwc_quirk):
    n = len(order)
    # all blocks to the device once: [step t, stream j] = block t of the j-th largest image (CHW, demo_compress.py:120)
    C = tiled[order[0]][0].shape[-1]
    host = np.zeros((max(nblk), n, C, 32, 32), dtype=np.uint8)
    for j, i in enumerate(order):
        host[:nblk[j], j] = _blocks_to_model(tiled[i][0], hwc_quirk)
    dev = torch.from_numpy(host).to(torch.device("cuda", codec.device))
    ext = _extents_dev([t[3] for t in tiled], order, nblk, codec.device)
    for t in range(max(nblk)):
        active = sum(1 for b in nblk if b > t)
        codec.encode(ss, dev[t, :active].contiguous(), first=0, scheme=scheme,
                     extents=None if ext is None else ext[t, :active])
    torch.cuda.synchronize()
    ss.raise_on_error()
    words, offs, heads, _ = ss.export()
    lo = ss.min_words()                                       # never-borrowed initial words (demo_compress.py:137,160)
    out = [None] * n
    for j, i in enumerate(order):
        ws = words[offs[j] + lo[j]:offs[j + 1]]
        hd = int(heads[j])
        _, h, wd, _ = tiled[i]
        tail = np.array([hd & 0xffffffff, hd >> 32, nblk[j], h, wd], dtype=np.uint32)           # demo_compress.py:272-279
        out[i] = np.concatenate([ws.astype(np.uint32), tail])
    return out


def decompress_images(codec, containers, channels=3, scheme=BITSWAP, hwc_quirk=False, headroom_words=None):
    """Inverse of compress_images: list of container arrays -> list of HWC uint8 images (the sizes in the headers: the
    cropped sizes of a crop=True container, the full image of a crop=False one)."""
    meta = [parse_container(c, hwc_quirk) for c in containers]
    order = sorted(range(len(containers)), key=lambda i: (-meta[i][2], i))
    nblk = [meta[i][2] for i in order]
    n = len(containers)
    # The receiver pushes too (it returns the borrowed bits, cifar_compress.py:306-313): one block's worth of latents,
    # nz * zdim symbols at <= 31 bits each, can sit on the stack above the container's own length.
    if headroom_words is None:
        headroom_words = codec.cfg.nz * codec.cfg.zdim + 64
    ss = StreamSet(n, max(len(meta[i][0]) for i in order) + headroom_words, device=codec.device)
    ss.import_lists([[int(v) for v in meta[i][0]] + [meta[i][1]] for i in order])
    dev = torch.zeros((max(nblk), n, channels, 32, 32), dtype=torch.uint8, device=torch.device("cuda", codec.device))
    ext = _extents_dev([block_extents(m[3], m[4]) for m in meta], order, nblk, codec.device)
    for t in reversed(range(max(nblk))):
        active = sum(1 for b in nblk if b > t)
        codec.decode(ss, active, first=0, scheme=scheme, out=dev[t, :active],
                     extents=None if ext is None else ext[t, :active])
    if hasattr(codec, "join"):                                             # (free-running multi-lane codec: lanes -> current stream)
        codec.join()
    host = dev.cpu().numpy()                                               # one transfer for every block of every image
    blocks = [_model_to_blocks(host[:nblk[j], j], hwc_quirk) for j in range(n)]
    ss.raise_on_error()
    out = [None] * n
    for j, i in enumerate(order):
        out[i] = unextract_blocks_full(blocks[j], meta[i][3], meta[i][4])
    return out
