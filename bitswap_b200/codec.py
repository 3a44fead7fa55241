"""Batched, device-resident Bit-Swap / BB-ANS codec (host-side handle of `bsw_codec`).

Replaces the sender/receiver loop bodies of the reference's compress()
(cifar_compress.py:175-250 and :283-352): one call codes one image per stream for
a whole batch of independent chains; the ANS state never leaves the GPU between
latent levels.  Chain more images onto the same streams by calling again.
"""
import ctypes

import numpy as np
import torch

from ._lib import lib, check, cuda_stream_ptr, device_index, on_device
from .config import CodecConfig
from .model import Model
from .streams import StreamSet

BITSWAP, BBANS = 0, 1


class Bins:
    """Device copy of the discretisation tables (zendpoints [nz,zdim,2^q-1], zcentres [nz,zdim,2^q],
    the layout discretize() returns, discretization.py:99)."""

    def __init__(self, cfg: CodecConfig, zendpoints, zcentres, device=None):
        self.device = device_index(device)
        ze = np.ascontiguousarray(zendpoints.detach().cpu().numpy() if torch.is_tensor(zendpoints) else zendpoints, dtype=np.float64)
        zc = np.ascontiguousarray(zcentres.detach().cpu().numpy() if torch.is_tensor(zcentres) else zcentres, dtype=np.float64)
        assert ze.shape == (cfg.nz, cfg.zdim, cfg.zsupport - 1) and zc.shape == (cfg.nz, cfg.zdim, cfg.zsupport)
        self._h = ctypes.c_void_p()
        with on_device(self.device):
            check(lib().bsw_bins_create(ctypes.byref(self._h), cfg.nz, cfg.zdim, cfg.quantbits, cfg.xdim, ze.ctypes.data, zc.ctypes.data))

    def level_is_uniform(self, level):
        """True if every endpoint row of latent level `level` (-1: the pixel row) is a uniform grid (affine-row kernels)."""
        return bool(lib().bsw_bins_level_is_uniform(self._h, int(level)))

    @property
    def handle(self):
        return self._h

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                lib().bsw_bins_destroy(h)
            except Exception:
                pass
            self._h = None


class BitSwapCodec:
    def __init__(self, cfg: CodecConfig, model: Model, bins: Bins, max_batch: int):
        self.cfg, self.model, self.bins, self.max_batch = cfg, model, bins, int(max_batch)
        self.device = model.device
        if bins.device != self.device:
            raise ValueError(f"model is on cuda:{model.device} but the bin tables are on cuda:{bins.device}")
        self._h = ctypes.c_void_p()
        with on_device(self.device):
            check(lib().bsw_codec_create(ctypes.byref(self._h), model.handle, bins.handle, self.max_batch))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                lib().bsw_codec_destroy(h)
            except Exception:
                pass
            self._h = None

    def encode(self, streams: StreamSet, x: torch.Tensor, first=0, scheme=BITSWAP, extents=None):
        """x: uint8 CUDA tensor [count, C, 32, 32]; pushes one image onto each of `count` streams. Async.

        extents: None (whole blocks) or a contiguous int32 CUDA tensor [count, 2] of (valid_rows, valid_cols), each in
        [1, 32]: partial blocks.  Only pixels (y, x) with y < valid_rows and x < valid_cols are coded; the others are
        replaced by the edge-replicate fill before the nets see the block.  An extent outside [1, 32] flags its stream
        (StreamSet.raise_on_error) and leaves the other streams alone."""
        assert x.is_cuda and x.dtype == torch.uint8 and x.is_contiguous()
        self._same_device(streams, x)
        count = x.shape[0]
        ext = self._extents_ptr(extents, count)
        with on_device(self.device):
            if ext is None:
                check(lib().bsw_codec_encode(self._h, streams.handle, first, count, x.data_ptr(), scheme, cuda_stream_ptr()))
            else:
                check(lib().bsw_codec_encode_ext(self._h, streams.handle, first, count, x.data_ptr(), ext, scheme, cuda_stream_ptr()))

    def _extents_ptr(self, extents, count):
        if extents is None:
            return None
        if not (torch.is_tensor(extents) and extents.is_cuda and extents.dtype == torch.int32 and extents.is_contiguous()
                and tuple(extents.shape) == (count, 2)):
            raise ValueError(f"extents: need a contiguous int32 CUDA tensor of shape ({count}, 2)")
        if extents.device.index != self.device:
            raise ValueError(f"codec is on cuda:{self.device}; extents on {extents.device}")
        return extents.data_ptr()

    def _same_device(self, streams, x=None):
        if streams.device != self.device or (x is not None and x.device.index != self.device):
            raise ValueError(f"codec is on cuda:{self.device}; streams on cuda:{streams.device}"
                             + (f", pixels on {x.device}" if x is not None else ""))

    def decode(self, streams: StreamSet, count: int, first=0, scheme=BITSWAP, out=None, extents=None):
        """Pops one image from each stream; returns uint8 CUDA tensor [count, C, 32, 32]. Async.
        extents: as for encode() (the same values the images were encoded with); masked pixels come back as the fill."""
        if out is None:
            out = torch.empty((count,) + tuple(self.cfg.xs), dtype=torch.uint8, device=torch.device("cuda", self.device))
        if not (out.is_cuda and out.dtype == torch.uint8 and out.is_contiguous() and out.numel() >= count * int(np.prod(self.cfg.xs))):
            raise ValueError("decode(out=...): need a contiguous uint8 CUDA tensor with room for `count` images")
        self._same_device(streams, out)
        ext = self._extents_ptr(extents, count)
        with on_device(self.device):
            if ext is None:
                check(lib().bsw_codec_decode(self._h, streams.handle, first, count, out.data_ptr(), scheme, cuda_stream_ptr()))
            else:
                check(lib().bsw_codec_decode_ext(self._h, streams.handle, first, count, out.data_ptr(), ext, scheme, cuda_stream_ptr()))
        return out

    @property
    def last_launches(self):
        return int(lib().bsw_codec_last_launches(self._h))

    CATEGORIES = ("misc", "conv_in", "conv_dense3x3", "conv_dense5x5", "conv_head", "pop_z", "push_z", "pop_x",
                  "push_x", "prior", "rows_z", "rows_x")

    def set_dual_stream(self, on=True):
        """True: overlap mode -- the recursion is enqueued as a dependency graph on three internal streams (nets, float64
        table kernels, serial coder kernels), so that the tensor-pipe and the FP64-pipe work of one chain share the SMs;
        False (default): plain program order on the caller's stream.  Same results either way."""
        check(lib().bsw_codec_set_dual_stream(self._h, int(on)))

    def set_two_phase(self, on=True):
        """True (default): parallel row-table kernel + serial coder; False: fused one-warp-per-stream kernels."""
        check(lib().bsw_codec_set_two_phase(self._h, int(on)))

    def profile(self, enable=-1):
        """Per-kernel-category device time since profiling was enabled: {name: (ms, launches)}.
        enable: True/False resets and starts/stops, -1 just reads."""
        ms = np.zeros(12, dtype=np.float64)
        n = np.zeros(12, dtype=np.int64)
        check(lib().bsw_codec_profile(self._h, int(enable), ms.ctypes.data, n.ctypes.data))
        return {k: (float(ms[i]), int(n[i])) for i, k in enumerate(self.CATEGORIES)}


class PipelinedCodec:
    """`lanes` BitSwapCodecs, each coding a contiguous sub-range of the streams on its own CUDA stream.

    The coder's row-table kernel is FP64-pipe bound and the dense convs are tensor-pipe bound; chains of
    different sub-batches drift apart in phase, so their kernels share SMs and the two pipes overlap
    (measured on B200, C8, 1024 streams: 379 -> 345 ms per encode+decode step with 4 lanes; more lanes do not
    help).  Results are identical to a single BitSwapCodec: every stream is independent and every kernel is
    batch-invariant.  Each lane owns a model replica (activations are per-lane anyway)."""

    def __init__(self, cfg: CodecConfig, state_dict, bins: Bins, max_batch: int, lanes: int = 4, use_tensor_cores=True, lane_size: int = 0,
                 free_running: bool = False):
        self.cfg, self.bins, self.max_batch = cfg, bins, int(max_batch)
        self.device = bins.device
        self.lanes = max(1, min(int(lanes), self.max_batch))
        self.per = -(-self.max_batch // self.lanes)
        if lane_size > 0:             # explicit sub-batch size (the last lane takes the remainder), e.g. a multiple of SMs/2
            self.per = min(int(lane_size), self.max_batch)
            self.lanes = -(-self.max_batch // self.per)
        self.models, self.codecs, self.streams = [], [], []
        self.serial = False          # True: run the lanes back to back on the current stream (clean per-kernel timing)
        # free_running: calls fork the lanes from the current stream but do NOT join them back -- consecutive encode()/
        # decode() calls then chain per lane (a lane may be decoding while its neighbour still encodes), and the caller orders
        # later work after the codec with join().  (A start offset between the lanes was tried -- all lanes run the same
        # program, so their latency-bound serial coder phases could coincide -- and measured no effect: they drift apart on
        # their own within a step.)
        self.free_running = bool(free_running)
        for _ in range(self.lanes):
            m = Model.from_config(cfg, max_batch=self.per, use_tensor_cores=use_tensor_cores, device=self.device).load_state_dict(state_dict)
            m.compress()
            self.models.append(m)
            self.codecs.append(BitSwapCodec(cfg, m, bins, self.per))
            self.streams.append(torch.cuda.Stream(device=self.device))

    def _ranges(self, count):
        out, b = [], 0
        while b < count:
            out.append((b, min(self.per, count - b)))
            b += self.per
        return out

    def _fan(self, count, fn):
        if self.serial:
            for i, (b, n) in enumerate(self._ranges(count)):
                fn(self.codecs[i], b, n)
            return
        cur = torch.cuda.current_stream(self.device)
        ev = torch.cuda.Event()
        ev.record(cur)
        for i, (b, n) in enumerate(self._ranges(count)):
            st = self.streams[i]
            st.wait_event(ev)
            with torch.cuda.stream(st):
                fn(self.codecs[i], b, n)
        if not self.free_running:
            self.join()

    def join(self):
        """The current stream waits for everything the lanes have been given so far."""
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            cur.wait_stream(st)

    def encode(self, streams: StreamSet, x: torch.Tensor, first=0, scheme=BITSWAP, extents=None):
        assert x.is_cuda and x.dtype == torch.uint8 and x.is_contiguous() and x.shape[0] <= self.max_batch
        self.codecs[0]._extents_ptr(extents, x.shape[0])          # (shape / dtype / device checked before any lane starts)
        self._fan(x.shape[0], lambda c, b, n: c.encode(streams, x[b:b + n], first=first + b, scheme=scheme,
                                                       extents=None if extents is None else extents[b:b + n]))

    def decode(self, streams: StreamSet, count: int, first=0, scheme=BITSWAP, out=None, extents=None):
        if out is None:
            out = torch.empty((count,) + tuple(self.cfg.xs), dtype=torch.uint8, device=torch.device("cuda", self.device))
        self.codecs[0]._extents_ptr(extents, count)
        self._fan(count, lambda c, b, n: c.decode(streams, n, first=first + b, scheme=scheme, out=out[b:b + n],
                                                  extents=None if extents is None else extents[b:b + n]))
        return out

    def set_two_phase(self, on=True):
        for c in self.codecs:
            c.set_two_phase(on)

    def set_dual_stream(self, on=True):
        for c in self.codecs:
            c.set_dual_stream(on)

    @property
    def last_launches(self):
        return sum(c.last_launches for c in self.codecs)

    def profile(self, enable=-1):
        tot = {}
        for c in self.codecs:
            for k, (ms, n) in c.profile(enable).items():
                a = tot.get(k, (0.0, 0))
                tot[k] = (a[0] + ms, a[1] + n)
        return tot
