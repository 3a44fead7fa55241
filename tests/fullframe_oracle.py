"""Test infrastructure: the oracle recursions with a partial pixel block (full-frame containers).

An independent restatement, on top of the pinned oracle/oracle.py (which stays exactly the reference's recursion), of
what `BitSwapCodec.encode/decode(extents=...)` does:
  * the block's masked pixels (y >= valid_rows or x >= valid_cols) are replaced by the edge-replicate fill before
    infer(0) sees the block -- here with np.pad(mode="edge");
  * the pixel level is a sequence of independent per-row ANS tables, so coding only the valid rows is exactly
    ANS(pmfs[valid]).encode(state, x[valid]) / ANS(pmfs[valid]).decode(state) with the oracle's coder classes;
  * after the x-level pop the decoder applies the same fill to the decoded symbols.
Everything else -- the latent levels and the prior -- is the base class's recursion, unchanged.  extent=None is the
base class's call.
"""
import numpy as np
import torch

from oracle import oracle as O


def fill_block(x, extent):
    """[C, 32, 32] block -> the same block with the masked pixels replaced by the edge-replicate fill."""
    vr, vc = int(extent[0]), int(extent[1])
    x = np.asarray(x)
    return np.pad(x[:, :vr, :vc], ((0, 0), (0, x.shape[1] - vr), (0, x.shape[2] - vc)), mode="edge")


def valid_rows(xs, extent):
    """Indices of the valid pixel rows of the flat CHW pixel level, ascending."""
    C, H, W = xs
    m = np.zeros((C, H, W), dtype=bool)
    m[:, :int(extent[0]), :int(extent[1])] = True
    return np.flatnonzero(m.reshape(-1))


class MaskedBitSwapOracle(O.BitSwapOracle):
    """BitSwapOracle whose encode/decode take `extent=(valid_rows, valid_cols)` of the pixel block."""

    def _push_x(self, mu, sc, state, x, valid):
        pm = self._pmfs(self.xend, mu, sc)
        return self._coder(pm[valid], 8).encode(state, x[valid])

    def _pop_x(self, mu, sc, state, valid, extent):
        pm = self._pmfs(self.xend, mu, sc)
        state, sv = self._coder(pm[valid], 8).decode(state)
        sym = np.zeros(self.cfg.xdim, dtype=np.int64)
        sym[valid] = np.asarray(sv)
        return state, torch.from_numpy(fill_block(sym.reshape(self.cfg.xs), extent).reshape(-1).copy())

    # -- Bit-Swap sender / receiver -------------------------------------------------------------------------------------------
    def encode_image(self, state, x, extent=None):
        if extent is None:
            return super().encode_image(state, x)
        c = self.cfg
        valid = valid_rows(c.xs, extent)
        x = torch.as_tensor(fill_block(np.asarray(x).reshape(c.xs), extent).reshape(-1).astype(np.int64))
        q = c.quantbits
        zsym = None
        for zi in range(c.nz):
            given = self.zcen[zi - 1, self.zr, zsym] if zi > 0 else self.xcen[self.xr, x]
            mu, sc = self._net("infer", zi, given)
            state, zsymtop = self._pop(self.zend[zi], mu, sc, q, state)
            zsymtop = torch.as_tensor(np.asarray(zsymtop))
            self._note(f"pop z{zi+1}", state)
            z = self.zcen[zi, self.zr, zsymtop]
            mu, sc = self._net("generate", zi, z)
            if zi > 0:
                state = self._push(self.zend[zi - 1], mu, sc, q, state, zsym.numpy())
            else:
                state = self._push_x(mu, sc, state, x.numpy(), valid)
            self._note(f"push {'z%d' % zi if zi > 0 else 'x'}", state)
            zsym = zsymtop
        state = self._coder(self._prior(), q).encode(state, zsym.numpy())
        self._note("push prior", state)
        return state

    def decode_image(self, state, extent=None):
        if extent is None:
            return super().decode_image(state)
        c = self.cfg
        valid = valid_rows(c.xs, extent)
        q = c.quantbits
        state, zsymtop = self._coder(self._prior(), q).decode(state)
        zsymtop = torch.as_tensor(np.asarray(zsymtop))
        for zi in reversed(range(c.nz)):
            z = self.zcen[zi, self.zr, zsymtop]
            mu, sc = self._net("generate", zi, z)
            if zi > 0:
                state, sym = self._pop(self.zend[zi - 1], mu, sc, q, state)
                sym = torch.as_tensor(np.asarray(sym))
            else:
                state, sym = self._pop_x(mu, sc, state, valid, extent)
            given = self.zcen[zi - 1, self.zr, sym] if zi > 0 else self.xcen[self.xr, sym]
            mu, sc = self._net("infer", zi, given)
            state = self._push(self.zend[zi], mu, sc, q, state, zsymtop.numpy())
            zsymtop = sym
        return state, zsymtop.numpy().astype(np.uint8)

    # -- BB-ANS sender / receiver ---------------------------------------------------------------------------------------------
    def encode_image_bbans(self, state, x, extent=None):
        if extent is None:
            return super().encode_image_bbans(state, x)
        c = self.cfg
        valid = valid_rows(c.xs, extent)
        x = torch.as_tensor(fill_block(np.asarray(x).reshape(c.xs), extent).reshape(-1).astype(np.int64))
        q = c.quantbits
        zs, zsym = [], None
        for zi in range(c.nz):
            given = self.zcen[zi - 1, self.zr, zsym] if zi > 0 else self.xcen[self.xr, x]
            mu, sc = self._net("infer", zi, given)
            state, zsym = self._coder(self._pmfs(self.zend[zi], mu, sc), q).decode(state)
            zsym = torch.as_tensor(np.asarray(zsym))
            zs.append(zsym)
        zsym = None
        for zi in range(c.nz):
            z = self.zcen[zi, self.zr, zs[zi]]
            mu, sc = self._net("generate", zi, z)
            if zi > 0:
                state = self._coder(self._pmfs(self.zend[zi - 1], mu, sc), q).encode(state, zsym.numpy())
            else:
                state = self._push_x(mu, sc, state, x.numpy(), valid)
            zsym = zs[zi]
        return self._coder(self._prior(), q).encode(state, zsym.numpy())

    def decode_image_bbans(self, state, extent=None):
        if extent is None:
            return super().decode_image_bbans(state)
        c = self.cfg
        valid = valid_rows(c.xs, extent)
        q = c.quantbits
        state, top = self._coder(self._prior(), q).decode(state)
        zs = [torch.as_tensor(np.asarray(top))]
        for zi in reversed(range(c.nz)):
            z = self.zcen[zi, self.zr, zs[-1]]
            mu, sc = self._net("generate", zi, z)
            if zi > 0:
                state, sym = self._coder(self._pmfs(self.zend[zi - 1], mu, sc), q).decode(state)
                sym = torch.as_tensor(np.asarray(sym))
            else:
                state, sym = self._pop_x(mu, sc, state, valid, extent)
            zs.append(sym)
        for zi in reversed(range(c.nz)):
            sym = zs[c.nz - zi]
            given = self.zcen[zi - 1, self.zr, sym] if zi > 0 else self.xcen[self.xr, sym]
            mu, sc = self._net("infer", zi, given)
            state = self._coder(self._pmfs(self.zend[zi], mu, sc), q).encode(state, zs[c.nz - zi - 1].numpy())
        return state, zs[-1].numpy().astype(np.uint8)
