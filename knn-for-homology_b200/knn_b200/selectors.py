"""faiss's search parameters for flat indexes: ``SearchParameters(sel=IDSelector...)``.

``index.search(x, k, params=faiss.SearchParameters(sel=faiss.IDSelectorRange(0, 1000)))`` restricts a search to the
selected rows.  Every selector becomes one packed bitmap of ``ntotal`` bits per call (32-bit words, least significant
bit first: the byte layout of faiss's IDSelectorBitmap), built on the device for device searches and on the host for
host searches, and the kernels apply it where each candidate is created (include/knn_b200.h, knn_search_params).  A
filtered search returns exactly what an unfiltered search returns on an index of the selected rows alone, with the ids
mapped back to row numbers.
"""
from __future__ import annotations

import numpy as np


def _n_words(n: int) -> int:
    return (int(n) + 31) // 32


def _pack_bool(mask, device):
    """Boolean row mask (numpy, or torch on `device`) -> uint32 words (numpy) / int32 words (torch), LSB first."""
    if device is None:
        b = np.packbits(np.asarray(mask, dtype=bool), bitorder="little")
        b = np.concatenate([b, np.zeros((-len(b)) % 4, np.uint8)])
        return b.view("<u4")
    import torch

    n = mask.shape[0]
    m = torch.nn.functional.pad(mask.to(torch.int64), (0, (-n) % 32)).view(-1, 32)
    w = (m << torch.arange(32, device=m.device, dtype=torch.int64)).sum(dim=1)
    return (w - (w >= 2 ** 31).to(torch.int64) * 2 ** 32).to(torch.int32)


class IDSelector:
    """A set of row ids (faiss.IDSelector)."""

    def bitmap(self, n: int, device=None):
        """Packed words of n bits (bit i: row i is selected).  device None: numpy uint32 array; else a torch int32
        tensor on that CUDA device."""
        raise NotImplementedError


class IDSelectorRange(IDSelector):
    """Rows imin <= i < imax (faiss.IDSelectorRange)."""

    def __init__(self, imin: int, imax: int, assume_sorted: bool = False):
        self.imin, self.imax = int(imin), int(imax)

    def bitmap(self, n: int, device=None):
        lo, hi = min(max(self.imin, 0), n), min(max(self.imax, 0), n)
        if device is None:
            m = np.zeros(n, dtype=bool)
            m[lo:hi] = True
            return _pack_bool(m, None)
        import torch

        m = torch.zeros(n, dtype=torch.bool, device=device)
        m[lo:hi] = True
        return _pack_bool(m, device)


class IDSelectorBatch(IDSelector):
    """The rows listed in ids (faiss.IDSelectorBatch(ids), or (n, ids) as in faiss's C++ signature)."""

    def __init__(self, *args):
        ids = args[-1] if len(args) in (1, 2) else None
        if ids is None:
            raise TypeError("IDSelectorBatch(ids) or IDSelectorBatch(n, ids)")
        if type(ids).__module__.startswith("torch"):
            ids = ids.detach().cpu().numpy()
        ids = np.asarray(ids, dtype=np.int64).ravel()
        self.ids = ids[: int(args[0])] if len(args) == 2 else ids

    def bitmap(self, n: int, device=None):
        ids = self.ids[(self.ids >= 0) & (self.ids < n)]
        if device is None:
            m = np.zeros(n, dtype=bool)
            m[ids] = True
            return _pack_bool(m, None)
        import torch

        m = torch.zeros(n, dtype=torch.bool, device=device)
        m[torch.from_numpy(ids).to(device)] = True
        return _pack_bool(m, device)


class IDSelectorBitmap(IDSelector):
    """Row i is selected iff bit i & 7 of byte i >> 3 is set (faiss.IDSelectorBitmap(bitmap), or (nbytes, bitmap));
    rows past the end of the bitmap are not."""

    def __init__(self, *args):
        bm = args[-1] if len(args) in (1, 2) else None
        if bm is None:
            raise TypeError("IDSelectorBitmap(bitmap) or IDSelectorBitmap(nbytes, bitmap)")
        if type(bm).__module__.startswith("torch"):
            bm = bm.detach().cpu().numpy()
        bm = np.ascontiguousarray(bm).view(np.uint8).ravel()
        self.bytes = bm[: int(args[0])] if len(args) == 2 else bm

    def bitmap(self, n: int, device=None):
        nb = 4 * _n_words(n)
        b = np.zeros(nb, dtype=np.uint8)
        m = min(nb, len(self.bytes))
        b[:m] = self.bytes[:m]
        if device is None:
            return b.view("<u4")
        import torch

        return torch.from_numpy(b).to(device).view(torch.int32)  # little-endian words, as on the host


class IDSelectorNot(IDSelector):
    """The rows sel does not select (faiss.IDSelectorNot)."""

    def __init__(self, sel: IDSelector):
        self.sel = sel

    def bitmap(self, n: int, device=None):
        w = self.sel.bitmap(n, device)
        return ~w  # bits past n are ignored (allow_nbits = n)


class SearchParameters:
    """faiss.SearchParameters: `sel` restricts the search to the rows it selects (None: every row)."""

    def __init__(self, sel: IDSelector | None = None):
        self.sel = sel

