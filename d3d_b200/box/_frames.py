"""Ragged frame batches: the host side of the frame-batched entry points of d3d_b200.box.

A batch call takes its frames in one of two forms.  The list form is one tensor or array per frame and per input set.  The packed form
is each set's frames back to back, with CPU int64 offsets [nframes + 1] per set: frame f holds rows rows[f]:rows[f + 1] of one set and
columns cols[f]:cols[f + 1] of the other.  A per-pair result of frame f is a [rows_f, cols_f] block; the blocks are packed back to
back at the block offsets, the running sum of rows_f * cols_f.  Outputs go back to the caller's side: numpy in gives numpy out, host
tensors in give host tensors out, and the list form gets per-frame views of the packed outputs."""
import functools
import itertools

import numpy as np
import torch


def host(x):
    """a numpy array as a tensor sharing its memory; tensors pass through"""
    return torch.from_numpy(x) if isinstance(x, np.ndarray) else x


def offsets_of(lens):
    """CPU int64 offsets [len(lens) + 1] of frames of the given lengths"""
    return torch.tensor([0] + list(lens), dtype=torch.int64).cumsum(0)


def _checked(given):
    """(CPU int64 offsets, the same as a list, frame lengths as a list) of offsets given in any integer form"""
    off = torch.as_tensor(given).to(torch.int64).cpu().reshape(-1)
    o = off.tolist()   # the check and the frame maxima work on this list: cheaper than tensor ops on the per-call path of a packed batch
    lens = [b - a for a, b in zip(o, o[1:])]
    if not o or o[0] != 0 or min(lens, default=0) < 0:
        raise ValueError("frame offsets must start at 0 and be ascending")
    return off, o, lens


def offsets(given):
    """CPU int64 offsets from offsets given in any integer form, checked to start at 0 and ascend"""
    return _checked(given)[0]


def to_device(dev, *arrays):
    """the given CPU int64 arrays on the device `dev`, with one copy"""
    d = torch.cat(arrays).to(dev, non_blocking=True)
    return torch.split(d, [a.numel() for a in arrays])


class Frames:
    """The frames of one batch call: row and column offsets, checked, and the caller's side that the outputs go back to (list form or
    packed, numpy in or not, device of the inputs)."""

    def __init__(self, rows, cols=None, as_list=False, numpy_in=False, device=None):
        """`rows`, `cols`: offsets [nframes + 1] in any integer form; `cols` None for frames of a single set, whose columns are its rows"""
        self.rows, self._r, self._nr = _checked(rows)
        self.cols, self._c, self._nc = (self.rows, self._r, self._nr) if cols is None else _checked(cols)
        if len(self._r) != len(self._c):
            raise ValueError("Numbers of frames in the offsets are inconsistent!")
        self.nframes = len(self._r) - 1
        self.as_list, self.numpy_in, self.device = as_list, numpy_in, device

    @property
    def T(self):
        """the same frames with rows and columns exchanged"""
        return Frames(self.cols, self.rows, self.as_list, self.numpy_in, self.device)

    def expect(self, n_rows, n_cols, what):
        """raise unless the offsets end at n_rows rows and n_cols columns"""
        if self._r[-1] != n_rows or self._c[-1] != n_cols:
            raise ValueError(f"Numbers of {what} and frame offsets are inconsistent!")

    def lengths(self):
        """(rows_f, cols_f) of every frame, CPU int64 [nframes]"""
        return self.rows[1:] - self.rows[:-1], self.cols[1:] - self.cols[:-1]

    def bounds(self, where=None):
        """(largest rows_f, largest cols_f) over all frames, or over those `where` (bool [nframes]) marks; 0 where there is none"""
        if where is None:
            return max(self._nr, default=0), max(self._nc, default=0)
        f = torch.nonzero(where).flatten().tolist()
        return max((self._nr[i] for i in f), default=0), max((self._nc[i] for i in f), default=0)

    @functools.cached_property
    def _k(self):
        return list(itertools.accumulate((r * c for r, c in zip(self._nr, self._nc)), initial=0))

    @functools.cached_property
    def blocks(self):
        """CPU int64 [nframes + 1]: where every frame's [rows_f, cols_f] block starts in a packed per-pair output, and the total"""
        return torch.tensor(self._k, dtype=torch.int64)

    def each(self, where=None):
        """(f, row slice, column slice, block slice) of every frame, or of the frames `where` (bool [nframes]) marks"""
        r, c, k = self._r, self._c, self._k
        for f in range(self.nframes) if where is None else torch.nonzero(where).flatten().tolist():
            yield f, slice(r[f], r[f + 1]), slice(c[f], c[f + 1]), slice(k[f], k[f + 1])

    def back(self, x):
        """an output on the caller's side: on the host unless the inputs were device tensors, and numpy if they were numpy"""
        if self.device.type != "cuda" or self.numpy_in:
            x = x.cpu()
        return x.detach().numpy() if self.numpy_in else x

    def matrices(self, flat):
        """a packed per-pair output on the caller's side: (flat, block offsets), or in the list form the per-frame [rows_f, cols_f] views"""
        flat = self.back(flat)
        if not self.as_list:
            return flat, self.blocks.numpy() if self.numpy_in else self.blocks
        return [flat[k].reshape(r.stop - r.start, c.stop - c.start) for _, r, c, k in self.each()]

    def outputs(self, rows=(), cols=()):
        """per-row and per-column outputs (along their last axis) on the caller's side: the tuple rows + cols, or in the list form per frame
        the tuple of their frame's slices"""
        rows, cols = tuple(map(self.back, rows)), tuple(map(self.back, cols))
        if not self.as_list:
            return rows + cols
        return [tuple(x[..., r] for x in rows) + tuple(x[..., c] for x in cols) for _, r, c, _ in self.each()]


def empty(*sets):
    """the list form without frames, whose result is []: every given set an empty list"""
    return all(isinstance(x, (list, tuple)) and len(x) == 0 for x in sets)


def inputs(a, b, a_offsets, b_offsets, check, names, dtype=None):
    """Both call forms of a batch entry point over two per-frame sets (not `empty`) -> (A, B, frames).

    A and B are the sets packed, on the caller's side; the frames have the rows of `a` and the columns of `b`.  `check(a_f, b_f)` is the
    entry point's shape check, `names` its names of the two sets in the error messages.  The frames of a set in the list form must share
    one dtype, unless `dtype` is given: then each is cast to it before the concatenation.  Argument errors are raised here, before any
    device work.  The list form is concatenated with torch.cat, so autograd reaches every per-frame tensor."""
    as_list = isinstance(a, (list, tuple))
    if as_list:
        if not isinstance(b, (list, tuple)) or len(a) != len(b):
            raise ValueError(f"{names[0]} and {names[1]} should hold the same number of frames")
        numpy_in = isinstance(a[0], np.ndarray)
        la, lb = [host(x) for x in a], [host(x) for x in b]
        for x, y in zip(la, lb):
            check(x, y)
        if dtype is not None:
            la, lb = [x.to(dtype) for x in la], [y.to(dtype) for y in lb]
        elif len({x.dtype for x in la}) != 1 or len({y.dtype for y in lb}) != 1:
            raise RuntimeError(f"the frames of {names[0]}, and those of {names[1]}, must have the same dtype")
        a_offsets, b_offsets = offsets_of(len(x) for x in la), offsets_of(len(y) for y in lb)
        A, B = torch.cat(la), torch.cat(lb)
    else:
        numpy_in = isinstance(a, np.ndarray)
        if numpy_in:
            assert isinstance(b, np.ndarray), "Input should be both numpy tensor or pytorch tensor!"
            a, b = torch.from_numpy(a), torch.from_numpy(b)
        if a_offsets is None or b_offsets is None:
            raise ValueError(f"packed {names[0]} and {names[1]} need the frame offsets")
        check(a, b)
        A, B = a, b
    frames = Frames(a_offsets, b_offsets, as_list, numpy_in, A.device)
    frames.expect(len(A), len(B), f"{names[0]}, {names[1]}")
    return A, B, frames
