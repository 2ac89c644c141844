"""Row panels of phyloselect's N x N distance matrix (DESIGN.md section 4.12).

K-medoids, HDBSCAN, t-SNE and the neighbour graph read the matrix in passes over its rows, so they do not need
it resident: a source hands out panels of rows [r0, r1) x all N columns as device views, in the matrix's dtype,
r1 - r0 a multiple of TILE except for the last panel, and ``rows(indices)``, a k x N device buffer with those
rows.  Three kinds:

- ``ResidentSource``: a device matrix; one panel, the matrix itself.
- ``ProfileSource``: recomputes every panel from the profiles with the distance tile kernels, bit for bit the
  rows of ``engine.distance_matrix_device(X, metric, torch.float32, symmetric=True)``.
- ``FileSource``: reads the panels of a row-major float32 / float64 matrix file (phyloligo.py --large memmap or
  h5py) with parallel pread into two pinned buffers, then one asynchronous copy to the device.

``profile_source`` and phyloselect's matrix readers choose: resident when the matrix and the consumers' working state fit in
free device memory (``device_budget``), panels otherwise, their height from the same budget.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from . import _lib, engine
from ._lib import PhyloligoError, TILE, FLAG_SKIP_LOWER, FLAG_MIRROR, FLAG_MIRROR_ONLY

# device bytes per matrix row that the consumers keep besides the panel (t-SNE: neighbour indices, float64
# conditional probabilities and the symmetrisation's sort keys at perplexity <= 100; HDBSCAN's MST workspace)
STATE_BYTES_PER_ROW = 32 << 10
STATE_BYTES_FIXED = 1 << 30
# a panel of a file is staged twice in pinned host memory: keep it small (page-locking costs ~0.5 s per GB)
FILE_PANEL_BYTES = 1 << 30
# rows per distance launch (grid limits), as in engine.distance_matrix_device
LAUNCH_ROWS = 65535 * 32


def device_budget(device=None):
    """Bytes of device memory a matrix or its panels may take: free memory plus what torch's caching allocator
    holds unused."""
    device = device or engine.require_cuda()
    free, _ = torch.cuda.mem_get_info(device)
    return int(free + torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device))


def state_bytes(n):
    return STATE_BYTES_FIXED + STATE_BYTES_PER_ROW * int(n)


def fits(n, element_size, budget=None):
    """True when an n x n matrix of element_size bytes and the consumers' working state fit in `budget`."""
    budget = device_budget() if budget is None else budget
    return int(n) * int(n) * int(element_size) + state_bytes(n) <= budget


def panel_rows_for(n, element_size, budget=None, cap_bytes=None):
    """Panel height: a multiple of TILE whose panel takes at most half of what the budget leaves after the
    working state (and at most cap_bytes)."""
    budget = device_budget() if budget is None else budget
    room = max(0, budget - state_bytes(n)) // 2
    if cap_bytes is not None:
        room = min(room, cap_bytes)
    rows = room // max(1, int(n) * int(element_size)) // TILE * TILE
    if rows < TILE:
        raise PhyloligoError("a panel of %d rows of %d columns needs %d bytes of device memory, %d are free" % (
            TILE, n, TILE * int(n) * int(element_size) + state_bytes(n), budget))
    return int(min(rows, max(TILE, -(-int(n) // TILE) * TILE)))


def _spans(n, h):
    return [(r0, min(n, r0 + h)) for r0 in range(0, n, h)]


class ResidentSource:
    """The matrix resident on the device: one panel, the matrix itself (a view, no copy)."""

    resident = True
    symmetric = True  # HDBSCAN checks the whole matrix at once

    def __init__(self, D):
        self.D = D
        self.n = int(D.shape[0])
        self.dtype = D.dtype
        self.device = D.device
        self.panel_rows = self.n

    def panels(self):
        yield 0, self.n, self.D

    def rows(self, indices):
        return self.D.index_select(0, indices.to(self.device))


class ProfileSource:
    """Panels recomputed from the profiles X (N x D) for `metric`, equal bit for bit to the rows of
    engine.distance_matrix_device(X, metric, torch.float32, symmetric=True).  One panel takes three launches:
    its diagonal square with SKIP_LOWER | MIRROR as the resident matrix computes it, the part right of it stored
    directly, and the part left of it computed from the block rows above (the column's profile is the row
    operand, as in the resident matrix's mirrored tiles) and stored transposed only (PO_FLAG_MIRROR_ONLY).  A
    pass over all panels computes N^2 pairs, twice the resident matrix's N^2 / 2."""

    resident = False
    symmetric = True  # every entry is a tile of the symmetric resident matrix

    def __init__(self, X, metric, panel_rows=None, prepared=None):
        self.device = engine.require_cuda()
        self.metric = metric
        self.P, self.aux, self.dim = prepared if prepared is not None else engine.prepare(X, metric)
        self.n = int(self.P.shape[0])
        self.dtype = torch.float32
        if panel_rows is None:
            panel_rows = panel_rows_for(self.n, 4)
        self.panel_rows = max(TILE, int(panel_rows) // TILE * TILE)
        self.buf = torch.empty((min(self.panel_rows, self.n), self.n), dtype=torch.float32, device=self.device)
        self.pairs_computed = 0

    def compute(self, r0, r1, out):
        """Rows [r0, r1) (r0 a multiple of TILE) into the device view out ((r1 - r0) x n, contiguous rows)."""
        n, m, P, aux, dim = self.n, self.metric, self.P, self.aux, self.dim
        engine.distance_block(m, P, aux, dim, r0, r1, r0, r1, out, r0, 0, FLAG_SKIP_LOWER | FLAG_MIRROR)
        if r1 < n:
            engine.distance_block(m, P, aux, dim, r0, r1, r1, n, out, r0, 0, 0)
        for a0 in range(0, r0, LAUNCH_ROWS):
            engine.distance_block(m, P, aux, dim, a0, min(r0, a0 + LAUNCH_ROWS), r0, r1, out, r0, 0,
                                  FLAG_MIRROR | FLAG_MIRROR_ONLY, mirror=out, mirror_row0=r0, mirror_col0=0)
        if dim < 2 and m == "KT":
            out.fill_(1.0)  # as distance_matrix_device: kendall() with no element pair
        self.pairs_computed += (r1 - r0) * n
        return out

    def panels(self):
        for r0, r1 in _spans(self.n, self.panel_rows):
            yield r0, r1, self.compute(r0, r1, self.buf[: r1 - r0])

    def rows(self, indices):
        idx = indices.to(self.device, torch.int64)
        out = torch.empty((int(idx.numel()), self.n), dtype=torch.float32, device=self.device)
        scratch = torch.empty((min(TILE, self.n), self.n), dtype=torch.float32, device=self.device)
        for b in torch.unique(idx // TILE).tolist():
            r0, r1 = b * TILE, min(self.n, (b + 1) * TILE)
            block = self.compute(r0, r1, scratch[: r1 - r0])
            sel = torch.nonzero(idx // TILE == b).flatten()
            out[sel] = block[idx[sel] - r0]
        return out


class FileSource:
    """Panels of the row-major n x n matrix stored at byte `offset` of the file at `path` (float32 or float64):
    each panel is read with parallel pread (po_host_pread) into one of two pinned buffers, then copied to the
    device with one asynchronous copy (po_copy2d_async), so that the next panel's read overlaps the consumer's
    kernels.  Nothing the size of the file is held in host memory."""

    resident = False
    symmetric = False  # HDBSCAN reads the column strip of every panel for its symmetry test

    def __init__(self, path, n, offset=0, dtype=np.float32, panel_rows=None, threads=8):
        self.device = engine.require_cuda()
        self.lib = _lib.load()
        self.path = path
        self.n = int(n)
        self.offset = int(offset)
        self.np_dtype = np.dtype(dtype)
        self.dtype = torch.float32 if self.np_dtype == np.float32 else torch.float64
        self.es = self.np_dtype.itemsize
        if panel_rows is None:
            panel_rows = panel_rows_for(self.n, self.es, cap_bytes=FILE_PANEL_BYTES)
        self.panel_rows = max(TILE, int(panel_rows) // TILE * TILE)
        self.threads = int(threads)
        h = min(self.panel_rows, self.n)
        self.pinned = [torch.empty((h, self.n), dtype=self.dtype).pin_memory() for _ in range(2)]
        self.buf = torch.empty((h, self.n), dtype=self.dtype, device=self.device)
        self.events = [None, None]
        self.fd = os.open(path, os.O_RDONLY)

    def close(self):
        if self.fd is not None:
            for ev in self.events:
                if ev is not None:
                    ev.synchronize()
            os.close(self.fd)
            self.fd = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def read_rows(self, r0, r1, host):
        """Rows [r0, r1) of the file into the pinned host tensor `host`."""
        nbytes = (r1 - r0) * self.n * self.es
        _lib.check(self.lib.po_host_pread(self.fd, self.offset + r0 * self.n * self.es, C.c_void_p(host.data_ptr()), nbytes,
                                          self.threads), "po_host_pread")

    def panels(self):
        for k, (r0, r1) in enumerate(_spans(self.n, self.panel_rows)):
            slot = k & 1
            if self.events[slot] is not None:
                self.events[slot].synchronize()  # the copy out of this pinned buffer has completed
            host = self.pinned[slot][: r1 - r0]
            self.read_rows(r0, r1, host)
            dev = self.buf[: r1 - r0]
            engine.copy2d(dev, host)  # stream-ordered after the previous panel's consumer
            ev = torch.cuda.Event()
            ev.record()
            self.events[slot] = ev
            yield r0, r1, dev

    def rows(self, indices):
        idx = indices.cpu().numpy().astype(np.int64).ravel()
        host = torch.empty((len(idx), self.n), dtype=self.dtype).pin_memory()
        for q, i in enumerate(idx.tolist()):
            self.read_rows(i, i + 1, host[q:q + 1])
        out = torch.empty((len(idx), self.n), dtype=self.dtype, device=self.device)
        engine.copy2d(out, host)
        torch.cuda.current_stream().synchronize()  # `host` is released on return
        return out

    def column_strip(self, r0, r1):
        """Columns [r0, r1) of every row, [0, n) x [r0, r1), as a device tensor: one strided read."""
        mm = np.memmap(self.path, dtype=self.np_dtype, mode="r", offset=self.offset, shape=(self.n, self.n))
        return torch.from_numpy(np.ascontiguousarray(mm[:, r0:r1])).to(self.device)


SOURCES = (ResidentSource, ProfileSource, FileSource)


def profile_source(X, metric, budget=None):
    """The source of the matrix of profiles X (a tensor or array, N x D) for `metric`: resident
    (distance_matrix_device) when it fits in device memory with the consumers' working state, ProfileSource
    otherwise."""
    Xd = X if isinstance(X, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(np.asarray(X)))
    Xd = Xd.to(engine.require_cuda())
    budget = device_budget() if budget is None else budget
    if fits(Xd.shape[0], 4, budget):
        return ResidentSource(engine.distance_matrix_device(Xd, metric, torch.float32, symmetric=True))
    return ProfileSource(Xd, metric, panel_rows=panel_rows_for(Xd.shape[0], 4, budget))


def file_matrix(path, large):
    """(n, byte offset, dtype) of the matrix phyloligo.py --large memmap / h5py wrote to `path`."""
    from . import io_formats
    if large == "memmap":
        size = os.path.getsize(path) // 4
        n = int(round(np.sqrt(size)))
        if n * n != size:
            raise PhyloligoError("Error, weird shape for matrix {}".format(path))
        return n, 0, np.float32
    shape, dtype, offset = io_formats.dataset_location(path, "distances")
    if len(shape) != 2 or shape[0] != shape[1]:
        raise PhyloligoError("a square distance matrix is expected, got shape %s" % (tuple(shape),))
    return int(shape[0]), offset, dtype


def as_source(D):
    """A source for a precomputed matrix: a source is returned as it is; a np.memmap of a row-major float32 /
    float64 file that does not fit on the device becomes a FileSource; anything else is made resident
    (as_device_matrix)."""
    if isinstance(D, SOURCES):
        return D
    if (isinstance(D, np.memmap) and D.ndim == 2 and D.shape[0] == D.shape[1] and D.flags.c_contiguous
            and D.dtype in (np.float32, np.float64) and getattr(D, "filename", None)
            and not fits(D.shape[0], D.dtype.itemsize)):
        return FileSource(D.filename, D.shape[0], offset=D.offset, dtype=D.dtype)
    from .phyloselect import as_device_matrix
    return ResidentSource(as_device_matrix(D))
