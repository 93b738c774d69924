"""Frame machinery shared by the dump-file analyses (RDF / CN, S(k), and the type handling of the others): the altered atom
types, the per-frame host caches, the class maps of the device histograms, the typed batch loop, the sharding of file
reads over the ranks and the merge of per-frame results.

Frames are sharded round-robin over the ranks of an initialised torch.distributed group.  With several ranks every rank
first READS only every world-th file (frame index = file index for the usual one-frame-per-file dumps); when some rank
meets a multi-frame file the whole call is repeated with every rank reading everything and selecting its frames
(``file_sharded``).  Per-frame results are merged with one all-reduce of a zero-padded [T, ...] tensor: exact for integer
histograms, and for fp64 sums too, since adding zeros is exact.
"""
from __future__ import annotations

import ctypes
import functools
from dataclasses import dataclass

import numpy as np
import torch

from .. import dist
from ..io.pipeline import FrameBatches


def calc_atom_type_ids(ids, num_mols, num_atoms):
    """_calc_atom_type (rdf_cn.py:197-215) vectorised: atom id -> 1-based position inside its molecule type block,
    offset by the atoms-per-molecule of the earlier molecule types.  ids beyond the last block are left as is."""
    ids = np.asarray(ids, dtype=np.float64)
    cut = np.cumsum(np.multiply(num_mols, num_atoms))
    out = ids.copy()
    which = np.searchsorted(cut, ids, side="left")          # first block with id <= cutoff
    for i in range(len(cut)):
        sel = which == i
        if not sel.any():
            continue
        v = np.mod(ids[sel] - cut[i], num_atoms[i])
        v[v == 0] = num_atoms[i]
        if i > 0:
            v = v + np.sum(num_atoms[:i])
        out[sel] = v
    return out


# ------------------------------------------------------------------------------------------------
# per-frame host caches
# ------------------------------------------------------------------------------------------------
def _same_values(a, b):
    """a == b element for element.  Contiguous arrays of one dtype and shape are compared with one memcmp (ctypes releases
    the GIL; 10^5 doubles take ~50 us, where ``np.array_equal`` builds a temporary and holds the GIL next to the pipeline's
    reader threads)."""
    if a is b:
        return True
    if a.shape != b.shape:
        return False
    if a.dtype == b.dtype and a.flags.c_contiguous and b.flags.c_contiguous:
        return _memcmp()(ctypes.c_void_p(a.ctypes.data), ctypes.c_void_p(b.ctypes.data), ctypes.c_size_t(a.nbytes)) == 0
    return bool(np.array_equal(a, b))


def _memcmp():
    fn = getattr(_memcmp, "fn", None)
    if fn is None:
        fn = ctypes.CDLL(None).memcmp
        fn.restype = ctypes.c_int
        fn.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t]
        _memcmp.fn = fn
    return fn


class _TypeCache:
    """Per-frame host work that depends only on the frame's id/type column: the altered types, the {type: count} table and
    the class of every atom.  Trajectories almost always repeat the same column frame after frame; one comparison (tens
    of microseconds for 10^5 atoms) then replaces ~1 ms of recomputation per frame, which is what the consumer thread of
    the file pipeline spent next to a pair kernel that needs 0.1 ms per frame."""

    def __init__(self):
        self.key = None
        self.val = None
        self.src = None            # the object last asked about (an identical object needs no comparison at all)

    def get(self, column, make):
        if column is self.src:
            return self.val
        if self.key is None or not _same_values(self.key, column):
            self.key = np.array(column, copy=True)
            self.val = make(column)
        self.src = column if column.base is None else None      # (a view into a staging buffer is not an identity)
        return self.val


class _DeviceCache:
    """The class vector on the device: uploaded again only when the host vector is another object than last time (a
    pageable H2D copy waits for the stream -- the consumer would stall behind its own kernels once per batch)."""

    def __init__(self):
        self.src, self.dev = None, None

    def get(self, arr, device):
        if arr is not self.src or self.dev is None or self.dev.device != device:
            self.dev = torch.from_numpy(arr).to(device)
            self.src = arr
        return self.dev


def _value_counts(typ):
    """{type: count}, keys ascending.  Types are small non-negative integers in practice: one bincount pass instead of
    np.unique's sort (this runs once per frame on the host, next to a pair kernel that takes 0.16 ms per frame)."""
    t = np.asarray(typ).astype(np.int64)
    if t.size and t.min() >= 0 and t.max() < (1 << 20):
        c = np.bincount(t)
        u = np.flatnonzero(c)
        return dict(zip(u.tolist(), c[u].tolist()))
    u, c = np.unique(t, return_counts=True)
    return dict(zip(u.tolist(), c.tolist()))


# ------------------------------------------------------------------------------------------------
# class maps: relation types -> small dense class ids for the device histogram
# ------------------------------------------------------------------------------------------------
class _ClassMap:
    """Types named by the relations get their own class; everything else shares the class 'other'."""

    def __init__(self, named_types, present_types=None):
        self.named = sorted(set(int(t) for t in named_types))
        self.index = {t: k for k, t in enumerate(self.named)}
        # the class 'other' is only materialised when some point actually has an unnamed type (one class fewer
        # keeps single-species runs on the kernel variant without per-pair class bookkeeping)
        self.has_other = present_types is None or bool(set(int(t) for t in present_types) - set(self.named))
        self.ncls = len(self.named) + (1 if self.has_other else 0)
        self.other = self.ncls - 1 if self.has_other else -1

    def classes_of(self, typ: np.ndarray) -> np.ndarray:
        t = np.asarray(typ).astype(np.int64)
        if t.size and t.min() >= 0 and t.max() < (1 << 20):      # one table lookup instead of a mask per named type
            lut = np.full(int(t.max()) + 1, self.other, dtype=np.int32)
            for ty, k in self.index.items():
                if 0 <= ty < len(lut):
                    lut[ty] = k
            cls = lut[t]
        else:
            cls = np.full(t.shape, self.other, dtype=np.int32)
            for ty, k in self.index.items():
                cls[t == ty] = k
        if not self.has_other and (cls < 0).any():
            raise ValueError("a frame contains atom types that were absent from the first frame")
        return cls

    def cls(self, t):
        return self.index.get(int(t), self.other)


# ------------------------------------------------------------------------------------------------
# the typed batch loop
# ------------------------------------------------------------------------------------------------
@dataclass
class TypedBatch:
    dev: torch.Tensor        # [F, C, N] on the device
    metas: list              # FrameMeta per frame
    atom_types: list         # {type: count} per frame
    props: list              # per_frame(meta, atom_types) per frame
    cmap: _ClassMap
    cls: list                # host class row per frame: one object for frames whose type columns are equal
    dcache: _DeviceCache

    def classes(self, k0, k1):
        """Device classes of frames [k0, k1): the cached [N] vector when they share one class row (no upload at all when it
        is the previous batch's), otherwise one [k1 - k0, N] upload."""
        if all(c is self.cls[k0] for c in self.cls[k0:k1]):
            return self.dcache.get(self.cls[k0], self.dev.device)
        return torch.from_numpy(np.stack(self.cls[k0:k1])).to(self.dev.device)


def typed_batches(batches, num_mols, num_atoms_per_mol, per_frame, cmap=None, named=None):
    """The batches of ``batches`` with the host work every frame needs before its kernels.  Per frame, in frame order: the
    type table (altered types from the id column when ``num_mols`` and ``num_atoms_per_mol`` are given, the type column
    otherwise), ``per_frame(meta, atom_types)`` (the caller's checks and props, which may raise), and the class row.  The
    class map is ``cmap``, or one made from ``named`` and the types present in the first frame."""
    altered = bool(num_mols and num_atoms_per_mol)
    tcache, ccache, dcache = _TypeCache(), _TypeCache(), _DeviceCache()

    def typ_and_counts(col):
        typ = calc_atom_type_ids(col, num_mols, num_atoms_per_mol) if altered else np.array(col, copy=True)
        return typ, _value_counts(typ)

    for batch in batches:
        dev = batch.wait()
        host = batch.host.numpy()
        ats, props, cls = [], [], []
        for k, meta in enumerate(batch.metas):
            typ, at = tcache.get(host[k, 0] if altered else host[k, 1], typ_and_counts)
            props.append(per_frame(meta, at))
            if cmap is None:
                cmap = _ClassMap(named, present_types=at.keys())
            ats.append(at)
            cls.append(ccache.get(typ, cmap.classes_of))
        yield TypedBatch(dev, batch.metas, ats, props, cmap, cls, dcache)


# ------------------------------------------------------------------------------------------------
# sharded file reads and the merge of per-frame results
# ------------------------------------------------------------------------------------------------
class _RetryUnsharded(Exception):
    """Some rank met a dump file with more than one frame while reading only its share of the files."""


def _frame_batches(filename, columns, shard_files):
    """This rank's frames: with several ranks and ``shard_files`` every rank reads only every world-th file; otherwise every
    rank reads everything and selects every world-th frame."""
    w, r = dist.world_size(), dist.rank()
    if w > 1 and shard_files:
        return FrameBatches(filename, columns, file_shard=(r, w))
    sel = (lambda i: i % w == r) if w > 1 else None
    return FrameBatches(filename, columns, frame_select=sel)


def _agree_sharding(batches, device):
    """Call after the batch loop and before the merge collective: all ranks learn whether the sharded read held."""
    if getattr(batches, "file_shard", None) is None:
        return
    flag = torch.tensor([1 if batches.multi_frame_seen else 0], dtype=torch.int64, device=device)
    dist.all_reduce_max_(flag)
    if int(flag.item()):
        raise _RetryUnsharded()


def file_sharded(fn):
    """Decorator of the file-based entry points, which take a keyword ``shard_files`` for ``_frame_batches``: run with
    sharded file reads, and once more with ``shard_files=False`` (on every rank at once) when a multi-frame file was met."""

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        try:
            return fn(*args, **kwargs)
        except _RetryUnsharded:
            return fn(*args, shard_files=False, **kwargs)

    return wrapper


def _merge_frames(per_frame: dict, total_frames: int, shape, device, dtype=torch.int64):
    """Place this rank's per-frame results into [T, *shape] and all-reduce (exact: every other rank adds zeros).  ``per_frame``
    maps a frame index to its [*shape] result, or a tuple of frame indices (a batch) to their [len(indices), *shape] results."""
    out = torch.zeros((total_frames,) + tuple(shape), dtype=dtype, device=device)
    for idx, t in per_frame.items():
        out[torch.tensor(idx, device=device) if isinstance(idx, tuple) else idx] = t
    dist.all_reduce_sum_(out)
    return out


def _gather_props(props: dict, total_frames: int) -> dict:
    """Every rank needs every frame's host-side normalisation inputs (tiny python objects)."""
    import torch.distributed as d

    gathered = [None] * d.get_world_size()
    d.all_gather_object(gathered, props)
    out = {}
    for g in gathered:
        out.update(g)
    assert len(out) == total_frames
    return out


def merge_results(batches, results: dict, props: dict, filename, shape, dtype=torch.int64):
    """The end of a file-based entry point, after its batch loop over ``batches``: agree on the sharding (raises
    _RetryUnsharded for ``file_sharded``), merge the per-frame ``results`` into [T, *shape] of ``dtype`` and gather the
    per-frame ``props`` on every rank -> (numpy [T, *shape], props of all T frames, T)."""
    device = torch.device("cuda", torch.cuda.current_device())   # a rank that receives no frames still joins the merge
    _agree_sharding(batches, device)
    T = batches.total_frames or 0
    if T == 0:
        raise ValueError(f"no dump frames found for {filename!r}")
    merged = _merge_frames(results, T, shape, device, dtype).cpu().numpy()
    if dist.world_size() > 1:
        props = _gather_props(props, T)
    return merged, props, T
