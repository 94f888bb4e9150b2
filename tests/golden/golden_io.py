"""Compact storage of golden arrays (every fixture file stays under 1 MB).

An array is stored as the exact pattern of its non-zero entries plus the values of a fixed subset of them.  The last axis is cut
into sections at the column offsets given for the array -- the record layout's field offsets (sections()); without offsets
the whole record is one section.  A group is one section of one row (all axes but the last) when per_row is set, else one
section over all rows.  A group keeps its non-zeros whole when it has at most min_keep of them; a larger one keeps the
max(min_keep, ceil(n / block)) whose positions hash lowest.  Arrays with at most KEEP_ALL non-zeros are stored whole.  The
subset is a pure function of the array's shape, non-zero pattern and these parameters, all of which are stored, so arrays
with the same pattern keep the same positions.

load() gives back arrays of the original shape: exact zeros where the array is zero, the stored values, and NaN at the
non-zeros that were not kept.  Comparisons go over the entries that are not NaN (finite())."""
import numpy as np

KEEP_ALL = 2048     # arrays with at most this many non-zeros are stored whole


def sections(layout, prefix, stride=None):
    """Column offsets of the fields of a record layout whose attribute names start with prefix (e.g. "r_", "k_", "c_")."""
    stride = stride if stride is not None else getattr(layout, prefix + "stride")
    offs = {v for k, v in vars(layout).items() if k.startswith(prefix) and isinstance(v, int) and not k.endswith(("_size", "stride"))}
    return sorted({0} | {o for o in offs if 0 <= o < stride})


def _hash(pos):
    """splitmix64 finaliser of the flat position."""
    z = pos.astype(np.uint64) + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def _kept(shape, nz_pos, starts, block, min_keep, per_row):
    """Boolean over nz_pos (flat, ascending): which non-zeros are stored."""
    n = nz_pos.size
    if n <= KEEP_ALL:
        return np.ones(n, dtype=bool)
    cols = shape[-1] if len(shape) else 1
    starts = np.asarray(starts, dtype=np.int64)
    group = np.searchsorted(starts, nz_pos % cols, side="right") - 1
    if per_row:
        group = group + (nz_pos // cols) * starts.size
    order = np.lexsort((_hash(nz_pos), group))
    g = group[order]
    first = np.ones(n, dtype=bool)
    first[1:] = g[1:] != g[:-1]
    begin = np.maximum.accumulate(np.where(first, np.arange(n), 0))
    rank = np.arange(n) - begin
    count = np.bincount(np.cumsum(first) - 1)[np.cumsum(first) - 1]
    quota = np.minimum(count, np.maximum(min_keep, -(-count // block)))
    keep = np.zeros(n, dtype=bool)
    keep[order[rank < quota]] = True
    return keep


def save(path, arrays, sections=None, block=16, min_keep=256, per_row=False):
    """arrays: name -> array; sections: name -> column offsets of its fields (see sections())."""
    out = {}
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float64)
        flat = a.ravel()
        nz = flat != 0.0
        pos = np.flatnonzero(nz)
        out[name + "__shape"] = np.array(a.shape, dtype=np.int64)
        starts = np.array((sections or {}).get(name, [0]), dtype=np.int64)
        out[name + "__sections"] = starts
        out[name + "__keep"] = np.array([block, min_keep, per_row], dtype=np.int64)
        out[name + "__nz"] = np.packbits(nz)
        out[name + "__val"] = flat[pos[_kept(a.shape, pos, starts, block, min_keep, per_row)]]
    np.savez_compressed(path, **out)


def load(path):
    z = np.load(path)
    out = {}
    for key in z.files:
        if not key.endswith("__shape"):
            continue
        name = key[:-len("__shape")]
        shape = tuple(int(s) for s in z[key])
        size = int(np.prod(shape))
        nz = np.unpackbits(z[name + "__nz"], count=size).astype(bool)
        pos = np.flatnonzero(nz)
        flat = np.zeros(size)
        flat[pos] = np.nan
        block, min_keep, per_row = (int(v) for v in z[name + "__keep"])
        flat[pos[_kept(shape, pos, z[name + "__sections"], block, min_keep, bool(per_row))]] = z[name + "__val"]
        out[name] = flat.reshape(shape)
    return out


def finite(b):
    """Mask of the entries of a loaded array that are known."""
    return ~np.isnan(b)
