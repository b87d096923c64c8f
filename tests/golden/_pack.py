"""Compact container for many small named arrays: one blob per dtype + a JSON index, stored in a
single compressed .npz (a plain .npz costs a few hundred bytes of zip header per array).  A pack
that would compress to more than MAX_FILE_BYTES is stored in parts, <stem>.part0.npz, .part1.npz,
..., each a pack of its own, so that no file of the repository grows past 1 MB (the limit keeps a
margin below that: the compressed size moves a little with the zlib that writes it)."""
import json
import os

import numpy as np

DTYPES = ("int32", "int64", "float64")
MAX_FILE_BYTES = 900_000


def _part(stem, k):
    return f"{stem}.part{k}.npz"


class Packer:
    def __init__(self):
        self.entries = {}

    def __setitem__(self, name, arr):
        a = np.asarray(arr)
        if a.dtype.kind == "f":
            a = a.astype(np.float64)
        elif a.dtype == np.int32:
            pass
        else:
            a = a.astype(np.int64)
        self.entries[name] = a

    def _write(self, path, names):
        index, blobs, sizes = {}, {dt: [] for dt in DTYPES}, {dt: 0 for dt in DTYPES}
        for name in names:
            a = self.entries[name]
            dt = str(a.dtype)
            flat = a.reshape(-1)
            index[name] = [dt, sizes[dt], int(flat.size), list(a.shape)]
            blobs[dt].append(flat)
            sizes[dt] += int(flat.size)
        out = {"index": np.frombuffer(json.dumps(index).encode(), dtype=np.uint8)}
        for dt, parts in blobs.items():
            out[dt] = np.concatenate(parts) if parts else np.empty(0, dtype=dt)
        np.savez_compressed(path, **out)

    def save(self, path):
        """Writes path, or -- when that file would exceed MAX_FILE_BYTES -- the entries, in insertion order, spread
        over as few parts of about equal raw size as keep every file under it."""
        stem = path[:-len(".npz")]
        k = 0
        while os.path.exists(_part(stem, k)):
            os.remove(_part(stem, k))
            k += 1
        names = list(self.entries)
        raw = np.cumsum([self.entries[n].nbytes for n in names])
        for parts in range(1, len(names) + 1):
            paths = [path] if parts == 1 else [_part(stem, k) for k in range(parts)]
            cuts = [0] + [int(np.searchsorted(raw, raw[-1] * k / parts)) for k in range(1, parts)] + [len(names)]
            for p, lo, hi in zip(paths, cuts, cuts[1:]):
                self._write(p, names[lo:hi])
            if all(os.path.getsize(p) <= MAX_FILE_BYTES for p in paths):
                return paths
            for p in paths:
                os.remove(p)
        raise ValueError(f"{path}: one entry alone compresses to more than {MAX_FILE_BYTES} bytes")


class Pack:
    def __init__(self, path):
        stem = path[:-len(".npz")]
        paths = [path] if os.path.exists(path) else []
        while not os.path.exists(path) and os.path.exists(_part(stem, len(paths))):
            paths.append(_part(stem, len(paths)))
        if not paths:
            raise FileNotFoundError(f"{path} (or its parts, {_part(stem, 0)}, ...)")
        self.index, self.blobs = {}, []
        for k, p in enumerate(paths):
            z = np.load(p)
            for name, entry in json.loads(bytes(z["index"]).decode()).items():
                self.index[name] = [k] + entry
            self.blobs.append({dt: z[dt] for dt in DTYPES})

    def __contains__(self, name):
        return name in self.index

    def __getitem__(self, name):
        k, dt, off, size, shape = self.index[name]
        return self.blobs[k][dt][off:off + size].reshape(shape).copy()
