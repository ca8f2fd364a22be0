"""File format of tests/golden/reference_golden.npz.  TEST INFRASTRUCTURE ONLY.

The reference's full-state snapshots repeat the same stored laps many times over, so every distinct array is stored once:
a key whose array equals that of an earlier key is listed in the string array ``aliases`` as "key=earlier_key".  Keys that
are stored themselves (track_table, pid_x, ... : the first of their kind) can still be read with plain ``np.load``."""
from collections.abc import Mapping
import numpy as np

ALIASES = "aliases"


def save(path, arrays):
    """np.savez_compressed of the dict ``arrays``, every distinct (dtype, shape, bytes) stored under its first key."""
    first, keep, alias = {}, {}, []
    for k, a in arrays.items():
        a = np.asarray(a)
        sig = (a.dtype.str, a.shape, a.tobytes())
        if sig in first:
            alias.append("%s=%s" % (k, first[sig]))
        else:
            first[sig] = k
            keep[k] = a
    np.savez_compressed(path, **keep, **{ALIASES: np.array(alias, dtype=str)})


class GoldenFile(Mapping):
    """Read-only mapping over a file written by save(); like np.load, every lookup returns a fresh array."""

    def __init__(self, path):
        with np.load(path) as z:
            self._arrays = {k: z[k] for k in z.files if k != ALIASES}
            self._source = {k: k for k in self._arrays}
            self._source.update(s.split("=", 1) for s in z[ALIASES])

    def __getitem__(self, key):
        return self._arrays[self._source[key]].copy()

    def __iter__(self):
        return iter(self._source)

    def __len__(self):
        return len(self._source)
