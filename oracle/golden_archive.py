"""Golden .npz archives that store each distinct array once -- TEST INFRASTRUCTURE ONLY.

The reference records several attributes of one embedding that are the same array (the
matrix, the random matrix, the source array, and the range array as its transpose).  save()
keeps the first of equal arrays and lists every later one in an alias table; load() reads
each name back bit for bit, so a test compares with exactly what the reference returned.
"""
import hashlib
import json

import numpy as np

ALIASES = "__aliases__"


def _signature(a):
    a = np.ascontiguousarray(a)
    return a.dtype.str, a.shape, hashlib.sha256(a.tobytes()).hexdigest()


def save(path, arrays):
    """np.savez_compressed(path, **arrays) with every array that equals an earlier one bit for
    bit, or equals its transpose, stored as an alias of it."""
    stored, aliases, seen = {}, {}, {}
    for name, a in arrays.items():
        a = np.asarray(a)
        for transposed, b in ((False, a), (True, a.T)):
            target = seen.get(_signature(b))
            if target is not None and np.array_equal(stored[target], b):
                aliases[name] = [target, transposed]
                break
        else:
            stored[name] = a
            seen.setdefault(_signature(a), name)
    np.savez_compressed(path, **stored, **{ALIASES: np.array(json.dumps(aliases))})


class load:
    """Read side of save(): `z[name]` and `z.files` as np.load gives them for the full archive."""

    def __init__(self, path):
        self._z = np.load(path)
        self._aliases = json.loads(str(self._z[ALIASES])) if ALIASES in self._z.files else {}
        self.files = [f for f in self._z.files if f != ALIASES] + list(self._aliases)

    def __contains__(self, name):
        return name in self._aliases or (name != ALIASES and name in self._z.files)

    def __getitem__(self, name):
        if name in self._aliases:
            target, transposed = self._aliases[name]
            a = self._z[target]
            return np.ascontiguousarray(a.T) if transposed else a
        return self._z[name]
