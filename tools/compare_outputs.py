"""Compare two `bench.py --dump-outputs` directories array by array: bit-identical, or the largest relative difference.

    python tools/compare_outputs.py <dir_a> <dir_b>

Relative difference of an entry: |a - b| / max(|a|, |b|), over the entries that are finite on both sides (0 where both are
0).  NaNs in the same places, and infinities of the same sign in the same places, count as equal values; an array that
differs only in such entries, or in the sign of a zero, is reported as equal in value but not bit-identical.
Prints one line per array.  Exit status 0 when every array is bit-identical on both sides, 1 otherwise (an array missing
from one side, a shape mismatch or any difference in the bits)."""
import os
import sys

import numpy as np


def compare(a: np.ndarray, b: np.ndarray) -> str:
    if a.shape != b.shape:
        return "shape %s vs %s" % (a.shape, b.shape)
    if a.dtype == b.dtype and a.tobytes() == b.tobytes():
        return "bit-identical"
    nan_a, nan_b = np.isnan(a), np.isnan(b)
    if (nan_a != nan_b).any():
        return "NaN in different places (%d vs %d)" % (nan_a.sum(), nan_b.sum())
    inf_a, inf_b = np.isinf(a), np.isinf(b)
    if (inf_a != inf_b).any() or (a[inf_a] != b[inf_b]).any():
        return "infinities differ (%d vs %d)" % (inf_a.sum(), inf_b.sum())
    fin = np.isfinite(a) & np.isfinite(b)
    if not fin.any():
        return "equal in value (NaN / inf in the same places), not bit-identical"
    x, y = a[fin].astype(np.float64), b[fin].astype(np.float64)
    d = np.abs(x - y)
    if not (d > 0).any():
        return "equal in value (signed zeros or NaN payloads differ), not bit-identical"
    scale = np.maximum(np.abs(x), np.abs(y))
    rel = np.divide(d, scale, out=np.zeros_like(d), where=scale > 0)
    i = int(np.argmax(rel))
    return "max rel %.3e (abs %.3e), %d of %d entries differ" % (rel[i], d[i], int((d > 0).sum()), d.size)


def main() -> int:
    if len(sys.argv) != 3:
        sys.stderr.write(__doc__ + "\n")
        return 2
    da, db = sys.argv[1:3]
    names = sorted(n for n in set(os.listdir(da)) | set(os.listdir(db)) if n.endswith(".npy"))
    rc = 0
    for name in names:
        pa, pb = os.path.join(da, name), os.path.join(db, name)
        if not (os.path.exists(pa) and os.path.exists(pb)):
            print("%-32s only in %s" % (name, da if os.path.exists(pa) else db))
            rc = 1
            continue
        res = compare(np.load(pa), np.load(pb))
        if res != "bit-identical":
            rc = 1
        print("%-32s %s" % (name, res))
    return rc


if __name__ == "__main__":
    sys.exit(main())
