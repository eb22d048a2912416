"""Results of the original NeRF-RPN implementation that the tests compare against, stored under tests/golden/reference/.

`recorded(name, compute)` returns the arrays stored in tests/golden/reference/<name>.npz, so that the comparison runs wherever the
repository does.  With NRPN_RECORD_REFERENCE=<dir> in the environment (and the reference staged by oracle/build_ref.py), it calls
`compute()` instead -- the test's own code that runs the reference -- writes the arrays it returns to <dir>/<name>.npz and returns them:
the same test refreshes the golden file and checks against the live reference.  Large outputs are stored as fixed, seeded samples
(`sample_index`) so that every file stays small."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")


def recording() -> bool:
    return bool(os.environ.get("NRPN_RECORD_REFERENCE"))


def recorded(name, compute):
    out_dir = os.environ.get("NRPN_RECORD_REFERENCE")
    if out_dir:
        arrays = {k: np.asarray(v) for k, v in compute().items()}
        os.makedirs(out_dir, exist_ok=True)
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), **arrays)
        return arrays
    with np.load(os.path.join(GOLDEN, name + ".npz")) as z:
        return {k: z[k] for k in z.files}


def sample_index(n, k, seed):
    """k distinct indices of range(n) in increasing order, the same on every run (all of them when k >= n)."""
    if k >= n:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))
