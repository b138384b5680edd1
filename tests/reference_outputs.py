"""Outputs of the original project's own code (compiled verbatim into oracle/_ref by `make -C oracle`) for the inputs a test builds.

Where oracle/_ref was built, the test compares against the live reference on every input, and the rows stored under
tests/golden/reference_functions.npz must still be what the reference returns.  Everywhere else (a checkout without the original
project) the test compares the same seeded inputs against those stored rows: a fixed subset of each array (`rows`), small enough to
keep in the repository.  tools/make_golden.py writes the file by running the tests' inputs through the live reference."""
import hashlib
import json
import os

import numpy as np

from common import ROOT

GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_functions.npz")
RECORD = os.environ.get("PPG_RECORD_REFERENCE_OUTPUTS")      # set by tools/make_golden.py: collect the rows instead of reading them
_stored = None
_recorded = {}


def rows(n, k=100):
    """The rows of an n-row array that are stored: the first 100 and the last 50 (where the tests put their edge cases) and k seeded picks."""
    pick = np.random.default_rng(n).choice(n, min(n, k), replace=False)
    return np.unique(np.concatenate([np.arange(min(n, 100)), pick, np.arange(max(0, n - 50), n)]))


def reference(key, live, n, k=100):
    """(row indices, [arrays]) of the reference's outputs for `key`: `live()` returns the full arrays when the reference library exists
    (it is None otherwise).  The caller compares its own outputs at those rows; with the live reference the rows are all n."""
    global _stored
    if live is not None:
        full = [np.asarray(a) for a in live()]
        idx = rows(n, k)
        if RECORD:
            for i, a in enumerate(full):
                _recorded[f"{key}/{i}"] = a[idx]
        else:
            stored = _load()
            for i, a in enumerate(full):
                s = stored[f"{key}/{i}"]
                assert np.array_equal(a[idx].view(np.uint8), s.view(np.uint8)), f"{key}/{i}: the stored reference rows are stale (tools/make_golden.py)"
        return np.arange(n), full
    stored = _load()
    out, i = [], 0
    while f"{key}/{i}" in stored:
        out.append(stored[f"{key}/{i}"]); i += 1
    assert out, f"no stored reference rows for {key}"
    return rows(n, k), out


def _load():
    global _stored
    if _stored is None:
        z = np.load(GOLDEN)
        _stored = {k: z[k] for k in z.files}
    return _stored


def save_recorded(path=GOLDEN):
    np.savez_compressed(path, **_recorded)
    return len(_recorded)


DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_digests.json")
_digests = None
_recorded_digests = {}


def digest(a):
    a = np.ascontiguousarray(a)
    return f"{a.dtype.str}{a.shape}:" + hashlib.sha256(a.tobytes()).hexdigest()


def reference_digests(key, live):
    """{name: digest} of the bit patterns of the arrays the reference returns for `key`: computed from `live()` ({name: array}) when the
    reference library exists (and then checked against tests/golden/reference_digests.json), read from that file otherwise.  For outputs
    too large to store row by row (trained SD-trees): equal digests mean equal bits."""
    global _digests
    if _digests is None:
        _digests = json.load(open(DIGESTS)) if os.path.exists(DIGESTS) else {}
    if live is None:
        assert key in _digests, f"no stored reference digests for {key}"
        return _digests[key]
    d = {name: digest(a) for name, a in live().items()}
    if RECORD:
        _recorded_digests[key] = d
    else:
        assert _digests.get(key) == d, f"{key}: the stored reference digests are stale (tools/make_golden.py)"
    return d


def save_recorded_digests(path=DIGESTS):
    json.dump(_recorded_digests, open(path, "w"), indent=1, sort_keys=True)
    return len(_recorded_digests)
