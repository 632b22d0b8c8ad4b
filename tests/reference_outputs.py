"""What the unmodified reference produced on the parity tests' inputs, stored in tests/golden/reference_outputs.json.

The tests build their inputs from fixed seeds and compare our outputs with the reference's outputs stored here. They do
not run the reference itself. tests/golden/make_golden.py records the file by calling those same test functions while
`RECORDING` is set: then `expected` runs the reference through `compute()` and keeps what it returns."""
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.json")
RECORDING = None        # make_golden.py: a dict that collects {key: value}
STOP_AFTER_RECORD = False


class Recorded(Exception):
    """Raised after recording when the rest of the test needs hardware the recording machine lacks."""


_stored = None


def digest(a):
    """sha256 of an array's dtype, shape and bytes: two arrays with equal digests are equal element by element."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(str((a.dtype.descr, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def expected(key, compute):
    global _stored
    if RECORDING is not None:
        RECORDING[key] = json.loads(json.dumps(compute()))
        if STOP_AFTER_RECORD:
            raise Recorded(key)
        return RECORDING[key]
    if _stored is None:
        with open(PATH) as f:
            _stored = json.load(f)
    assert key in _stored, f"no stored reference output for {key!r}: regenerate with tests/golden/make_golden.py"
    return _stored[key]
