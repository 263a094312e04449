"""What the unmodified reference returned, stored as digests, for the tests that compare this library against it.

The reference is compiled into oracle/_ref/ by oracle/Makefile only where its source tree is present, so every such
test checks this library against tests/golden/reference_digests.json, and where oracle/_ref/ exists also checks that
the reference still returns what is stored.  Each entry keeps the digest of the test's input next to the reference's
output, so a change of the generated inputs is reported as such rather than as a mismatch of the code under test.

To record the entries again (needs oracle/_ref/):  SCN_RECORD_REFERENCE=1 python -m pytest tests"""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATH = os.path.join(ROOT, "tests", "golden", "reference_digests.json")
RECORD = os.environ.get("SCN_RECORD_REFERENCE") == "1"
_table = None


def have(lib: str) -> bool:
    """whether the compiled reference artefact oracle/_ref/<lib> is present"""
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", lib))


def digest(*parts) -> str:
    """sha256 over byte strings, text and arrays (raw bytes of a C-contiguous copy), each prefixed by its length"""
    h = hashlib.sha256()
    for p in parts:
        if isinstance(p, str):
            p = p.encode()
        elif not isinstance(p, (bytes, bytearray)):
            p = np.ascontiguousarray(p).tobytes()
        h.update(len(p).to_bytes(8, "little"))
        h.update(p)
    return h.hexdigest()


def _load():
    global _table
    if _table is None:
        with open(PATH) as fh:
            _table = json.load(fh)
    return _table


def expect(key: str, lib: str, inputs: str, reference) -> str:
    """The reference's output digest for `key`.  `inputs` is the digest of what the test feeds it; `reference` is a callable
    that runs oracle/_ref/<lib> on those inputs and returns the digest of its output, called only where that file exists."""
    table = _load()
    live = reference() if have(lib) else None
    if RECORD and live is not None:
        table[key] = {"inputs": inputs, "output": live}
        with open(PATH, "w") as fh:
            json.dump(table, fh, indent=1, sort_keys=True)
            fh.write("\n")
        return live
    assert key in table, f"no stored reference output for {key}"
    assert table[key]["inputs"] == inputs, f"{key}: the test's inputs changed since the reference output was recorded"
    if live is not None:
        assert live == table[key]["output"], f"{key}: oracle/_ref/{lib} no longer returns the recorded output"
    return table[key]["output"]
