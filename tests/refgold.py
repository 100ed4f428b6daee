"""Observations of the reference stored under tests/golden/, so that the tests comparing the oracle with the reference
run on machines without the reference's sources.  The generators in tests/golden/ record them from the compiled
reference; `digest` turns what a test compares into the stored form (arrays and long lists become SHA-256 digests, so
equality of digests is equality of the bytes)."""
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def sha(b) -> str:
    return hashlib.sha256(np.ascontiguousarray(b).tobytes() if isinstance(b, np.ndarray) else bytes(b)).hexdigest()


def digest(x):
    if isinstance(x, np.ndarray):
        return "sha256:" + sha(x)
    if isinstance(x, dict):
        return {str(k): digest(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        items = [digest(v) for v in x]
        if len(items) > 64:
            return f"sha256:{hashlib.sha256(repr(items).encode()).hexdigest()} ({len(items)} items)"
        return items
    if isinstance(x, np.integer):
        return int(x)
    return x


_loaded = {}


def recorded(name: str) -> dict:
    """The recordings in tests/golden/<name>, keyed by scenario."""
    if name not in _loaded:
        with open(os.path.join(GOLDEN, name)) as f:
            _loaded[name] = json.load(f)["recordings"]
    return _loaded[name]


def write(name: str, source: str, recordings: dict):
    """One recording per line."""
    lines = [f"{json.dumps(k)}: {json.dumps(recordings[k], separators=(',', ':'), sort_keys=True)}" for k in sorted(recordings)]
    with open(os.path.join(GOLDEN, name), "w") as f:
        f.write(f'{{"source": {json.dumps(source)},\n "recordings": {{\n' + ",\n".join(lines) + "\n}}\n")
