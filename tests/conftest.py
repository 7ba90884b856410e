import hashlib
import json
import lzma
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
if GOLDEN not in sys.path:
    sys.path.insert(0, GOLDEN)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def load_json(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def cfg1_head_stats():
    """The reference's run on cfg1_iq: READER_STATS, print_results text, window count and TX commands."""
    return load_json("cfg1_head_ref_stats.json")


@pytest.fixture(scope="session")
def cfg1_iq(cfg1_head_stats):
    """The first 300,000 samples (15 inventory rounds) of the reference's recorded capture
    misc/data/file_source_test (committed xz-compressed)."""
    raw = lzma.decompress(open(os.path.join(GOLDEN, "file_source_test_head.c64.xz"), "rb").read())
    iq = np.frombuffer(raw, dtype=np.complex64)
    assert iq.size == cfg1_head_stats["samples"] == 300000
    assert hashlib.sha256(raw).hexdigest() == cfg1_head_stats["sha256"]
    return iq


@pytest.fixture(scope="session")
def cfg1_full_golden():
    """Records of the reference's run on the whole recording (all 142 windows)."""
    return np.load(os.path.join(GOLDEN, "cfg1_ref_records.npy"))


@pytest.fixture(scope="session")
def cfg1_golden(cfg1_full_golden, cfg1_head_stats):
    """Records of the reference's run on cfg1_iq: the first windows of its run on the whole recording."""
    return cfg1_full_golden[:cfg1_head_stats["n_windows"]]


@pytest.fixture(scope="session")
def oracle():
    from oracle.pyoracle import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def ref_outputs():
    """What the reference's own blocks (oracle/_ref) computed for the comparisons in tests/golden/make_golden.py."""
    with np.load(os.path.join(GOLDEN, "reference_outputs.npz")) as z:
        return {k: z[k] for k in z.files}


def ref_segments(ref_outputs, n, seed, kw, iq):
    """The reference's (records, counts) for synth.make_capture(n, seed=seed, **kw); iq must be that capture."""
    from make_golden import iq_digest, synth_key
    key = synth_key(n, seed, kw)
    assert iq_digest(iq) == str(ref_outputs[key + "_sha256"]), "synth.make_capture no longer produces the stored input"
    return ref_outputs[key + "_records"], ref_outputs[key + "_counts"]


def records_equal(a, b):
    """bit-exact comparison of two record arrays; returns list of differing field names"""
    bad = []
    if a.shape != b.shape:
        return ["shape %s vs %s" % (a.shape, b.shape)]
    for f in a.dtype.names:
        if a[f].tobytes() != b[f].tobytes():
            bad.append(f)
    return bad
