"""Shared helpers for the tests (not product code)."""
import atexit
import gzip
import os
import shutil
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "golden_v1.npz"))


# every 40th state of HH-suite's data/context_data.crf (4000 states, 7 MB): a CRF library small enough to store
CRF_SAMPLE = "context_data_every40.crf"


def ref_data(name):
    """Bytes of a file of HH-suite's data/ directory (query.hhm, query.a3m, cs219.lib, CRF_SAMPLE; stored gzipped)."""
    with gzip.open(os.path.join(ROOT, "tests", "golden", "data", name + ".gz"), "rb") as f:
        return f.read()


_ref_dir = None


def ref_data_path(name):
    """Path of an uncompressed copy of ref_data(name) in a temporary directory of this process."""
    global _ref_dir
    if _ref_dir is None:
        _ref_dir = tempfile.mkdtemp(prefix="hhg_refdata_")
        atexit.register(shutil.rmtree, _ref_dir, True)
    path = os.path.join(_ref_dir, name)
    if not os.path.exists(path):
        with open(path, "wb") as f:
            f.write(ref_data(name))
    return path


def bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


def rasterize_exclusion(Lq, Lt, i_steps, j_steps, nsteps):
    """Numpy restatement of Viterbi::ExcludeAlignment (src/hhviterbi.cpp:61-77) for test inputs."""
    m = np.zeros((Lq + 1, Lt + 1), np.uint8)
    for s in range(1, nsteps):
        i, j = int(i_steps[s]), int(j_steps[s])
        m[max(i - 40, 1):min(i + 40, Lq) + 1, j] = 1
        m[i, max(j - 40, 1):min(j + 40, Lt) + 1] = 1
    return m
