import gzip
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _ensure_built():
    """Compile libsourmash_b200.so if it is missing or stale (needs nvcc; the GPU box receives the
    prebuilt file with the snapshot).  Loaded by path so the package is not imported first."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_smb_build", os.path.join(ROOT, "sourmash_b200", "_build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    try:
        if mod.needs_build():
            mod.build()
    except Exception as exc:                      # no nvcc on this machine: use what is there
        if not os.path.exists(mod.LIB):
            raise RuntimeError(f"cannot build {mod.LIB}: {exc}")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    _ensure_built()


def read_fasta(path):
    """Minimal FASTA reader -> list of (name, bytes)."""
    opener = gzip.open if path.endswith(".gz") else open
    recs, name, chunks = [], None, []
    with opener(path, "rb") as fh:
        for line in fh:
            line = line.rstrip(b"\r\n")
            if line.startswith(b">"):
                if name is not None:
                    recs.append((name, b"".join(chunks)))
                name, chunks = line[1:].decode(), []
            elif line:
                chunks.append(line)
    if name is not None:
        recs.append((name, b"".join(chunks)))
    return recs


@pytest.fixture(scope="session")
def golden():
    arrays = np.load(os.path.join(GOLDEN, "golden_arrays.npz"))
    with open(os.path.join(GOLDEN, "golden_meta.json")) as fh:
        meta = json.load(fh)
    return {"arrays": arrays, "meta": meta}


@pytest.fixture(scope="session")
def ecoli_seq():
    recs = read_fasta(os.path.join(GOLDEN, "ecoli_k12.fna.gz"))
    assert len(recs) == 1
    return recs[0][1]


@pytest.fixture(scope="session")
def s10_records():
    return read_fasta(os.path.join(GOLDEN, "genome-s10.fa.gz"))


@pytest.fixture(scope="session")
def reference_corpus(tmp_path_factory):
    """golden/reference_corpus.tar.gz extracted: sourmash's test data, shrunk (golden/make_reference_corpus.py), laid out
    as in a sourmash checkout (tests/test-data/, data/).  Returns the directory."""
    import tarfile
    root = tmp_path_factory.mktemp("reference_corpus")
    with tarfile.open(os.path.join(GOLDEN, "reference_corpus.tar.gz")) as tar:
        tar.extractall(root, filter="data")
    return str(root)


@pytest.fixture(scope="session")
def golden_dir():
    import pathlib
    return pathlib.Path(GOLDEN)
