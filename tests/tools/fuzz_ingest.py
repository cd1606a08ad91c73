"""Mutation fuzzing of the native readers (csrc/ingest.cu, csrc/zipread.h): .sig JSON, .zip collections, FASTA / FASTQ
(plain and gzip).  Host code only -- runs against the real library without a GPU.  Run by hand:

    python tests/tools/fuzz_ingest.py [seconds] [seed]
    SMB_EMUL_ASAN=1 python tests/tools/fuzz_ingest.py [seconds] [seed]     # the same readers under AddressSanitizer + UBSan
                                                                            # (the g++ build of tests/host_emul/emul_lib.py)

Every batch of mutated inputs is parsed in a child process: the parent only looks at how the child ended.  A parse
error (an exception through the ABI) is a fine outcome; a signal (SIGSEGV, SIGABRT, SIGBUS), a timeout or a Python-level
error that is not one of the library's own is a finding, and the offending input is kept under the temp directory.
"""
import glob
import gzip
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
GOLDEN = os.path.join(ROOT, "tests", "golden")
CORPUS = os.path.join(GOLDEN, "reference_corpus.tar.gz")         # sourmash's test data, shrunk

CHILD = r'''
import os, sys
sys.path.insert(0, %(root)r)
if os.environ.get("SMB_EMUL_ASAN") == "1":            # the host code compiled with AddressSanitizer + UBSan (emul_lib.py)
    sys.path.insert(0, os.path.join(%(root)r, "tests", "host_emul"))
    import emulated_boot
    emulated_boot.install()
import sourmash_b200 as smb
from sourmash_b200.exceptions import SourmashError
from sourmash_b200.sigset import SignatureSet
from sourmash_b200.sketch import RecordBatch
from sourmash_b200.sbt_storage import ZipStorage
from sourmash_b200.signature import load_signatures_from_json
ok = err = 0
for path in sys.argv[1:]:
    kind = os.path.basename(path).split("_")[0]
    try:
        if kind == "sig":
            with open(path, "rb") as fh:
                data = fh.read()
            for s in load_signatures_from_json(data, do_raise=True):
                s.md5sum(); len(s.minhash)
            ss = SignatureSet.from_files([path])
            for i in range(len(ss)):
                ss.name(i); ss.md5sum(i)
            ss.csr_host()
        elif kind == "zip":
            ss = SignatureSet.from_files([path])
            for i in range(len(ss)):
                ss.name(i); ss.location(i)
            ss.csr_host()
            SignatureSet.from_files([path], use_manifest=False, traverse_yield_all=True)
            with ZipStorage(path) as z:
                for name in z._filenames():
                    z.load(name)
        else:
            rb = RecordBatch([path], n_threads=1)
            rb.names()
            for r in range(min(len(rb), 4)):
                rb.sequence(r)
        ok += 1
    except (SourmashError, ValueError, OSError, KeyError, IndexError, UnicodeDecodeError) as exc:
        err += 1
print("CHILD DONE", ok, err)
'''


def seeds():
    "small valid inputs of every kind: (kind, suffix, bytes)"
    out = []
    for p in sorted(glob.glob(os.path.join(GOLDEN, "*.sig")))[:3]:
        with open(p, "rb") as fh:
            out.append(("sig", ".sig", fh.read()))
    with open(os.path.join(GOLDEN, "2.fa.sig"), "rb") as fh:
        out.append(("sig", ".sig.gz", gzip.compress(fh.read())))
    import tarfile
    with tarfile.open(CORPUS) as tar:                               # sourmash's own collections (not the SBTs)
        zips = [m for m in sorted(tar.getmembers(), key=lambda m: m.name)
                if m.name.endswith(".zip") and "sbt" not in os.path.basename(m.name)]
        for m in zips[:6]:
            out.append(("zip", ".zip", tar.extractfile(m).read()))
    import io
    import zipfile
    for method in (zipfile.ZIP_STORED, zipfile.ZIP_DEFLATED):       # collections made here (beside
        buf = io.BytesIO()                                          # sourmash's): no manifest, two members
        with zipfile.ZipFile(buf, "w", method) as z:
            for name in ("2.fa.sig", "47.fa.sig"):
                z.write(os.path.join(GOLDEN, name), "signatures/" + name)
        out.append(("zip", ".zip", buf.getvalue()))
    fa = b">r1 first\nACGTACGTNNACGT\nACGT\n>r2\n\nGGGG\r\n>r3\n" + b"ACGT" * 300 + b"\n"
    fq = b"@r1 x\nACGTN\n+\nIIIII\n@r2\nAC\nGT\n+r2\nII\nII\n@r3\nTTTT\n+\n@@@@\n"
    out += [("fa", ".fa", fa), ("fa", ".fa.gz", gzip.compress(fa)), ("fa", ".fq", fq), ("fa", ".fq.gz", gzip.compress(fq))]
    return out


def mutate(rng, data):
    b = bytearray(data)
    n = len(b)
    for _ in range(int(rng.integers(1, 6))):
        how = int(rng.integers(0, 7))
        if n == 0:
            break
        i = int(rng.integers(0, n))
        if how == 0:
            b[i] = int(rng.integers(0, 256))
        elif how == 1:
            b[i] ^= 1 << int(rng.integers(0, 8))
        elif how == 2:                                          # truncate
            b = b[: int(rng.integers(0, n))]
        elif how == 3:                                          # overwrite 4 / 8 bytes with an extreme integer
            w = int(rng.choice([4, 8]))
            v = int(rng.choice([0, 0xFFFFFFFF, 0x7FFFFFFF, 0xFFFFFFFFFFFFFFFF, 0xFFFFFFFFFFFFFF00, 1 << 31]))
            b[i:i + w] = (v & ((1 << (8 * w)) - 1)).to_bytes(w, "little")[: max(0, min(w, n - i))]
        elif how == 4:                                          # duplicate a slice
            j = int(rng.integers(i, min(n, i + 64) + 1))
            b[i:i] = b[i:j]
        elif how == 5:                                          # delete a slice
            j = int(rng.integers(i, min(n, i + 64) + 1))
            del b[i:j]
        else:                                                   # structural characters of JSON / FASTA
            b[i:i + 1] = bytes(rng.choice([b"[", b"]", b"{", b"}", b'"', b",", b":", b">", b"@", b"+", b"\n", b"\0", b"-", b"e", b"9" * 25]))
        n = len(b)
    return bytes(b)


def main():
    seconds = float(sys.argv[1]) if len(sys.argv) > 1 else 60
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 1
    rng = np.random.default_rng(seed)
    corpus = seeds()
    tmp = tempfile.mkdtemp(prefix="smb_fuzz_ingest_")
    child = os.path.join(tmp, "child.py")
    with open(child, "w") as fh:
        fh.write(CHILD % {"root": ROOT})
    env = dict(os.environ)
    if env.get("SMB_EMUL_ASAN") == "1":
        asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
        cxx = subprocess.run(["gcc", "-print-file-name=libstdc++.so.6"], capture_output=True, text=True).stdout.strip()
        # libstdc++ next to it: the sanitizer resolves its __cxa_throw interceptor when it starts, python itself has no C++
        env.update(LD_PRELOAD=asan + " " + cxx, ASAN_OPTIONS="detect_leaks=0:abort_on_error=1", UBSAN_OPTIONS="print_stacktrace=1")
    t0, batches, inputs, findings = time.time(), 0, 0, []
    while time.time() - t0 < seconds:
        paths = []
        for k in range(40):
            kind, suffix, data = corpus[int(rng.integers(0, len(corpus)))]
            blob = mutate(rng, data)
            if suffix.endswith(".gz") and rng.random() < 0.5:      # mutate below the compression too
                try:
                    blob = gzip.compress(mutate(rng, gzip.decompress(data)))
                except Exception:
                    pass
            p = os.path.join(tmp, "%s_%d_%d%s" % (kind, batches, k, suffix))
            with open(p, "wb") as fh:
                fh.write(blob)
            paths.append(p)
        try:
            r = subprocess.run([sys.executable, child] + paths, capture_output=True, text=True, timeout=300, env=env)
            bad = r.returncode != 0 or "CHILD DONE" not in r.stdout
            why = "exit %d: %s" % (r.returncode, (r.stderr or "")[-3000:])
        except subprocess.TimeoutExpired:
            bad, why = True, "timeout"
        if bad:                                                   # find the input: one at a time
            for p in paths:
                try:
                    r1 = subprocess.run([sys.executable, child, p], capture_output=True, text=True, timeout=120, env=env)
                    if r1.returncode != 0 or "CHILD DONE" not in r1.stdout:
                        findings.append((p, "exit %d: %s" % (r1.returncode, (r1.stderr or "")[-3000:])))
                except subprocess.TimeoutExpired:
                    findings.append((p, "timeout"))
            if not findings:
                findings.append(("(batch %d, not reproduced one by one)" % batches, why))
            break
        for p in paths:
            os.unlink(p)
        batches += 1
        inputs += len(paths)
    print("fuzz_ingest: %d mutated inputs in %d batches, seed %d, %.0f s" % (inputs, batches, seed, time.time() - t0))
    for p, why in findings:
        print("FINDING", p, why)
    print("no findings" if not findings else "%d findings (inputs kept under %s)" % (len(findings), tmp))
    return 1 if findings else 0


if __name__ == "__main__":
    sys.exit(main())
