"""Writes tests/golden/reference_corpus.tar.gz: a shrunken copy of the signature and sequence files that sourmash ships
as test data (tests/test-data/ and data/ of a sourmash checkout, same layout), for the native-reader tests of test_ingest.py.

    python tests/golden/make_reference_corpus.py <sourmash checkout>

Signature files keep every record and every key; each sketch keeps its first MAX_MINS hashes (and abundances), so the
archive stays small, and gets the md5sum of the hashes it keeps (see sketch_md5): a sketch whose stored md5sum does not
match its hashes is a broken file, on which sourmash and this package would rightly disagree.  Files (and zip members) Python's json cannot read --
deliberately broken fixtures -- keep their first BROKEN_BYTES bytes.
Sequence files keep their first SEQ_BYTES bytes (decompressed), cut at a line end, gzip-compressed again when they were.
Zip collections keep every member, in order and with its compression: signatures (SBT leaves too) shrunk as above, the md5 and n_hashes columns of a manifest recomputed to match, other members (SBT nodes) cut to their first BROKEN_BYTES bytes.
"""
import csv
import glob
import gzip
import hashlib
import io
import json
import os
import sys
import tarfile
import zipfile

MAX_MINS = 48
BROKEN_BYTES = 2048
SEQ_BYTES = 12_000
SEQ_PATTERNS = ("*.fa", "*.fa.gz", "*.fna", "*.fna.gz", "*.faa", "*.faa.gz", "*.fq.gz", "*.fq", "*.fastq", "*.fasta")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_corpus.tar.gz")


def _read(path):
    with (gzip.open if path.endswith(".gz") else open)(path, "rb") as fh:
        return fh.read()


def _encode(path, data):
    return gzip.compress(data, mtime=0) if path.endswith(".gz") else data


def sketch_md5(sk):
    """The md5sum sourmash gives a sketch, as its signature format documents it: md5 over the k-mer size, then every hash
    in ascending order, each as decimal text.  Computed here with hashlib, independently of the code under test."""
    h = hashlib.md5(str(sk["ksize"]).encode())
    for x in sorted(sk["mins"]):
        h.update(str(x).encode())
    return h.hexdigest()


def shrink_signature_file(path, raw=None):
    given = raw is not None
    raw = raw if given else _read(path)
    try:
        doc = json.loads(raw)
    except Exception:                                     # noqa: BLE001 -- kept as the broken bytes they are
        if given:
            return raw[:BROKEN_BYTES]
        with open(path, "rb") as fh:
            return fh.read()[:BROKEN_BYTES]
    for rec in doc if isinstance(doc, list) else [doc]:
        for sk in rec.get("signatures", []) if isinstance(rec, dict) else []:
            for key in ("mins", "abundances"):
                if isinstance(sk.get(key), list):
                    sk[key] = sk[key][:MAX_MINS]
            if isinstance(sk.get("mins"), list) and "md5sum" in sk:
                sk["md5sum"] = sketch_md5(sk)
    return _encode(path, json.dumps(doc).encode())


def shrink_zip(path):
    src = zipfile.ZipFile(path)
    members, n_hashes = {}, {}
    for info in src.infolist():
        data = src.read(info)
        plain = gzip.decompress(data) if data[:2] == b"\x1f\x8b" else data
        if plain.lstrip()[:1] == b"[" or info.filename.endswith((".sig", ".sig.gz")):   # signatures, SBT leaves too
            small = shrink_signature_file(info.filename.removesuffix(".gz"), raw=plain)
            data = gzip.compress(small, mtime=0) if data[:2] == b"\x1f\x8b" else small
            try:
                before, after = json.loads(plain), json.loads(small)
                for rec0, rec in zip(before, after):
                    for sk0, sk in zip(rec0["signatures"], rec["signatures"]):
                        n_hashes[sk0["md5sum"]] = (sk["md5sum"], len(sk["mins"]))
            except Exception:                             # noqa: BLE001
                pass
        elif not info.filename.endswith((".csv", ".json", "/")):
            data = data[:BROKEN_BYTES]
        members[info.filename] = (info, data)
    manifest = members.get("SOURMASH-MANIFEST.csv")
    if manifest:
        lines = manifest[1].decode().splitlines(keepends=True)
        head = [ln for ln in lines if ln.startswith("#")]
        rows = list(csv.DictReader([ln for ln in lines if not ln.startswith("#")]))
        out = io.StringIO()
        out.write("".join(head))
        w = csv.DictWriter(out, fieldnames=list(rows[0].keys()) if rows else [], lineterminator="\n")
        w.writeheader()
        for r in rows:
            if r["md5"] in n_hashes:
                md5, n = n_hashes[r["md5"]]
                r["md5"], r["n_hashes"] = md5, str(n)
                if "md5short" in r:
                    r["md5short"] = md5[:8]
            w.writerow(r)
        members["SOURMASH-MANIFEST.csv"] = (manifest[0], out.getvalue().encode())
    buf = io.BytesIO()
    with zipfile.ZipFile(buf, "w") as dst:
        for info, data in members.values():
            dst.writestr(info, data, compress_type=info.compress_type)
    return buf.getvalue()


def shrink_sequence_file(path):
    raw = _read(path)
    if len(raw) > SEQ_BYTES:
        raw = raw[: raw.rfind(b"\n", 0, SEQ_BYTES) + 1]
    return _encode(path, raw)


def main(checkout):
    data = os.path.join(checkout, "tests", "test-data")
    files = {}
    for p in glob.glob(os.path.join(data, "**", "*.sig"), recursive=True) + \
            glob.glob(os.path.join(data, "**", "*.sig.gz"), recursive=True):
        files["tests/test-data/" + os.path.relpath(p, data)] = shrink_signature_file(p)
    for p in glob.glob(os.path.join(data, "**", "*.zip"), recursive=True):
        try:
            files["tests/test-data/" + os.path.relpath(p, data)] = shrink_zip(p)
        except zipfile.BadZipFile:
            with open(p, "rb") as fh:
                files["tests/test-data/" + os.path.relpath(p, data)] = fh.read()[:BROKEN_BYTES]
    for pat in SEQ_PATTERNS:
        for p in glob.glob(os.path.join(data, "**", pat), recursive=True):
            if os.path.getsize(p) > 0:
                files["tests/test-data/" + os.path.relpath(p, data)] = shrink_sequence_file(p)
        for p in glob.glob(os.path.join(checkout, "data", pat)):
            if os.path.getsize(p) > 0:
                files["data/" + os.path.basename(p)] = shrink_sequence_file(p)
    buf = io.BytesIO()
    with tarfile.open(fileobj=buf, mode="w") as tar:
        for name in sorted(files):
            info = tarfile.TarInfo(name)
            info.size, info.mode = len(files[name]), 0o644
            tar.addfile(info, io.BytesIO(files[name]))
    with open(OUT, "wb") as fh:
        fh.write(gzip.compress(buf.getvalue(), compresslevel=9, mtime=0))
    print("%s: %d files, %d bytes" % (OUT, len(files), os.path.getsize(OUT)))


if __name__ == "__main__":
    main(sys.argv[1])
