"""Native ingest (csrc/ingest.cu, SURVEY §8 f1/f2): FASTA/FASTQ(.gz) reader and .sig JSON
parser/writer, checked on the CPU against plain-Python readers of the same files and against the
reference-written fixtures."""
import gzip
import json
import os

import numpy as np
import pytest

import oracle as orc
import sourmash_b200 as smb
from sourmash_b200.sigset import SignatureSet
from sourmash_b200.sketch import RecordBatch, read_sequences

from tests.conftest import GOLDEN, read_fasta


def test_fasta_reader_matches_python_reader():
    paths = [os.path.join(GOLDEN, f) for f in ("genome-s10.fa.gz", "ecoli.faa", "ecoli.genes.fna", "ecoli_k12.fna.gz")]
    rb = RecordBatch(paths, n_threads=3)
    want = [(i, n, s) for i, p in enumerate(paths) for n, s in read_fasta(p)]
    assert len(rb) == len(want)
    names = rb.names()
    for r, (fi, name, seq) in enumerate(want):
        assert int(rb.files[r]) == fi and names[r] == name
        assert rb.sequence(r) == seq
    assert rb.total_bytes == sum(len(s) for _, _, s in want)
    assert [int(x) for x in rb.lengths[:3]] == [len(w[2]) for w in want[:3]]
    first = np.concatenate([[True], rb.files[1:] != rb.files[:-1]])
    assert int(rb.starts[0]) == 0 and all(int(x) % 16 == 0 for x in rb.starts[first])      # file regions
    inner = np.nonzero(~first)[0]                                                           # records packed inside
    assert all(int(rb.starts[i]) == int(rb.starts[i - 1]) + int(rb.lengths[i - 1]) for i in inner) and len(inner) > 0


def test_fastq_crlf_blank_lines_and_errors(tmp_path):
    fq = tmp_path / "r.fastq"
    fq.write_bytes(b"@r1 first read\nACGTN\n+\nIIIII\n@r2\nAC\nGT\n+r2\nII\nII\n\n@r3\nTTTT\n+\n@@@@\n")
    assert read_sequences(fq) == [("r1 first read", b"ACGTN"), ("r2", b"ACGT"), ("r3", b"TTTT")]
    gz = tmp_path / "r.fq.gz"
    gz.write_bytes(gzip.compress(fq.read_bytes()))
    assert read_sequences(gz) == read_sequences(fq)
    fa = tmp_path / "w.fa"
    fa.write_bytes(b"\n>a desc  \r\nACGT\r\nAC\r\n\r\n>b\r\n>c\nGG")
    assert read_sequences(fa) == [("a desc", b"ACGTAC"), ("b", b""), ("c", b"GG")]
    (tmp_path / "empty.fa").write_bytes(b"")
    assert read_sequences(tmp_path / "empty.fa") == []
    bad = tmp_path / "bad.txt"
    bad.write_bytes(b"hello\n")
    with pytest.raises(Exception, match="neither FASTA nor FASTQ"):
        read_sequences(bad)
    with pytest.raises(Exception, match="cannot open"):
        read_sequences(tmp_path / "missing.fa")


def _py_sketches(path):
    opener = gzip.open if str(path).endswith(".gz") else open
    with opener(path, "rt") as fh:
        for rec in json.load(fh):
            for sk in rec["signatures"]:
                yield rec, sk


def test_sig_parser_matches_python_json(golden):
    paths = [os.path.join(GOLDEN, f) for f in ("47.fa.sig", "genome-s10.fa.gz.sig")]
    ss = SignatureSet.from_files(paths, n_threads=2)
    want = [(i, rec, sk) for i, p in enumerate(paths) for rec, sk in _py_sketches(p)]
    assert len(ss) == len(want)
    for i, (fi, rec, sk) in enumerate(want):
        assert int(ss.file[i]) == fi and int(ss.ksize[i]) == sk["ksize"] and int(ss.seed[i]) == sk["seed"]
        assert int(ss.max_hash[i]) == sk.get("max_hash", 0)
        assert int(ss.num[i]) == (0 if sk.get("max_hash", 0) else sk["num"])
        assert ss.moltype(i).lower() == sk["molecule"].lower() and ss.md5sum(i) == sk["md5sum"]
        assert ss.name(i) == rec.get("name", "") and ss.filename(i) == rec.get("filename", "")
        assert np.array_equal(ss.row(i), np.array(sorted(sk["mins"]), dtype=np.uint64))
        assert orc.md5sum(sk["ksize"], ss.row(i)) == sk["md5sum"]          # the stored md5 is the md5 of the mins
        mh = ss.minhash(i)
        assert mh.md5sum() == sk["md5sum"] and len(mh) == len(sk["mins"])
    assert np.array_equal(ss.row(0), golden["arrays"]["s47"])
    assert list(ss.select(ksize=31, moltype="DNA", scaled=1000)) == [0]
    assert list(ss.select(moltype="protein")) == [i for i, (_, _, sk) in enumerate(want) if sk["molecule"] == "protein"]


def test_sig_unsorted_mins_abundances_escapes_and_filters():
    doc = [{"class": "sourmash_signature", "email": "", "filename": None, "hash_function": "0.murmur64",
            "name": 'we"ird \\ name é\n', "license": "CC0", "version": 0.4, "extra": {"a": [1, {"b": "x"}]},
            "signatures": [
                {"num": 0, "ksize": 31, "seed": 42, "max_hash": 1000, "mins": [30, 10, 20], "md5sum": "x",
                 "abundances": [3, 1, 2], "molecule": "DNA"},
                {"num": 4294967295, "ksize": 21, "seed": 7, "max_hash": 500, "mins": [5, 1], "md5sum": "y", "molecule": "protein"},
                {"num": 3, "ksize": 21, "seed": 42, "max_hash": 0, "mins": [], "md5sum": "z", "molecule": "hp"}]},
           {"signatures": [{"num": 2, "ksize": 4, "seed": 42, "max_hash": 0, "mins": [18446744073709551615, 0],
                            "md5sum": "w", "molecule": "dna"}]}]
    text = json.dumps(doc)
    for payload in (text, text.encode(), gzip.compress(text.encode())):
        ss = SignatureSet.from_json(payload)
        assert len(ss) == 4 and [int(x) for x in ss.sig_index] == [0, 0, 0, 1]
        assert ss.row(0).tolist() == [10, 20, 30] and ss.abunds[:3].tolist() == [1, 2, 3]     # sorted as pairs
        assert ss.row(1).tolist() == [1, 5] and int(ss.num[1]) == 0 and ss.moltype(1) == "protein"
        assert len(ss.row(2)) == 0 and ss.moltype(2) == "hp" and int(ss.num[2]) == 3
        assert ss.row(3).tolist() == [0, 2**64 - 1]
        assert ss.name(0) == doc[0]["name"] and ss.filename(0) == "" and ss.name(3) == ""
        assert ss.has_abund.tolist() == [True, False, False, False]
    sigs = list(smb.load_signatures(text))
    assert len(sigs) == 4 and sigs[0].minhash.hashes == {10: 1, 20: 2, 30: 3} and sigs[0].name == doc[0]["name"]
    assert [s.minhash.moltype for s in sigs] == ["DNA", "protein", "hp", "DNA"]
    assert len(list(smb.load_signatures(text, ksize=21))) == 2
    assert len(list(smb.load_signatures(text, ksize=21, select_moltype="hp"))) == 1
    assert len(list(smb.load_signatures(text, select_moltype="dayhoff"))) == 0
    assert list(smb.load_signatures("[{]")) == []
    with pytest.raises(Exception):
        list(smb.load_signatures("[{]", do_raise=True))
    with pytest.raises(ValueError):
        smb.signature.load_one_signature_from_json(text)
    # writer -> parser round trip, compact serde field order (signature.rs:401-445, minhash.rs:103-131)
    out = smb.save_signatures_to_json(sigs[:1])
    assert out.startswith(b'[{"class":"sourmash_signature","email":"","hash_function":"0.murmur64","filename":null,"name":')
    assert out.endswith(b'"molecule":"DNA"}],"version":0.4}]')
    d = json.loads(out)[0]
    assert d["name"] == doc[0]["name"] and d["signatures"][0]["mins"] == [10, 20, 30]
    assert d["signatures"][0]["abundances"] == [1, 2, 3]
    assert d["signatures"][0]["md5sum"] == orc.md5sum(31, np.array([10, 20, 30], dtype=np.uint64))
    back = list(smb.load_signatures(smb.save_signatures_to_json(sigs, compression=6)))
    assert [b.md5sum() for b in back] == [s.md5sum() for s in sigs]
    assert [b.minhash.hashes for b in back] == [s.minhash.hashes for s in sigs]


def test_writer_reproduces_a_reference_written_file_byte_for_byte():
    """genome-s10.fa.gz.sig was written by the reference's serde writer: loading it and saving it
    again gives the same bytes (field order, separators, number formatting, md5sums), except that
    the file predates the `Display for HashFunctions` that spells the DNA molecule in capitals
    (src/core/src/encodings.rs:55-69)."""
    path = os.path.join(GOLDEN, "genome-s10.fa.gz.sig")
    raw = open(path, "rb").read()
    out = smb.save_signatures_to_json(list(smb.load_signatures(path)))
    assert out == raw.replace(b'"molecule":"dna"', b'"molecule":"DNA"')


def test_reference_written_files_roundtrip_through_the_writer(tmp_path):
    for f in ("47.fa.sig", "genome-s10.fa.gz.sig"):
        sigs = list(smb.load_signatures(os.path.join(GOLDEN, f)))
        p = tmp_path / (f + ".gz")
        with open(p, "wb") as fh:
            smb.save_signatures_to_json(sigs, fh, compression=1)
        again = list(smb.load_signatures(str(p)))
        assert [a.md5sum() for a in again] == [s.md5sum() for s in sigs]
        assert [a.name for a in again] == [s.name for s in sigs]
        want = {sk["md5sum"] for _, sk in _py_sketches(os.path.join(GOLDEN, f))}
        assert {a.md5sum() for a in again} == want


def test_gather_fixture_bruteforce_matches_reference_expectation(golden):
    """The 12-genome gather of tests/test_index_protocol.py:1057-1097, replayed with Python sets on
    the natively parsed fixtures: pins the fixture copies, the parser and the brute-force loop the
    GPU gather tests use as their checker."""
    import glob
    d = os.path.join(GOLDEN, "gather")
    q = SignatureSet.from_files([os.path.join(d, "combined.sig")])
    qi, = q.select(ksize=21)
    subjects = SignatureSet.from_files(sorted(glob.glob(os.path.join(d, "GCF*.sig"))))
    rows = subjects.select(ksize=21)
    assert len(rows) == 12 and int(q.max_hash[qi]) == int(subjects.max_hash[rows[0]])
    remaining = set(q.row(qi).tolist())
    sets = {int(i): set(subjects.row(i).tolist()) for i in rows}
    counters = {i: len(remaining & s) for i, s in sets.items() if remaining & s}
    got = []
    while counters:
        best = max(counters.values())
        i = next(k for k, v in counters.items() if v == best)
        isect = remaining & sets[i]
        got.append([subjects.name(i).split()[0], len(isect)])
        remaining -= sets[i]
        for k in list(counters):
            counters[k] -= len(isect & sets[k])
            if counters[k] <= 0:
                del counters[k]
    assert got == golden["meta"]["gather_k21_expected"]


@pytest.fixture(scope="module")
def ref_data(reference_corpus):
    "sourmash's test-data directory (shrunk; see the reference_corpus fixture)"
    return os.path.join(reference_corpus, "tests", "test-data")


def test_native_parser_on_the_reference_fixture_corpus(ref_data):
    """Every .sig / .sig.gz the reference ships as test data (hundreds of files: old writers,
    abundances, protein / dayhoff / hp, num and scaled, multi-signature files) through the native
    parser, against Python's json on the same bytes."""
    import glob
    paths = sorted(glob.glob(os.path.join(ref_data, "**", "*.sig"), recursive=True) +
                   glob.glob(os.path.join(ref_data, "**", "*.sig.gz"), recursive=True))
    assert len(paths) > 100
    checked = sketches = 0
    for p in paths:
        try:
            want = list(_py_sketches(p))
        except Exception:
            continue                                   # deliberately broken fixtures
        if not all("mins" in sk and "ksize" in sk for _, sk in want):
            continue                                   # other sketch types (e.g. HLL) are out of scope
        ss = SignatureSet.from_files([p])
        assert len(ss) == len(want), p
        for i, (rec, sk) in enumerate(want):
            mins = np.array(sk["mins"], dtype=np.uint64)
            order = np.argsort(mins, kind="stable")
            assert np.array_equal(ss.row(i), mins[order]), p
            if "abundances" in sk:
                assert np.array_equal(ss.abunds[int(ss.offsets[i]):int(ss.offsets[i + 1])],
                                      np.array(sk["abundances"], dtype=np.uint64)[order]), p
            assert int(ss.ksize[i]) == sk["ksize"] and ss.moltype(i).lower() == sk.get("molecule", "dna").lower()
            assert ss.md5sum(i) == sk.get("md5sum", "") and ss.name(i) == (rec.get("name") or "")
            sketches += 1
        checked += 1
    assert checked > 90 and sketches > 150, (checked, sketches)


def _py_records(path):
    opener = gzip.open if path.endswith(".gz") else open
    with opener(path, "rb") as fh:
        data = fh.read()
    lines = data.split(b"\n")
    out, i = [], 0
    fastq = data[:1] == b"@"
    while i < len(lines):
        ln = lines[i].rstrip(b"\r ")
        if not ln:
            i += 1
            continue
        name = ln[1:].decode("utf-8", "replace")
        i += 1
        seq = []
        if fastq:
            while i < len(lines) and not lines[i].startswith(b"+"):
                seq.append(lines[i].strip()); i += 1
            i += 1
            need, got = sum(len(s) for s in seq), 0
            while i < len(lines) and got < need:
                got += len(lines[i].rstrip(b"\r")); i += 1
        else:
            while i < len(lines) and not lines[i].startswith(b">"):
                seq.append(lines[i].strip()); i += 1
        out.append((name, b"".join(seq)))
    return out


def test_native_reader_on_the_reference_sequence_files(ref_data):
    import glob
    paths = []
    for pat in ("*.fa", "*.fa.gz", "*.fna", "*.fna.gz", "*.faa", "*.faa.gz", "*.fq.gz", "*.fq", "*.fastq", "*.fasta"):
        paths += glob.glob(os.path.join(ref_data, "**", pat), recursive=True)
        paths += glob.glob(os.path.join(os.path.dirname(os.path.dirname(ref_data)), "data", pat))
    paths = sorted(set(p for p in paths if os.path.getsize(p) > 0))
    assert len(paths) > 12
    checked = 0
    for p in paths:
        with (gzip.open if p.endswith(".gz") else open)(p, "rb") as fh:
            head = fh.read(1)
        if head not in (b">", b"@"):
            continue
        want = _py_records(p)
        got = read_sequences(p)
        assert [n for n, _ in got] == [n for n, _ in want], p
        assert [s for _, s in got] == [s for _, s in want], p
        checked += 1
    assert checked > 10, checked


def test_bzip2_inputs(tmp_path):
    "bzip2 sequence and signature files (single stream, concatenated streams, truncated)."
    import bz2
    fa = b">a first\nACGTACGTNN\nACG\n>b\nGGGGCCCC\n"
    one = tmp_path / "x.fa.bz2"
    one.write_bytes(bz2.compress(fa))
    assert read_sequences(one) == [("a first", b"ACGTACGTNNACG"), ("b", b"GGGGCCCC")]
    two = tmp_path / "multi.fa.bz2"                                   # pbzip2-style: two streams back to back
    two.write_bytes(bz2.compress(fa[:28]) + bz2.compress(fa[28:]))
    assert read_sequences(two) == read_sequences(one)
    big = os.urandom(1 << 16).hex().upper().encode().replace(b"0", b"A").replace(b"1", b"C")   # incompressible-ish
    rec = b">big\n" + b"\n".join(big[i:i + 80] for i in range(0, len(big), 80)) + b"\n"
    bigf = tmp_path / "big.fa.bz2"
    bigf.write_bytes(bz2.compress(rec, compresslevel=1))
    assert read_sequences(bigf) == [("big", big)]
    src = os.path.join(GOLDEN, "47.fa.sig")
    with open(src, "rb") as fh:
        raw = fh.read()
    sigbz = tmp_path / "47.fa.sig.bz2"
    sigbz.write_bytes(bz2.compress(raw))
    a, b = SignatureSet.from_files([str(sigbz)]), SignatureSet.from_files([src])
    assert np.array_equal(a.mins, b.mins) and np.array_equal(a.offsets, b.offsets) and a.md5sums() == b.md5sums()
    cut = tmp_path / "cut.fa.bz2"
    cut.write_bytes(bigf.read_bytes()[:-200])
    with pytest.raises(Exception, match="corrupt or truncated"):
        read_sequences(cut)
    mixed = RecordBatch([str(one), os.path.join(GOLDEN, "genome-s10.fa.gz"), str(two)], n_threads=2)
    assert mixed.names()[:2] == ["a first", "b"] and mixed.names()[-2:] == ["a first", "b"]


def test_xz_and_zstd_inputs(tmp_path):
    "the other two compression formats the reference's readers sniff (niffler): xz and zstd."
    import ctypes
    import lzma
    fa = b">a first\nACGTACGTNN\nACG\n>b\nGGGGCCCC\n"
    want = [("a first", b"ACGTACGTNNACG"), ("b", b"GGGGCCCC")]
    xz = tmp_path / "x.fa.xz"
    xz.write_bytes(lzma.compress(fa))
    assert read_sequences(xz) == want
    multi = tmp_path / "multi.fa.xz"                                    # concatenated streams
    multi.write_bytes(lzma.compress(fa[:28]) + lzma.compress(fa[28:]))
    assert read_sequences(multi) == want
    big = os.urandom(1 << 16).hex().upper().encode().replace(b"0", b"A").replace(b"1", b"C")
    rec = b">big\n" + b"\n".join(big[i:i + 80] for i in range(0, len(big), 80)) + b"\n"
    bigxz = tmp_path / "big.fa.xz"
    bigxz.write_bytes(lzma.compress(rec, preset=0))
    assert read_sequences(bigxz) == [("big", big)]
    cut = tmp_path / "cut.fa.xz"
    cut.write_bytes(bigxz.read_bytes()[:-300])
    with pytest.raises(Exception, match="corrupt or truncated"):
        read_sequences(cut)
    src = os.path.join(GOLDEN, "47.fa.sig")
    with open(src, "rb") as fh:
        raw = fh.read()
    sigxz = tmp_path / "47.fa.sig.xz"
    sigxz.write_bytes(lzma.compress(raw))
    assert np.array_equal(SignatureSet.from_files([str(sigxz)]).mins, SignatureSet.from_files([src]).mins)
    try:
        z = ctypes.CDLL("libzstd.so.1")
    except OSError:
        pytest.skip("libzstd.so.1 not present")
    z.ZSTD_compressBound.restype = ctypes.c_size_t
    z.ZSTD_compressBound.argtypes = [ctypes.c_size_t]
    z.ZSTD_compress.restype = ctypes.c_size_t
    z.ZSTD_compress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_int]

    def zcompress(data):
        cap = z.ZSTD_compressBound(len(data))
        buf = ctypes.create_string_buffer(cap)
        n = z.ZSTD_compress(buf, cap, data, len(data), 3)
        return buf.raw[:n]
    zs = tmp_path / "x.fa.zst"
    zs.write_bytes(zcompress(fa))
    assert read_sequences(zs) == want
    zs2 = tmp_path / "two.fa.zst"                                       # two frames back to back
    zs2.write_bytes(zcompress(fa[:28]) + zcompress(fa[28:]))
    assert read_sequences(zs2) == want
    bigz = tmp_path / "big.fa.zst"
    bigz.write_bytes(zcompress(rec))
    assert read_sequences(bigz) == [("big", big)]
    cutz = tmp_path / "cut.fa.zst"
    cutz.write_bytes(bigz.read_bytes()[:-300])
    with pytest.raises(Exception, match="corrupt or truncated"):
        read_sequences(cutz)
    sigz = tmp_path / "47.fa.sig.zst"
    sigz.write_bytes(zcompress(raw))
    assert np.array_equal(SignatureSet.from_files([str(sigz)]).mins, SignatureSet.from_files([src]).mins)


@pytest.mark.timeout(300)
def test_malformed_inputs_give_parse_errors_not_crashes():
    """tests/tools/fuzz_ingest.py for a few seconds with a fixed seed: mutated .sig / .zip / FASTA / FASTQ inputs, each batch
    parsed in a child process -- an exception through the ABI is fine, a signal or a hang is not (longer runs, also under
    AddressSanitizer: profiles/r2q_cpu_side_checks.md)."""
    import subprocess
    import sys
    tool = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools", "fuzz_ingest.py")
    r = subprocess.run([sys.executable, tool, "8", "5"], capture_output=True, text=True, timeout=280)
    assert r.returncode == 0 and "no findings" in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]
