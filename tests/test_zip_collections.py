""".zip signature collections without a GPU: the library's zip reader against Python's ``zipfile``,
the collection loader against the plain-file loader, and the ``ZipFileLinearIndex`` /
``CollectionManifest`` scenarios of the reference (tests/test_index.py:688-1064,
tests/test_manifest.py) -- on archives built here from the golden fixtures, and on the reference's
own archives when its checkout is present (build container only).  The one-vs-many kernel is
replaced by the oracle where a search is involved (GPU counterpart: tests/test_gpu_zip.py)."""
import glob
import gzip
import io
import os
import zipfile

import numpy as np
import pytest

import oracle as orc
import sourmash_b200 as smb
from sourmash_b200 import batch as B
from sourmash_b200.exceptions import SourmashError
from sourmash_b200.index import LinearIndex, ZipFileLinearIndex
from sourmash_b200.manifest import CollectionManifest
from sourmash_b200.sbt_storage import ZipStorage
from sourmash_b200.sigset import SignatureSet
from tests.conftest import GOLDEN
from tests.test_index_glue import _FakeSet, cpu_kernels  # noqa: F401  (fixture)

GATHER = sorted(glob.glob(os.path.join(GOLDEN, "gather", "GCF*.sig")))


def _read(path):
    with open(path, "rb") as fh:
        return fh.read()


def _manifest_text(members):
    "SOURMASH-MANIFEST.csv for [(member name, source .sig path)], rows written like the reference does."
    rows = []
    for name, src in members:
        for ss in smb.signature.load_signatures_from_json(src):
            rows.append(CollectionManifest.make_manifest_row(ss, name, include_signature=False))
    out = io.StringIO()
    CollectionManifest(rows).write_to_csv(out, write_header=True)
    return out.getvalue()


def make_zip(path, members, *, manifest=True, compress=zipfile.ZIP_DEFLATED, gz=(), extra=(), zip64=False,
             comment=b"", manifest_members=None):
    """Stored members written through ZipInfo (so zip64 headers can be forced).
    members: [(member name, source .sig path)].  gz: member names stored gzip-compressed
    (like `sourmash sig cat -o x.zip`: signatures/<md5>.sig.gz)."""
    with zipfile.ZipFile(path, "w", compression=compress) as z:
        for name, src in members:
            data = _read(src)
            if name in gz:
                data = gzip.compress(data)
            with z.open(zipfile.ZipInfo(name), "w", force_zip64=zip64) as fh:
                fh.write(data)
        for name, data in extra:
            z.writestr(name, data)
        if manifest:
            z.writestr("SOURMASH-MANIFEST.csv", _manifest_text(manifest_members if manifest_members is not None else members))
        z.comment = comment
    return str(path)


def make_zip_deflated(path, members, **kw):
    "Same as make_zip, every member deflated (writestr honours the archive's compression)."
    manifest = kw.pop("manifest", True)
    gz = kw.pop("gz", ())
    extra = kw.pop("extra", ())
    manifest_members = kw.pop("manifest_members", None)
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_DEFLATED) as z:
        for name, src in members:
            data = _read(src)
            z.writestr(name, gzip.compress(data) if name in gz else data)
        for name, data in extra:
            z.writestr(name, data)
        if manifest:
            z.writestr("SOURMASH-MANIFEST.csv", _manifest_text(manifest_members if manifest_members is not None else members))
    return str(path)


# ---------------------------------------------------------------------------------------------
# zip reader vs zipfile
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["stored", "deflated", "zip64", "comment"])
def test_zipstorage_matches_zipfile(tmp_path, variant):
    members = [("signatures/%d.sig" % i, p) for i, p in enumerate(GATHER[:4])]
    path = tmp_path / "c.zip"
    if variant == "deflated":
        make_zip_deflated(path, members, gz={members[1][0]}, extra=[("build.sh", b"echo hi\n"), ("empty.txt", b"")])
    else:
        make_zip(path, members, compress=zipfile.ZIP_STORED, zip64=variant == "zip64",
                 comment=b"x" * 300 if variant == "comment" else b"", extra=[("build.sh", b"echo hi\n")])
    st = ZipStorage(path)
    with zipfile.ZipFile(path) as z:
        assert st._filenames() == [i.filename for i in z.infolist()]
        for name in z.namelist():
            assert st.load(name) == z.read(name)
    assert st.path == str(path) and st.list_sbts() == []
    with pytest.raises(FileNotFoundError):
        st.load("signatures/nope.sig")


def test_zipstorage_subdir_and_sbts(tmp_path):
    "One directory entry becomes the default subdir (storage/mod.rs:324-363); *.sbt.json are listed."
    path = tmp_path / "s.zip"
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("inner/", b"")
        z.writestr("inner/a.sig", _read(GATHER[0]))
        z.writestr("tree.sbt.json", b"{}")
    st = ZipStorage(path)
    assert st.subdir == "inner/" and st.list_sbts() == ["tree.sbt.json"]
    assert st.load("a.sig") == st.load("inner/a.sig") == _read(GATHER[0])
    st.subdir = "other/"
    assert st.subdir == "other/"
    with pytest.raises(FileNotFoundError):
        st.load("a.sig")


def test_zipstorage_rejects_broken_archives(tmp_path):
    members = [("a.sig", GATHER[0])]
    good = make_zip_deflated(tmp_path / "good.zip", members, manifest=False)
    raw = bytearray(_read(good))
    with pytest.raises(Exception):
        ZipStorage(os.path.join(GOLDEN, "47.fa.sig"))                        # not a zip
    # flip one byte of the compressed stream: inflate fails or the CRC does
    with zipfile.ZipFile(good) as z:
        info = z.getinfo("a.sig")
    raw[info.header_offset + 30 + len("a.sig") + info.compress_size // 2] ^= 0xFF
    bad = tmp_path / "bad.zip"
    bad.write_bytes(bytes(raw))
    with pytest.raises(FileNotFoundError):                                   # reference: ValueError -> FileNotFoundError
        ZipStorage(bad).load("a.sig")
    with pytest.raises(SourmashError, match="CRC|corrupt"):
        SignatureSet.from_files([str(bad)])
    trunc = tmp_path / "trunc.zip"
    trunc.write_bytes(_read(good)[:-30])
    with pytest.raises(Exception):
        ZipStorage(trunc)
    assert not ZipStorage.can_open(os.path.join(GOLDEN, "47.fa.sig")) and ZipStorage.can_open(good)


# ---------------------------------------------------------------------------------------------
# collection loader
# ---------------------------------------------------------------------------------------------
def _same_sets(a, b):
    assert len(a) == len(b)
    assert np.array_equal(a.offsets, b.offsets) and np.array_equal(a.mins, b.mins) and np.array_equal(a.abunds, b.abunds)
    for col in ("ksize", "num", "max_hash", "seed", "hash_function", "has_abund", "n_mins"):
        assert np.array_equal(getattr(a, col), getattr(b, col)), col
    assert [a.name(i) for i in range(len(a))] == [b.name(i) for i in range(len(b))]
    assert a.md5sums() == b.md5sums()


@pytest.mark.parametrize("manifest", [True, False])
@pytest.mark.parametrize("deflate", [True, False])
def test_collection_equals_plain_files(tmp_path, manifest, deflate):
    members = [("signatures/%s" % os.path.basename(p), p) for p in GATHER]
    gz = {members[2][0], members[5][0]}
    maker = make_zip_deflated if deflate else make_zip
    path = maker(tmp_path / "db.zip", members, manifest=manifest, gz=gz, extra=[("README.md", b"not a signature")])
    plain = SignatureSet.from_files(GATHER)
    for threads in (1, 4):
        z = SignatureSet.from_files([path], n_threads=threads)
        _same_sets(z, plain)
        assert z.locations() == [m for m, p in members for _ in smb.signature.load_signatures_from_json(p)]
        assert set(z.file.tolist()) == {0}
    assert plain.locations() == [""] * len(plain)
    # a zip among plain files keeps its place in the input order
    mixed = SignatureSet.from_files([GATHER[0], path, GATHER[1]])
    assert len(mixed) == len(plain) + 2 * (len(plain) // len(GATHER))
    assert mixed.file.tolist() == [0] * (len(plain) // len(GATHER)) + [1] * len(plain) + [2] * (len(plain) // len(GATHER))
    # ... but the reference-ABI JSON loader does NOT take an archive: signatures_load_path parses one (compressed) JSON file
    # like Signature::from_path, and the reference's loader chain (save_load.py) relies on it failing for a zip
    assert list(smb.signature.load_signatures_from_json(path)) == []
    with pytest.raises(Exception):
        list(smb.signature.load_signatures_from_json(path, do_raise=True))


def test_manifest_order_and_md5_filter(tmp_path):
    """With a manifest the members come in manifest order and only listed sketches are kept
    (`if ss in manifest`, index/__init__.py:644-657); without, directory order and *.sig only."""
    members = [("z_first.sig", GATHER[3]), ("a_second.sig", GATHER[1]), ("noext", GATHER[2])]
    listed = [members[1], members[2]]                              # manifest: a_second, then noext; z_first unlisted
    path = make_zip_deflated(tmp_path / "m.zip", members, manifest_members=listed)
    with_mf = SignatureSet.from_files([path])
    want = SignatureSet.from_files([GATHER[1], GATHER[2]])
    _same_sets(with_mf, want)
    no_mf = SignatureSet.from_files([path], use_manifest=False)
    _same_sets(no_mf, SignatureSet.from_files([GATHER[3], GATHER[1]]))
    every = SignatureSet.from_files([path], use_manifest=False, traverse_yield_all=True)
    _same_sets(every, SignatureSet.from_files([GATHER[3], GATHER[1], GATHER[2]]))
    # one member holding several sketches, the manifest lists one of them: the others are dropped
    multi = os.path.join(GOLDEN, "2.fa.sig")
    sigs = list(smb.signature.load_signatures_from_json(multi))
    assert len(sigs) > 1
    rows = [CollectionManifest.make_manifest_row(sigs[1], "multi.sig", include_signature=False)]
    out = io.StringIO()
    CollectionManifest(rows).write_to_csv(out, write_header=True)
    p2 = tmp_path / "multi.zip"
    with zipfile.ZipFile(p2, "w", compression=zipfile.ZIP_DEFLATED) as z:
        z.writestr("multi.sig", _read(multi))
        z.writestr("SOURMASH-MANIFEST.csv", out.getvalue())
    one = SignatureSet.from_files([str(p2)])
    assert len(one) == 1 and one.md5sums() == [sigs[1].md5sum()] and one.n_mins[0] == len(sigs[1].minhash)
    assert lib_n_signatures(one) == 1
    # a manifest naming a member that is not there is an error, like storage.load raising
    p3 = tmp_path / "dangling.zip"
    with zipfile.ZipFile(p3, "w") as z:
        z.writestr("SOURMASH-MANIFEST.csv", out.getvalue())
    with pytest.raises(SourmashError, match="multi.sig"):
        SignatureSet.from_files([str(p3)])


def lib_n_signatures(sset):
    from sourmash_b200._lowlevel import lib
    return int(lib.smb_sigs_n_signatures(sset._ptr))


def test_empty_archive(tmp_path):
    path = tmp_path / "empty.zip"
    with zipfile.ZipFile(path, "w"):
        pass
    assert len(SignatureSet.from_files([str(path)])) == 0
    idx = ZipFileLinearIndex.load(str(path))
    assert len(idx) == 0 and not idx and list(idx.signatures()) == []


# ---------------------------------------------------------------------------------------------
# manifests
# ---------------------------------------------------------------------------------------------
def test_manifest_csv_round_trip_and_select(tmp_path):
    members = [("signatures/%s" % os.path.basename(p), p) for p in GATHER[:3]] + [("p/2.sig", os.path.join(GOLDEN, "2.fa.sig"))]
    text = _manifest_text(members)
    mf = CollectionManifest.load_from_csv(io.StringIO(text))
    out = io.StringIO()
    mf.write_to_csv(out, write_header=True)
    assert out.getvalue() == text
    assert list(mf.locations()) == [m for m, _ in members]
    path = make_zip_deflated(tmp_path / "db.zip", members)
    sset = SignatureSet.from_files([path])
    built = CollectionManifest.from_signature_set(sset, md5s=sset.md5sums())
    assert built == mf and len(built) == len(mf) == len(sset)
    k31 = mf.select_to_manifest(ksize=31)
    assert 0 < len(k31) < len(mf) and all(r["ksize"] == 31 for r in k31.rows)
    assert len(mf.select_to_manifest(moltype="protein")) == 0
    assert len(mf.select_to_manifest(num=500)) == len([r for r in mf.rows if r["num"] == 500])
    assert len(mf.select_to_manifest(scaled=1000)) == len([r for r in mf.rows if r["scaled"]])
    assert len(mf.select_to_manifest(abund=True)) == len([r for r in mf.rows if r["with_abundance"]])
    some = next(smb.signature.load_signatures_from_json(GATHER[0]))
    assert some in mf and some not in mf.select_to_manifest(ksize=12345)
    with pytest.raises(ValueError):
        mf.select_to_manifest(moltype="rna")
    with pytest.raises(ValueError):
        CollectionManifest.load_from_csv(io.StringIO("internal_location,md5\n"))
    with pytest.raises(ValueError):
        CollectionManifest.load_from_csv(io.StringIO("# SOURMASH-MANIFEST-VERSION: 2.0\n"))


# ---------------------------------------------------------------------------------------------
# ZipFileLinearIndex (tests/test_index.py:688-1064)
# ---------------------------------------------------------------------------------------------
@pytest.fixture
def zip_db(tmp_path):
    members = [("signatures/%s" % os.path.basename(p), p) for p in GATHER]
    return make_zip_deflated(tmp_path / "gather.zip", members, extra=[("extra.noext", _read(os.path.join(GOLDEN, "47.fa.sig")))],
                             manifest_members=members + [("extra.noext", os.path.join(GOLDEN, "47.fa.sig"))])


def test_zipfile_does_not_exist(tmp_path):                                    # :688-697
    with pytest.raises(FileNotFoundError):
        ZipFileLinearIndex.load(str(tmp_path / "missing.zip"))


@pytest.mark.parametrize("use_manifest", [True, False])
def test_zipfile_api(zip_db, use_manifest):                                   # :821-860, :1001-1029
    idx = ZipFileLinearIndex.load(zip_db, use_manifest=use_manifest)
    n_plain = len(SignatureSet.from_files(GATHER))
    want = n_plain + 1 if use_manifest else n_plain                           # extra.noext only through the manifest
    sigs = list(idx.signatures())
    assert len(sigs) == len(idx) == want and bool(idx)
    assert idx.location == zip_db and idx.is_database
    assert (idx.manifest is not None) == use_manifest
    with pytest.raises(NotImplementedError):
        idx.insert(sigs[0])
    with pytest.raises(NotImplementedError):
        idx.save("xxx")
    everything = ZipFileLinearIndex.load(zip_db, traverse_yield_all=True, use_manifest=use_manifest)
    assert len(everything) == len(list(everything.signatures())) == n_plain + 1
    assert len(everything.storage._filenames()) == len(GATHER) + 2
    assert all(s.md5sum() == m for s, m in zip(sigs, idx._sigset.md5sums()))
    assert [loc for _, loc in idx.signatures_with_location()] == [zip_db] * want
    internal = list(everything._signatures_with_internal())
    assert len(internal) == n_plain + 1 and internal[-1][1] == "extra.noext"


@pytest.mark.parametrize("use_manifest", [True, False])
def test_zipfile_select(zip_db, use_manifest):                                # :909-999
    idx = ZipFileLinearIndex.load(zip_db, use_manifest=use_manifest)
    pre = LinearIndex(idx.signatures())
    for kw in ({"ksize": 21}, {"ksize": 31, "moltype": "DNA"}, {"moltype": "protein"}, {"scaled": 10000},
               {"num": 500}, {"abund": True}, {"abund": False}, {"scaled": 1000, "containment": True}):
        sel = idx.select(**kw)
        assert len(sel) == len(list(sel.signatures())) == len(pre.select(**kw)), kw
        assert [s.md5sum() for s in sel.signatures()] == [s.md5sum() for s in pre.select(**kw).signatures()]
    twice = idx.select(ksize=21).select(moltype="DNA")
    assert len(twice) == len(pre.select(ksize=21, moltype="DNA")) > 0
    if use_manifest:
        assert len(twice.manifest) == len(twice)
        assert len(idx.select(ksize=21).select(ksize=31)) == 0
    else:
        with pytest.raises(ValueError, match="incompatible select"):
            idx.select(ksize=21).select(ksize=31)
    with pytest.raises(ValueError):
        idx.select(ksize="21")
    if use_manifest:                                    # manifest.py:300-320 only filters on scaled
        assert len(idx.select(containment=True)) == len(pre.select(scaled=1, containment=True))
    else:                                               # select_signature, index/__init__.py:367-371
        with pytest.raises(ValueError):
            idx.select(containment=True)


def test_zipfile_search_matches_linear_index(zip_db, cpu_kernels, monkeypatch):
    "search / prefetch over the archive == over the same signatures loaded one by one."
    monkeypatch.setattr(SignatureSet, "to_sketchset",
                        lambda self, rows=None, scaled=None, with_abunds=False:
                        _FakeSet([self.row(i) for i in (range(len(self)) if rows is None else rows)]))
    idx = ZipFileLinearIndex.load(zip_db).select(ksize=21)
    lin = LinearIndex(idx.signatures())
    query = smb.signature.load_one_signature_from_json(os.path.join(GOLDEN, "gather", "combined.sig"), ksize=21)
    a = idx.search(query, threshold=0.0, do_containment=True)
    b = lin.search(query, threshold=0.0, do_containment=True)
    assert [(r.score, r.signature.md5sum()) for r in a] == [(r.score, r.signature.md5sum()) for r in b] and len(a) == 12
    assert all(r.location == zip_db for r in a)
    pa = [(r.score, r.signature.md5sum()) for r in idx.prefetch(query, 50000)]
    assert pa == [(r.score, r.signature.md5sum()) for r in lin.prefetch(query, 50000)] and pa
    assert len(idx._objects) <= 12                                             # objects built only for returned subjects


# ---------------------------------------------------------------------------------------------
# the reference's own archives, shrunk (golden/make_reference_corpus.py: every member kept, sketches cut short)
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ref_data(reference_corpus):
    "sourmash's test-data directory (shrunk; see the reference_corpus fixture)"
    return os.path.join(reference_corpus, "tests", "test-data")


def test_reference_archives_load_like_zipfile_and_json(ref_data):
    import json
    paths = [p for p in glob.glob(os.path.join(ref_data, "**", "*.zip"), recursive=True)]
    assert len(paths) > 10
    checked = 0
    for path in paths:
        try:
            z = zipfile.ZipFile(path)
        except zipfile.BadZipFile:
            continue
        st = ZipStorage(path)
        assert st._filenames() == [i.filename for i in z.infolist()]
        for info in z.infolist():
            if not info.is_dir():
                assert st.load(info.filename) == z.read(info), (path, info.filename)
        names = z.namelist()
        sset = SignatureSet.from_files([path])
        if "SOURMASH-MANIFEST.csv" in names:
            mf = CollectionManifest.load_from_csv(io.StringIO(z.read("SOURMASH-MANIFEST.csv").decode()))
            locs = list(mf.locations())
            assert sorted(set(sset.locations()), key=locs.index) == [loc for loc in locs if loc in set(sset.locations())]
            assert set(sset.md5sums()) <= mf._md5_set
            built = CollectionManifest.from_signature_set(sset, md5s=sset.md5sums())
            by_md5 = {r["md5"]: r for r in mf.rows}
            for row in built.rows:
                ref = by_md5[row["md5"]]
                for key in ("ksize", "moltype", "num", "scaled", "n_hashes", "with_abundance", "name"):
                    assert row[key] == ref[key], (path, key)
        else:
            members = [n for n in names if n.endswith(".sig") or n.endswith(".sig.gz")]
            n = 0
            for m in members:
                data = z.read(m)
                if data[:2] == b"\x1f\x8b":
                    data = gzip.decompress(data)
                n += sum(len(s["signatures"]) for s in json.loads(data))
            assert len(sset) == n, path
        checked += 1
    assert checked > 10


@pytest.mark.parametrize("use_manifest", [True, False])
def test_reference_all_zip_scenarios(ref_data, use_manifest):                           # tests/test_index.py:821-927
    path = os.path.join(ref_data, "prot", "all.zip")
    idx = ZipFileLinearIndex.load(path, use_manifest=use_manifest)
    assert len(list(idx.signatures())) == len(idx) == (8 if use_manifest else 7)
    all_idx = ZipFileLinearIndex.load(path, traverse_yield_all=True, use_manifest=use_manifest)
    assert len(list(all_idx.signatures())) == len(all_idx) == 8
    assert len(all_idx.storage._filenames()) == 13
    assert len(all_idx.select(moltype="DNA")) == 2
    assert len(idx.select(moltype="DNA")) == (2 if use_manifest else 1)
    assert len(LinearIndex(idx.signatures()).select(moltype="DNA")) == (2 if use_manifest else 1)
    assert len(idx.select(ksize=19, moltype="protein")) == 2
    abund = ZipFileLinearIndex.load(os.path.join(ref_data, "track_abund", "track_abund.zip"), use_manifest=use_manifest)
    assert len(abund.select(abund=False)) == 2 and len(abund.select(abund=True)) == 2 and len(abund.select(abund=None)) == 2
    twice = ZipFileLinearIndex.load(path, use_manifest=use_manifest).select(ksize=19).select(moltype="protein")
    assert len(list(twice.signatures())) == 2
