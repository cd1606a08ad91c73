"""`sourmash scripts b200sketch | b200compare | b200search | b200gather | b200prefetch` against the REFERENCE's own commands.

north_star asks for the hot paths "behind the reference's own plugin API": the reference loads command plugins from the
entry-point group `sourmash.cli_script` (src/sourmash/plugins.py:8-12, 91-186).  Every plugin command is compared with the
reference's own command on the same inputs:

    sourmash sketch dna / protein / translate   vs   sourmash scripts b200sketch      -> equal signatures
    sourmash compare                            vs   sourmash scripts b200compare     -> equal matrix, labels, CSV
    sourmash search / gather / prefetch         vs   sourmash scripts b200search ...  -> byte-identical CSV files

The reference's outputs are stored in golden/plugin_cli.tar.gz; the plugin commands run here (`python -m
sourmash_b200.plugin`, on the emulated library, so no GPU is needed).  The inputs are the sourmash test data the suite
stores: golden/reference_corpus.tar.gz with the full-size files of golden/ laid over it.  With SOURMASH_CHECKOUT naming a
sourmash checkout, the reference's commands run live instead (its package loaded in place over the emulated library, as in
test_reference_python_over_abi.py, and finding this package's entry points in a dist-info written next to it) and the
archive is written anew from what they produce."""
import csv
import glob
import gzip
import io
import json
import os
import shutil
import subprocess
import sys
import tarfile
import zipfile
import zlib
from types import SimpleNamespace

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_reference_python_over_abi as over_abi  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
STORED = os.path.join(GOLDEN, "plugin_cli.tar.gz")
CHECKOUT = os.environ.get("SOURMASH_CHECKOUT")
DATA = "data"                   # the inputs, relative to the working directory: the reports quote these paths
WORK_MARK = "{WORK}"            # the absolute working directory in stored text (a zip database reports its absolute path)
FULL_SIZE = ["gather", "47.fa.sig", "63.fa.sig", "2.fa.sig", "genome-s10.fa.gz", "ecoli.faa", "ecoli.genes.fna"]

COMMANDS = ("B200Sketch", "B200Compare", "B200Search", "B200Gather", "B200Prefetch")


def _outputs(args):
    "the files a reference command line writes: -o, --csv, and the labels next to a compare matrix"
    out = [args[i + 1] for i, a in enumerate(args[:-1]) if a in ("-o", "--csv")]
    return out + [o + ".labels.txt" for o in out if o.endswith(".npy")]


def cat_signatures(paths, out):
    "the signatures of `paths` in one .sig file, or in one .zip with a manifest and one signatures/<md5>.sig.gz per sketch, as `sig cat` writes them"
    records = []
    for p in paths:
        with open(p) as fh:
            records += json.load(fh)
    if not out.endswith(".zip"):
        with open(out, "w") as fh:
            json.dump(records, fh)
        return
    rows = ["# SOURMASH-MANIFEST-VERSION: 1.0\n"
            "internal_location,md5,md5short,ksize,moltype,num,scaled,n_hashes,with_abundance,name,filename\n"]
    with zipfile.ZipFile(out, "w") as z:
        for rec, sk in ((r, sk) for r in records for sk in r["signatures"]):      # one member and one row per sketch
            member = "signatures/%s.sig.gz" % sk["md5sum"]
            z.writestr(member, gzip.compress(json.dumps([dict(rec, signatures=[sk])]).encode(), mtime=0))
            scaled = (2**64 - 1) // sk["max_hash"] if sk.get("max_hash") else 0      # what sourmash derives from max_hash
            rows.append(",".join([member, sk["md5sum"], sk["md5sum"][:8], str(sk["ksize"]), sk.get("molecule", "dna").upper(),
                                  str(0 if scaled else sk.get("num", 0)), str(scaled), str(len(sk["mins"])), str(int("abundances" in sk)),
                                  '"%s"' % (rec.get("name") or ""), '"%s"' % (rec.get("filename") or "")]) + "\n")
        z.writestr("SOURMASH-MANIFEST.csv", "".join(rows))


@pytest.fixture(scope="module")
def cli(tmp_path_factory, reference_corpus):
    sys.path.insert(0, os.path.join(HERE, "host_emul"))
    try:
        import emul_lib
    finally:
        sys.path.pop(0)
    tmp = str(tmp_path_factory.mktemp("refcli"))
    site = os.path.join(tmp, "site")
    os.makedirs(site)
    env = dict(os.environ, PYTHONPATH=site, PYTHONDONTWRITEBYTECODE="1")
    if CHECKOUT:
        over_abi.REF = CHECKOUT
        over_abi._stub_package(tmp, emul_lib.build())
        info = os.path.join(site, "sourmash_b200-0.1.0.dist-info")     # what `pip install .` writes from pyproject.toml
        os.makedirs(info)
        with open(os.path.join(info, "METADATA"), "w") as fh:
            fh.write("Metadata-Version: 2.1\nName: sourmash_b200\nVersion: 0.1.0\n")
        with open(os.path.join(info, "entry_points.txt"), "w") as fh:
            fh.write("[sourmash.cli_script]\n" + "".join("%s = sourmash_b200.plugin:Command_%s\n" % (c.lower(), c) for c in COMMANDS))
        env["PYTHONPATH"] = os.pathsep.join([site, os.path.join(tmp, "reftests")])
    with open(os.path.join(ROOT, "pyproject.toml")) as fh:
        declared = [line.split("=")[0].strip() for line in fh if "sourmash_b200.plugin:Command_" in line]
    assert declared == [c.lower() for c in COMMANDS]                   # the entry points are the declared ones
    with open(os.path.join(site, "sitecustomize.py"), "w") as fh:       # this package binds the emulated library
        fh.write("import sys\nsys.path.insert(0, %r); sys.path.insert(0, %r)\nimport emulated_boot\nemulated_boot.install()\n"
                 % (os.path.join(HERE, "host_emul"), ROOT))
    work = os.path.join(tmp, "work")
    shutil.copytree(os.path.join(reference_corpus, "tests", "test-data"), os.path.join(work, DATA))
    for name in FULL_SIZE:                                               # full-size copies of the files golden/ holds
        src = os.path.join(GOLDEN, name)
        if os.path.isdir(src):
            shutil.copytree(src, os.path.join(work, DATA, name), dirs_exist_ok=True)
        else:
            shutil.copy(src, os.path.join(work, DATA, name))
    stored = {}
    if not CHECKOUT:
        with tarfile.open(STORED) as tar:
            stored = {m.name: tar.extractfile(m).read() for m in tar.getmembers()}

    def _text(data, to_stored):
        a, b = (work.encode(), WORK_MARK.encode()) if to_stored else (WORK_MARK.encode(), work.encode())
        return data.replace(a, b)

    def run(*args, rc=(0,)):
        args = [str(a) for a in args]
        if args[0] == "scripts" and len(args) > 1 and args[1].startswith("b200"):   # the plugin: this package, here
            r = subprocess.run([sys.executable, "-m", "sourmash_b200.plugin"] + args[1:], capture_output=True, text=True,
                               env=env, cwd=work, timeout=900)
            assert r.returncode in rc, " ".join(args) + "\n" + r.stdout[-2000:] + r.stderr[-3000:]
            return r
        key = " ".join(args)                                             # the reference: stored outputs, or run live
        if CHECKOUT:
            r = subprocess.run([sys.executable, "-m", "sourmash"] + args, capture_output=True, text=True, env=env,
                               cwd=work, timeout=900)
            assert r.returncode in rc, key + "\n" + r.stdout[-2000:] + r.stderr[-3000:]
            stored["console/" + key.replace("/", "|")] = _text((r.stdout + r.stderr).encode(), True)
            for name in _outputs(args):
                with open(os.path.join(work, name), "rb") as fh:
                    stored[name] = _text(fh.read(), True)
            return r
        for name in _outputs(args):
            assert name in stored, "no stored reference output for: " + key
            with open(os.path.join(work, name), "wb") as fh:
                fh.write(_text(stored[name], False))
        out = _text(stored.get("console/" + key.replace("/", "|"), b""), False).decode()
        return SimpleNamespace(returncode=0, stdout=out, stderr="")

    def load(path):                                                      # this package's loader
        code = ("import sourmash_b200 as s, sys, json\n"
                "print(json.dumps(sorted([ss.name, ss.filename, ss.md5sum(), ss.minhash.ksize, ss.minhash.moltype, "
                "ss.minhash.scaled, ss.minhash.num, int(ss.minhash.track_abundance), sorted(ss.minhash.hashes.items())] "
                "for ss in s.load_file_as_signatures(sys.argv[1]))))")
        r = subprocess.run([sys.executable, "-c", code, path], capture_output=True, text=True, env=env, cwd=work, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        return r.stdout

    def together(*cmdlines):
        "several command lines at once (each is a process that spends a second importing its package)"
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(len(cmdlines)) as pool:
            return list(pool.map(lambda c: run(*c), cmdlines))

    def loads(*paths):
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(len(paths)) as pool:
            return list(pool.map(load, paths))

    run.work, run.load, run.loads, run.together = work, load, loads, together
    run.glob = lambda pattern: [os.path.relpath(p, work) for p in glob.glob(os.path.join(work, pattern))]
    yield run
    if CHECKOUT:                                                         # the reference's outputs, for runs without it
        buf = io.BytesIO()
        with tarfile.open(fileobj=buf, mode="w") as tar:
            for name in sorted(stored):
                ti = tarfile.TarInfo(name)
                ti.size, ti.mode = len(stored[name]), 0o644
                tar.addfile(ti, io.BytesIO(stored[name]))
        with open(STORED, "wb") as fh:
            fh.write(gzip.compress(buf.getvalue(), compresslevel=9, mtime=0))


def test_the_reference_lists_the_plugin_commands(cli):
    r = cli("scripts", rc=(0, 1))                          # no command given: the list of commands, exit status 1
    out = r.stderr + r.stdout
    from sourmash_b200 import plugin
    for c in COMMANDS:
        assert "sourmash scripts %s" % c.lower() in out
        assert getattr(plugin, "Command_" + c).description in out


@pytest.mark.parametrize("kind,params,files", [
    ("dna", "k=21,k=31,k=51,scaled=1000", ["genome-s10.fa.gz", "genome-s11.fa.gz", "genome-s12.fa.gz"]),
    ("dna", "k=31,scaled=100,abund", ["short.fa", "short2.fa"]),
    ("dna", "k=21,num=500", ["genome-s10.fa.gz"]),
    ("protein", "k=7,scaled=10", ["ecoli.faa"]),
    ("translate", "k=7,scaled=10,dayhoff", ["short.fa"]),
])
def test_sketch_commands_write_equal_signatures(cli, kind, params, files):
    paths = [os.path.join(DATA, f) for f in files]
    tag = "%s_%08x" % (kind, zlib.crc32(params.encode()))
    extra, plugin_params = [], params
    if kind != "dna":
        moltype = "dayhoff" if "dayhoff" in params else "hp" if ",hp" in params else "protein"
        extra = ["--moltype", moltype] + (["--input-is-protein"] if kind == "protein" else [])
        plugin_params = params.replace(",dayhoff", "").replace(",hp", "")
    cli.together(["sketch", kind, "-p", params, *paths, "-o", tag + "_ref.sig"],
                 ["scripts", "b200sketch", "-p", plugin_params, *paths, "-o", tag + "_b200.sig", *extra])
    want, got = cli.loads(tag + "_ref.sig", tag + "_b200.sig")
    assert len(want) > 100 and got == want
    assert open(os.path.join(cli.work, tag + "_ref.sig")).read() == open(os.path.join(cli.work, tag + "_b200.sig")).read()   # the .sig files themselves


@pytest.mark.parametrize("flags,files", [
    (["--singleton"], ["short.fa"]),
    (["--name-from-first"], ["short.fa", "short2.fa"]),
    (["--merge", "all of them"], ["short.fa", "short2.fa", "short3.fa"]),
    (["--singleton", "--name-from-first"], ["ecoli.genes.fna"]),
])
def test_sketch_naming_modes_write_equal_signatures(cli, flags, files):
    "--singleton (one signature per record), --name-from-first, --merge NAME: names, filenames and sketches (command_sketch.py:662-789)"
    paths = [os.path.join(DATA, f) for f in files]
    tag = "naming_" + "".join(f.strip("-")[:4] for f in flags if f.startswith("--"))
    cli.together(["sketch", "dna", "-p", "k=21,k=31,scaled=10", *paths, "-o", tag + "_ref.sig", *flags],
                 ["scripts", "b200sketch", "-p", "k=21,k=31,scaled=10", *paths, "-o", tag + "_b200.sig", *flags])
    want, got = cli.loads(tag + "_ref.sig", tag + "_b200.sig")
    assert len(want) > 100 and got == want
    assert open(os.path.join(cli.work, tag + "_ref.sig")).read() == open(os.path.join(cli.work, tag + "_b200.sig")).read()   # the .sig files themselves


def test_sketch_of_fastq_and_invalid_bases(cli):
    "a FASTQ file; records with N and IUPAC codes (skipped k-mers, force = the CLI default)"
    reads = [("r1", "ACGTTGCAACGTTGCATGCATGCAAGCTNNACGTACGATCGATCGTACGATGCATGCA"),
             ("r2 second", "acgtacgtRYacgtagctagctagcatcgatcgatcgatgcatgcatgcatgcag")]
    with open(os.path.join(cli.work, "reads.fq"), "w") as fh:
        for name, seq in reads:
            fh.write("@%s\n%s\n+\n%s\n" % (name, seq, "I" * len(seq)))
    cli.together(["sketch", "dna", "-p", "k=11,scaled=1", "reads.fq", "-o", "fq_ref.sig"],
                 ["scripts", "b200sketch", "-p", "k=11,scaled=1", "reads.fq", "-o", "fq_b200.sig"])
    want, got = cli.loads("fq_ref.sig", "fq_b200.sig")
    assert len(want) > 100 and got == want


def test_compare_command_writes_the_same_matrix(cli):
    sigs = sorted(cli.glob(os.path.join(DATA, "gather", "GCF*.sig")))
    cli.together(["compare", *sigs, "-k", "21", "-o", "ref.npy", "--csv", "ref_cmp.csv"],
                 ["scripts", "b200compare", *sigs, "-k", "21", "-o", "b200.npy", "--csv", "b200_cmp.csv"])
    w = cli.work
    a, b = np.load(os.path.join(w, "ref.npy")), np.load(os.path.join(w, "b200.npy"))
    assert a.shape == (12, 12) and np.array_equal(a, b) and 0 < a[a < 1].max() < 1
    assert open(os.path.join(w, "ref.npy.labels.txt")).read() == open(os.path.join(w, "b200.npy.labels.txt")).read()
    assert list(csv.reader(open(os.path.join(w, "ref_cmp.csv")))) == list(csv.reader(open(os.path.join(w, "b200_cmp.csv"))))


@pytest.mark.parametrize("flags", [["--containment"], ["--max-containment"], ["--avg-containment"], ["--estimate-ani"],
                                   ["--containment", "--estimate-ani"], ["--max-containment", "--estimate-ani"],
                                   ["--distance-matrix"], ["--scaled", "2000"]])
def test_compare_flags_write_the_same_matrix(cli, flags):
    "the other matrices of `sourmash compare`: containment forms, ANI, distances, a coarser --scaled"
    sigs = sorted(cli.glob(os.path.join(DATA, "gather", "GCF*.sig")))[:6]
    tag = "cmp" + "".join(flags).replace("-", "")
    cli.together(["compare", *sigs, "-k", "21", "-o", tag + "_ref.npy", "--csv", tag + "_ref.csv", *flags],
                 ["scripts", "b200compare", *sigs, "-k", "21", "-o", tag + "_b200.npy", "--csv", tag + "_b200.csv", *flags])
    w = cli.work
    a, b = np.load(os.path.join(w, tag + "_ref.npy")), np.load(os.path.join(w, tag + "_b200.npy"))
    assert a.shape == (6, 6) and np.array_equal(a, b)
    assert open(os.path.join(w, tag + "_ref.csv")).read() == open(os.path.join(w, tag + "_b200.csv")).read()


@pytest.mark.parametrize("flags", [[], ["--ignore-abundance"], ["--containment"]])
def test_compare_of_abundance_sketches(cli, flags):
    "sketches with abundances: angular similarity unless --ignore-abundance; a flat sketch among them; containment ignores abundances"
    sigs = [os.path.join(DATA, "track_abund", f) for f in ("47.fa.sig", "63.fa.sig")] + [os.path.join(DATA, "2.fa.sig")]
    tag = "cmpab" + "".join(flags).replace("-", "")
    cli.together(["compare", *sigs, "-k", "31", "-o", tag + "_ref.npy", *flags],
                 ["scripts", "b200compare", *sigs, "-k", "31", "-o", tag + "_b200.npy", *flags])
    a, b = np.load(os.path.join(cli.work, tag + "_ref.npy")), np.load(os.path.join(cli.work, tag + "_b200.npy"))
    assert a.shape == (3, 3) and np.array_equal(a, b) and 0 < a[0, 1] < 1


def _same_file(cli, a, b, min_rows):
    ta, tb = open(os.path.join(cli.work, a)).read(), open(os.path.join(cli.work, b)).read()
    assert ta.count("\n") > min_rows and ta == tb


@pytest.mark.parametrize("flags", [[], ["--containment"], ["--max-containment"], ["--best-only"]])
def test_search_command_writes_the_same_csv(cli, flags):
    sigs = sorted(cli.glob(os.path.join(DATA, "gather", "GCF*.sig")))
    tag = "search" + "".join(flags).replace("-", "")
    cli.together(["search", sigs[0], *sigs, "-k", "21", "--threshold", "0.01", "-o", tag + "_ref.csv", *flags],
                 ["scripts", "b200search", sigs[0], *sigs, "-k", "21", "--threshold", "0.01", "-o", tag + "_b200.csv", *flags])
    _same_file(cli, tag + "_ref.csv", tag + "_b200.csv", 1 if "--best-only" in flags else 5)


@pytest.mark.parametrize("threshold_bp", ["0", "50000"])
def test_gather_and_prefetch_commands_write_the_same_csv(cli, threshold_bp):
    query = os.path.join(DATA, "gather", "combined.sig")
    sigs = sorted(cli.glob(os.path.join(DATA, "gather", "GCF*.sig")))
    for cmd in ("gather", "prefetch"):
        tag = "%s_%s" % (cmd, threshold_bp)
        cli.together([cmd, query, *sigs, "-k", "21", "--threshold-bp", threshold_bp, "-o", tag + "_ref.csv"],
                     ["scripts", "b200" + cmd, query, *sigs, "-k", "21", "--threshold-bp", threshold_bp, "-o", tag + "_b200.csv"])
        _same_file(cli, tag + "_ref.csv", tag + "_b200.csv", 5)


def test_gather_of_an_abundance_query_writes_the_same_csv(cli):
    "weighted columns (average_abund, f_unique_weighted, ...): a query with abundances against flat genomes"
    query = os.path.join(DATA, "track_abund", "47.fa.sig")
    dbs = [os.path.join(DATA, f) for f in ("47.fa.sig", "63.fa.sig", "2.fa.sig")]
    cli.together(["gather", query, *dbs, "-k", "31", "--threshold-bp", "0", "-o", "abund_ref.csv"],
                 ["scripts", "b200gather", query, *dbs, "-k", "31", "--threshold-bp", "0", "-o", "abund_b200.csv"])
    _same_file(cli, "abund_ref.csv", "abund_b200.csv", 1)


@pytest.mark.parametrize("flags", [[], ["--best-only"], ["--containment", "--best-only"]])
def test_search_of_one_multi_signature_database(cli, flags):
    "all subjects in ONE file: --best-only ratchets its threshold inside a database"
    sigs = sorted(cli.glob(os.path.join(DATA, "gather", "GCF*.sig")))
    if not os.path.exists(os.path.join(cli.work, "all12.sig")):
        cat_signatures([os.path.join(cli.work, p) for p in sigs[::-1]], os.path.join(cli.work, "all12.sig"))   # query's own last
    tag = "one" + "".join(flags).replace("-", "")
    cli.together(["search", sigs[3], "all12.sig", "-k", "21", "--threshold", "0.01", "-o", tag + "_ref.csv", *flags],
                 ["scripts", "b200search", sigs[3], "all12.sig", "-k", "21", "--threshold", "0.01", "-o", tag + "_b200.csv", *flags])
    _same_file(cli, tag + "_ref.csv", tag + "_b200.csv", 1)
    if flags:
        rows = open(os.path.join(cli.work, tag + "_ref.csv")).read().count("\n") - 1
        assert 1 <= rows < 8                                            # fewer than without the ratchet


def test_a_zip_collection_as_the_database(cli):
    "the twelve genomes in one .zip: every command, same files; a zip reports its absolute path"
    sigs = sorted(cli.glob(os.path.join(DATA, "gather", "GCF*.sig")))
    query = os.path.join(DATA, "gather", "combined.sig")
    cat_signatures([os.path.join(cli.work, p) for p in sigs], os.path.join(cli.work, "all12.zip"))
    cli.together(["gather", query, "all12.zip", "-k", "21", "--threshold-bp", "0", "-o", "zip_gather_ref.csv"],
                 ["scripts", "b200gather", query, "all12.zip", "-k", "21", "--threshold-bp", "0", "-o", "zip_gather_b200.csv"],
                 ["prefetch", query, "all12.zip", "-k", "21", "--threshold-bp", "0", "-o", "zip_prefetch_ref.csv"],
                 ["scripts", "b200prefetch", query, "all12.zip", "-k", "21", "--threshold-bp", "0", "-o", "zip_prefetch_b200.csv"])
    cli.together(["search", sigs[0], "all12.zip", "-k", "21", "--threshold", "0.01", "-o", "zip_search_ref.csv"],
                 ["scripts", "b200search", sigs[0], "all12.zip", "-k", "21", "--threshold", "0.01", "-o", "zip_search_b200.csv"],
                 ["compare", "all12.zip", "-k", "21", "-o", "zip_ref.npy"],
                 ["scripts", "b200compare", "all12.zip", "-k", "21", "-o", "zip_b200.npy"])
    for name in ("gather", "prefetch", "search"):
        _same_file(cli, "zip_%s_ref.csv" % name, "zip_%s_b200.csv" % name, 5)
    assert np.array_equal(np.load(os.path.join(cli.work, "zip_ref.npy")), np.load(os.path.join(cli.work, "zip_b200.npy")))
    assert open(os.path.join(cli.work, "zip_ref.npy.labels.txt")).read() == open(os.path.join(cli.work, "zip_b200.npy.labels.txt")).read()


def test_a_directory_as_the_database_and_the_scaled_option(cli):
    """A directory (with a sub-directory) of .sig files is one database whose matches report the file they came from; --scaled
    downsamples the query first, and the reports then quote that sketch; protein sketches."""
    import shutil
    sigs = sorted(cli.glob(os.path.join(DATA, "gather", "GCF*.sig")))
    query = os.path.join(DATA, "gather", "combined.sig")
    db = os.path.join(cli.work, "dbdir")
    os.makedirs(os.path.join(db, "sub"))
    for i, p in enumerate(sigs):
        shutil.copy(os.path.join(cli.work, p), os.path.join(db, "sub") if i % 3 == 0 else db)
    cli.together(["gather", query, "dbdir", "-k", "21", "--threshold-bp", "0", "-o", "dir_gather_ref.csv"],
                 ["scripts", "b200gather", query, "dbdir", "-k", "21", "--threshold-bp", "0", "-o", "dir_gather_b200.csv"],
                 ["search", sigs[0], "dbdir", "--best-only", "-k", "21", "--threshold", "0.01", "-o", "dir_search_ref.csv"],
                 ["scripts", "b200search", sigs[0], "dbdir", "--best-only", "-k", "21", "--threshold", "0.01", "-o", "dir_search_b200.csv"])
    cli.together(["gather", query, *sigs, "-k", "21", "--threshold-bp", "0", "--scaled", "20000", "-o", "sc_gather_ref.csv"],
                 ["scripts", "b200gather", query, *sigs, "-k", "21", "--threshold-bp", "0", "--scaled", "20000", "-o", "sc_gather_b200.csv"],
                 ["compare", "dbdir", "-k", "21", "-o", "dir_ref.npy"],
                 ["scripts", "b200compare", "dbdir", "-k", "21", "-o", "dir_b200.npy"])
    _same_file(cli, "dir_gather_ref.csv", "dir_gather_b200.csv", 5)
    _same_file(cli, "dir_search_ref.csv", "dir_search_b200.csv", 1)
    _same_file(cli, "sc_gather_ref.csv", "sc_gather_b200.csv", 3)
    assert np.array_equal(np.load(os.path.join(cli.work, "dir_ref.npy")), np.load(os.path.join(cli.work, "dir_b200.npy")))
    prot = sorted(cli.glob(os.path.join(DATA, "prot", "protein", "*.sig")))
    cli.together(["search", prot[0], *prot, "--protein", "--threshold", "0.0", "-o", "prot_search_ref.csv"],
                 ["scripts", "b200search", prot[0], *prot, "--moltype", "protein", "--threshold", "0.0", "-o", "prot_search_b200.csv"],
                 ["gather", prot[0], *prot, "--protein", "--threshold-bp", "0", "-o", "prot_gather_ref.csv"],
                 ["scripts", "b200gather", prot[0], *prot, "--moltype", "protein", "--threshold-bp", "0", "-o", "prot_gather_b200.csv"])
    _same_file(cli, "prot_search_ref.csv", "prot_search_b200.csv", 1)
    _same_file(cli, "prot_gather_ref.csv", "prot_gather_b200.csv", 0)


def test_confidence_interval_columns(cli):
    "--estimate-ani-ci: the four (gather, prefetch) / two (containment search) extra columns"
    query = os.path.join(DATA, "gather", "combined.sig")
    sigs = sorted(cli.glob(os.path.join(DATA, "gather", "GCF*.sig")))
    pairs = []
    for cmd, first, flags in (("gather", query, ["--threshold-bp", "0"]), ("prefetch", query, ["--threshold-bp", "0"]),
                              ("search", sigs[0], ["--threshold", "0.01", "--containment"])):
        pairs += [[cmd, first, *sigs, "-k", "21", "--estimate-ani-ci", "-o", "ci_%s_ref.csv" % cmd, *flags],
                  ["scripts", "b200" + cmd, first, *sigs, "-k", "21", "--estimate-ani-ci", "-o", "ci_%s_b200.csv" % cmd, *flags]]
    cli.together(*pairs)
    for cmd in ("gather", "prefetch", "search"):
        _same_file(cli, "ci_%s_ref.csv" % cmd, "ci_%s_b200.csv" % cmd, 5)
        assert "ani_low" in open(os.path.join(cli.work, "ci_%s_ref.csv" % cmd)).readline()
