"""Randomised differential test: the reference's Python (its per-pair loops over this library's ABI) against this package's
batched functions, on the same seeded random signature lists.

The reference's results for a seed and a trial count are stored in golden/differential_seed<seed>_trials<n>.json.gz and
only this package runs (bound to the emulated library, so no GPU is needed).  With SOURMASH_CHECKOUT naming a sourmash
checkout, both packages run side by side in one process (`sourmash` = the reference loaded in place over the emulated
library, as in test_reference_python_over_abi.py) and the file is written anew from the reference's results.  For every random
list -- equal or mixed scaled, flat and abundance sketches, empty sketches, num sketches -- the matrices of
compare_all_pairs / compare_serial_containment / _max_containment / _avg_containment (with and without ANI) must be equal
bit for bit, and LinearIndex.search / search_abund / prefetch and a gather loop must return the same matches with the same
scores.  Then random FASTA files are sketched both ways (every molecule type), and random query / database sets go through
the reference's `gather`, `prefetch` and `search` commands and the plugin's: the CSV files must be byte-identical (query at a
finer, equal or coarser scaled than the databases; abundance queries with and without --ignore-abundance; thresholds)."""
import os
import subprocess
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_reference_python_over_abi as over_abi  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CHECKOUT = os.environ.get("SOURMASH_CHECKOUT")

TRIALS = r'''
import gzip
import hashlib
import json
import sys
import warnings
import numpy as np
import sourmash_b200 as smb
import sourmash_b200.compare as our_compare
import sourmash_b200.index as our_index

seed, n_trials, store = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3]
RECORD = sys.argv[4] == "record"                # run the reference and write its results to `store`; else read them
if RECORD:
    import sourmash as ref
    import sourmash.compare as ref_compare
    import sourmash.index as ref_index
    STORED = []
else:
    with gzip.open(store, "rt") as fh:
        STORED = json.load(fh)
    STORED.reverse()
rng = np.random.default_rng(seed)
stats = {"compare": 0, "containment": 0, "ani": 0, "search": 0, "prefetch": 0, "gather": 0, "errors": 0}   # comparisons made


def make(pkg, spec):
    mh = pkg.MinHash(n=spec["num"], ksize=spec["ksize"], scaled=spec["scaled"], track_abundance=spec["abund"])
    if spec["abund"]:
        mh.set_abundances(dict(zip(spec["hashes"], spec["abunds"])))
    else:
        mh.add_many(spec["hashes"])
    return pkg.SourmashSignature(mh, name=spec["name"], filename=spec["name"] + ".fa").to_frozen()   # what loading a file gives


def random_list(rng):
    n = int(rng.integers(2, 8))
    kind = rng.choice(["scaled", "scaled", "mixed_scaled", "num", "abund"])
    pool = rng.integers(1, 2**64 - 1, size=int(rng.integers(20, 400)), dtype=np.uint64)
    specs = []
    for i in range(n):
        scaled, num = 1000, 0
        if kind == "mixed_scaled":
            scaled = int(rng.choice([500, 1000, 2000]))
        if kind == "num":
            scaled, num = 0, 50
        hashes = rng.choice(pool, size=int(rng.integers(0, len(pool))), replace=False)
        if scaled:
            hashes = hashes[hashes <= np.uint64((2**64 - 1) // scaled)] if rng.random() < 0.5 else hashes % np.uint64((2**64) // scaled)
        hashes = np.unique(hashes)
        if rng.random() < 0.08:
            hashes = hashes[:0]                                     # an empty sketch
        abund = kind == "abund" and rng.random() < 0.8
        specs.append(dict(num=num, ksize=21, scaled=scaled, abund=bool(abund), name="s%d" % i,
                          hashes=[int(h) for h in hashes], abunds=[int(a) for a in rng.integers(1, 30, size=len(hashes))]))
    return kind, specs


def plain(x):
    "a value as JSON would give it back: arrays as {shape, values}, tuples as lists, float64 scalars as floats"
    if isinstance(x, np.ndarray):
        return {"shape": list(x.shape), "values": [plain(v) for v in x.ravel().tolist()]}
    if isinstance(x, (list, tuple)):
        return [plain(v) for v in x]
    if isinstance(x, np.generic):
        return x.item()
    return x


def outcome(fn):
    "['ok', value] or ['raises', exception type name, message], in plain form"
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            return plain(("ok", fn()))
        except Exception as exc:                                    # noqa: BLE001 -- the comparison IS about what is raised
            return ["raises", type(exc).__name__, str(exc)]


def digest(value):
    "a stored result: the value, or -- above 2 kB of JSON -- its sha256 and its first 300 characters"
    text = json.dumps(value)
    if len(text) <= 2000:
        return value
    return {"sha256": hashlib.sha256(text.encode()).hexdigest(), "head": text[:300]}


def expected(fn, whole=False):
    "the reference's result (digest form unless `whole`): computed with `fn` (recording) or the next one stored"
    if RECORD:
        STORED.append(fn() if whole else digest(fn()))
        return STORED[-1]
    return STORED.pop()


def differs(want, got):
    "whether this package's plain result `got` differs from the reference's stored `want`: bit for bit, NaN == NaN"
    return json.dumps(digest(got)) != json.dumps(want)


def same(a, b, what, specs):
    if isinstance(a, dict):                                         # a large result, stored as its digest
        if differs(a, b):
            raise AssertionError("%s differs\nreference %s...\nhere      %s...\n%r" % (what, a["head"], json.dumps(b)[:300], specs))
        return
    if a[0] != b[0]:
        raise AssertionError("%s: reference %r, here %r\n%r" % (what, a[:3], b[:3], specs))
    if a[0] == "raises":
        if a[1] != b[1]:
            raise AssertionError("%s raises %s(%s) in the reference, %s(%s) here" % (what, a[1], a[2], b[1], b[2]))
        stats["errors"] += 1
        return
    if differs(a[1], b[1]):                                         # floats bit for bit (repr round-trips), NaN == NaN
        raise AssertionError("%s differs\nreference %r\nhere      %r\n%r" % (what, a[1], b[1], specs))


for trial in range(n_trials):
    kind, specs = random_list(rng)
    R, O = [make(ref, s) for s in specs] if RECORD else None, [make(smb, s) for s in specs]
    down = kind == "mixed_scaled"
    for ignore in (True, False):
        same(expected(lambda: outcome(lambda: ref_compare.compare_all_pairs(R, ignore, downsample=down, n_jobs=None))),
             outcome(lambda: our_compare.compare_all_pairs(O, ignore, downsample=down, n_jobs=None)),
             "compare_all_pairs(ignore_abundance=%s) on %s" % (ignore, kind), specs)
        stats["compare"] += 1
    for name in ("compare_serial_containment", "compare_serial_max_containment", "compare_serial_avg_containment"):
        same(expected(lambda: outcome(lambda: getattr(ref_compare, name)(R, downsample=down))),
             outcome(lambda: getattr(our_compare, name)(O, downsample=down)), "%s on %s" % (name, kind), specs)
        stats["containment"] += 1
        if kind in ("scaled", "mixed_scaled"):
            same(expected(lambda: outcome(lambda: getattr(ref_compare, name)(R, downsample=down, return_ani=True))),
                 outcome(lambda: getattr(our_compare, name)(O, downsample=down, return_ani=True)),
                 "%s(return_ani) on %s" % (name, kind), specs)
            stats["ani"] += 1
    if kind == "mixed_scaled":             # without the flag the avg ANI form downsamples anyway (FracMinHashComparison)
        for name in ("compare_serial_avg_containment",):
            same(expected(lambda: outcome(lambda: getattr(ref_compare, name)(R, return_ani=True))),
                 outcome(lambda: getattr(our_compare, name)(O, return_ani=True)), "%s(return_ani, no downsample) on %s" % (name, kind), specs)
            stats["ani"] += 1
    if kind in ("scaled", "mixed_scaled"):
        same(expected(lambda: outcome(lambda: ref_compare.compare_all_pairs(R, True, downsample=down, return_ani=True, n_jobs=None))),
             outcome(lambda: our_compare.compare_all_pairs(O, True, downsample=down, return_ani=True, n_jobs=None)),
             "compare_all_pairs(return_ani) on %s" % kind, specs)
        stats["ani"] += 1
    # one-vs-many: the first signature against an index of the rest
    if kind in ("scaled", "mixed_scaled") and len(specs[0]["hashes"]):
        ri, oi = ref_index.LinearIndex(R[1:], "db") if RECORD else None, our_index.LinearIndex(O[1:], "db")

        def names(results):
            return [(float(r.score), r.signature.name, r.location) for r in results]
        for kw in (dict(threshold=0.0), dict(threshold=0.05, do_containment=True), dict(threshold=0.05, do_max_containment=True),
                   dict(threshold=0.0, best_only=True)):
            same(expected(lambda: outcome(lambda: names(ri.search(R[0], **kw)))), outcome(lambda: names(oi.search(O[0], **kw))),
                 "LinearIndex.search(%r) on %s" % (kw, kind), specs)
            stats["search"] += 1
        same(expected(lambda: outcome(lambda: names(ri.prefetch(R[0], threshold_bp=0)))), outcome(lambda: names(oi.prefetch(O[0], threshold_bp=0))),
             "LinearIndex.prefetch on %s" % kind, specs)
        stats["prefetch"] += 1

        def best(index, query, tbp):
            r = index.best_containment(query, threshold_bp=tbp)
            return None if not r else (float(r.score), r.signature.name, r.location)
        for tbp in (0, 5000):
            same(expected(lambda: outcome(lambda: best(ri, R[0], tbp))), outcome(lambda: best(oi, O[0], tbp)),
                 "LinearIndex.best_containment(threshold_bp=%d) on %s" % (tbp, kind), specs)
            stats["search"] += 1

        def gather_rounds(index, query):
            counter = index.counter_gather(query, 0)
            cur, out = query.minhash.flatten().to_mutable(), []
            while True:
                res = counter.peek(cur)
                if not res:
                    return out
                sr, intersect = res
                out.append((float(sr.score), sr.signature.name, len(intersect)))
                counter.consume(intersect)
                cur = cur.downsample(scaled=counter.scaled).to_mutable() if counter.scaled > cur.scaled else cur
                cur.remove_many(intersect.downsample(scaled=cur.scaled) if intersect.scaled < cur.scaled else intersect)
        same(expected(lambda: outcome(lambda: gather_rounds(ri, R[0]))), outcome(lambda: gather_rounds(oi, O[0])), "gather rounds on %s" % kind, specs)
        stats["gather"] += 1
    if kind == "abund":
        ri, oi = ref_index.LinearIndex(R[1:], "db") if RECORD else None, our_index.LinearIndex(O[1:], "db")
        same(expected(lambda: outcome(lambda: [(float(r.score), r.signature.name) for r in ri.search_abund(R[0], threshold=0.0)])),
             outcome(lambda: [(float(r.score), r.signature.name) for r in oi.search_abund(O[0], threshold=0.0)]),
             "LinearIndex.search_abund", specs)
        stats["search"] += 1
# ---- sketching: the reference's record-by-record add_sequence / add_protein against this package's batched file sketcher
import gzip
from sourmash_b200.sketch import sketch_fasta_files
stats["sketch"] = 0
for trial in range(max(4, n_trials // 5)):
    mode = rng.choice(["dna", "dna", "dna_abund_num", "protein", "dayhoff", "hp", "translate"])
    n_files = int(rng.integers(1, 4))
    paths, records = [], []
    for f in range(n_files):
        recs = []
        for r in range(int(rng.integers(0, 5))):
            L = int(rng.choice([0, 5, 20, 21, 60, 300, 2500]))
            if mode in ("protein", "dayhoff", "hp"):
                seq = "".join(rng.choice(list("ACDEFGHIKLMNPQRSTVWYX*"), size=L))
            else:
                seq = "".join(rng.choice(list("ACGT"), size=L))
                if L and rng.random() < 0.5:                       # invalid bases, lower case
                    pos = rng.integers(0, L, size=max(1, L // 40))
                    seq = "".join(("N" if i in set(pos.tolist()) else c) for i, c in enumerate(seq))
                if rng.random() < 0.3:
                    seq = seq.lower()
            recs.append(("f%dr%d some description" % (f, r), seq))
        path = "sk%d_%d.fa%s" % (trial, f, ".gz" if rng.random() < 0.3 else "")
        text = "".join(">%s\n%s\n" % (n, "\n".join(sq[i:i + 70] for i in range(0, len(sq), 70))) for n, sq in recs)
        (gzip.open if path.endswith(".gz") else open)(path, "wt").write(text)
        paths.append(path); records.append(recs)
    if mode in ("dna", "dna_abund_num"):
        ksizes, kw = [21, 31, 51], dict(is_protein=False)
    else:
        ksizes, kw = [7, 10], dict(is_protein=mode in ("protein", "translate"), dayhoff=mode == "dayhoff", hp=mode == "hp")
    scaled, num, abund = (0, 30, True) if mode == "dna_abund_num" else (int(rng.choice([1, 10, 100])), 0, bool(rng.random() < 0.3))
    ours = sketch_fasta_files(paths, ksizes=ksizes, scaled=scaled, num=num, track_abundance=abund,
                              moltype={"dna": "dna", "dna_abund_num": "dna", "translate": "protein"}.get(mode, mode),
                              input_is_protein=mode in ("protein", "dayhoff", "hp"))
    got = plain(sorted((ss.filename, mh.ksize, sorted(mh.hashes.items())) for ss in ours for mh in ss.sketches()))   # one per file

    def reference_sketches():
        want = []
        for path, recs in zip(paths, records):
            if not recs:
                continue                                            # no sequences found: no signature
            for k in ksizes:
                mh = ref.MinHash(n=num, ksize=k, scaled=scaled, track_abundance=abund, **kw)
                for _name, seq in recs:
                    if mode in ("protein", "dayhoff", "hp"):
                        mh.add_protein(seq)
                    else:
                        mh.add_sequence(seq, force=True)            # translate: is_protein sketch fed DNA = six frames
                want.append((path, k, sorted(mh.hashes.items())))
        return plain(sorted(want))
    want = expected(reference_sketches)
    if differs(want, got):
        raise AssertionError("sketch (%s, scaled=%s num=%s abund=%s) differs for %r\nreference %r\nhere      %r" % (
            mode, scaled, num, abund, records, (want["head"] if isinstance(want, dict) else [(w[0], w[1], len(w[2])) for w in want]), [(g[0], g[1], len(g[2])) for g in got]))
    stats["sketch"] += 1
# ---- reports: the reference's gather / prefetch / search commands against the plugin commands, CSV files byte for byte
import contextlib, io
from sourmash_b200.plugin import main as plugin_main
stats["reports"] = 0


def cli(*args):
    "`sourmash ARGS` (the reference) or, for `scripts b200CMD ARGS`, this package's plugin command: the exit status"
    args = [str(a) for a in args]
    if args[0] == "scripts":
        run = lambda: plugin_main(args[1:])
    else:
        from sourmash.__main__ import main as sourmash_main
        run = lambda: sourmash_main(args)
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        try:
            run()
        except SystemExit as exc:
            return exc.code or 0
        except Exception as exc:                                    # noqa: BLE001
            return type(exc).__name__
    return 0


def read(path):
    try:
        return open(path).read()
    except FileNotFoundError:
        return None


for trial in range(max(3, n_trials // 8)):
    top = (2**64 - 1) // 1000
    pool = np.unique(rng.integers(1, top, size=3000, dtype=np.uint64))
    n_subj = int(rng.integers(2, 9))
    # one scaled per database set, finer / equal / coarser than the query's 1000 (databases of DIFFERENT scaled values are
    # the one case the plugin does not follow: the reference lowers the resolution as coarser matches get picked, DESIGN 8)
    db_scaled = int(rng.choice([500, 1000, 2000]))
    subjects, files = [], []
    for i in range(n_subj):
        own = rng.choice(pool, size=int(rng.integers(30, 600)), replace=False)
        mh = smb.MinHash(n=0, ksize=31, scaled=db_scaled)
        mh.add_many([int(h) for h in own])
        ss = smb.SourmashSignature(mh, name="subject %d" % i, filename="subj%d.fa" % i)
        subjects.append(ss)
        path = "rep%d_s%d.sig" % (trial, i)
        with open(path, "wb") as fp:
            smb.save_signatures_to_json([ss], fp)
        files.append(path)
    qh = {}
    for ss in subjects[: max(1, n_subj - 1)]:                      # the query: parts of most subjects + hashes of its own
        for h in sorted(ss.minhash.hashes)[:: int(rng.integers(1, 4))]:
            qh[h] = int(rng.integers(1, 40))
    for h in rng.integers(1, top, size=int(rng.integers(0, 200)), dtype=np.uint64):
        qh[int(h)] = int(rng.integers(1, 5))
    abund = bool(rng.random() < 0.6)
    qmh = smb.MinHash(n=0, ksize=31, scaled=1000, track_abundance=abund)
    if abund:
        qmh.set_abundances(qh)
    else:
        qmh.add_many(list(qh))
    qpath = "rep%d_query.sig" % trial
    with open(qpath, "wb") as fp:
        smb.save_signatures_to_json([smb.SourmashSignature(qmh, name="the query", filename="query.fa")], fp)
    tbp = int(rng.choice([0, 20000, 100000]))
    runs = [("gather", ["--threshold-bp", tbp] + (["--ignore-abundance"] if abund and rng.random() < 0.4 else [])),
            ("prefetch", ["--threshold-bp", tbp]),
            ("search", ["--threshold", "0.02"] + ([[], ["--containment"], ["--max-containment"]][int(rng.integers(0, 3))])
             + (["--ignore-abundance"] if abund and rng.random() < 0.6 else []))]
    for cmd, flags in runs:
        a, b = "rep%d_%s_ref.csv" % (trial, cmd), "rep%d_%s_b200.csv" % (trial, cmd)
        ra, ta = expected(lambda: [cli(cmd, qpath, *files, "-o", a, *flags), read(a)], whole=True)
        rb = cli("scripts", "b200" + cmd, qpath, *files, "-o", b, *flags)
        tb = read(b)
        if ra == "AssertionError":                                  # an `assert` of the reference's own tripped: nothing to follow
            continue
        if (ra == 0) != (rb == 0) or ta != tb:
            la, lb = (ta or "").splitlines(), (tb or "").splitlines()
            diff = [(x, y) for x, y in zip(la, lb) if x != y][:2] or [("%d lines" % len(la), "%d lines" % len(lb))]
            raise AssertionError("%s %r (abund query: %s, %d subjects, db scaled %d): exit %r / %r\n%s\n%s" % (
                cmd, flags, abund, n_subj, db_scaled, ra, rb, la[:1],
                "\n".join("reference %s\nplugin    %s" % d for d in diff)))
        stats["reports"] += 1
if RECORD:
    with gzip.open(store, "wt") as fh:
        json.dump(STORED, fh)
else:
    assert not STORED, "%d stored results left over" % len(STORED)
print("DIFFERENTIAL OK", stats)
'''


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("seed", [int(x) for x in os.environ.get("SMB_DIFF_SEEDS", "1").split(",")])   # others: record first
def test_batched_functions_equal_the_reference_loops_on_random_lists(tmp_path, seed):
    sys.path.insert(0, os.path.join(HERE, "host_emul"))
    try:
        import emul_lib
    finally:
        sys.path.pop(0)
    tmp = str(tmp_path)
    trials = int(os.environ.get("SMB_DIFF_TRIALS", "40"))
    store = os.path.join(HERE, "golden", "differential_seed%d_trials%d.json.gz" % (seed, trials))
    site = os.path.join(tmp, "site")
    os.makedirs(site)
    paths = [site]
    if CHECKOUT:                                                        # the reference in place over the emulated library
        over_abi.REF = CHECKOUT
        over_abi._stub_package(tmp, emul_lib.build())
        paths.append(os.path.join(tmp, "reftests"))
    with open(os.path.join(site, "sitecustomize.py"), "w") as fh:       # this package binds the emulated library
        fh.write("import sys\nsys.path.insert(0, %r); sys.path.insert(0, %r)\nimport emulated_boot\nemulated_boot.install()\n"
                 % (os.path.join(HERE, "host_emul"), ROOT))
    script = os.path.join(tmp, "trials.py")
    with open(script, "w") as fh:
        fh.write(TRIALS)
    env = dict(os.environ, PYTHONPATH=os.pathsep.join(paths), PYTHONDONTWRITEBYTECODE="1")
    r = subprocess.run([sys.executable, script, str(seed), str(trials), store, "record" if CHECKOUT else "replay"],
                       capture_output=True, text=True, env=env, cwd=tmp, timeout=int(os.environ.get("SMB_DIFF_TIMEOUT", "1500")))
    assert r.returncode == 0 and "DIFFERENTIAL OK" in r.stdout, r.stdout[-3000:] + r.stderr[-6000:]
