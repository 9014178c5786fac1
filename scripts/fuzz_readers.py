#!/usr/bin/env python
"""Differential fuzz of the host-side readers of jellyfish-b200 (dump, histo, stats, query, merge: plain
CPU code in jellyfish_b200/csrc/host/jf_cli.cc) against the reference's own tools, on random databases
written by the reference's `count`.
    python scripts/fuzz_readers.py [N] [SEED] [--record FILE | --replay FILE]
Without a switch the reference binary is asked directly.  --record also keeps its answers (exit status and md5 of what it
wrote) in FILE; --replay takes them from FILE instead of the binary, and the databases the readers chew on are written by the
C restatement (oracle/_ref/jf_oracle), held to the reference's md5s, so the comparison runs where the reference does not.
"""
import os
import random
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import jfutil  # noqa: E402

argv = sys.argv[1:]
mode, golden = "live", None
for sw in ("--record", "--replay"):
    if sw in argv:
        i = argv.index(sw)
        mode, golden = sw[2:], argv[i + 1]
        del argv[i:i + 2]
n_iter = int(argv[0]) if len(argv) > 0 else 50
rng = random.Random(int(argv[1]) if len(argv) > 1 else 1)
ref = jfutil.RefLog(golden, mode)


def rand_fasta(path, total):
    out = []
    for r in range(rng.randrange(1, 5)):
        n = rng.choice([50, 500, total])
        s = "".join(rng.choice("ACGT") for _ in range(n))
        if rng.random() < 0.4:
            s = s[:40] * (n // 40 + 1)
        out.append(">r%d\n%s\n" % (r, s))
    open(path, "w").write("".join(out))


def rel(args):
    return " ".join(os.path.relpath(a, d) if a.startswith(d) else a for a in args)


def db_answer(rc, path):
    if rc != 0:
        return {"rc": rc}
    h, b = jfutil.split_db(path)
    return {"rc": rc, "header": jfutil.semantic_md5(h), "md5": jfutil.md5(b)}


def both(args):
    """-> (the reference's exit status and md5 of its standard output, ours)"""
    a = ref.answer(rel(args), lambda: (lambda r: {"rc": r.returncode, "md5": jfutil.md5(r.stdout)})(
        subprocess.run([jfutil.REF_JF] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE)))
    b = subprocess.run([jfutil.OUR_JF] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    return a, {"rc": b.returncode, "md5": jfutil.md5(b.stdout)}


def ref_count(args, db, fa):
    """A database written by the reference's count (replayed: by the restatement, which must write the same one)."""
    want = ref.answer(rel(["count"] + args + [fa]), lambda: db_answer(subprocess.run(
        [jfutil.REF_JF, "count", "-t", "2"] + args + ["-o", db, fa], check=True).returncode, db))
    if mode == "replay":
        subprocess.run([jfutil.ORACLE_C, "count"] + args + ["-o", db, fa], check=True, stderr=subprocess.PIPE)
        if db_answer(0, db) != want:
            report(it, "restatement's database differs from the reference's", args + [fa])


def ref_merge(args, out):
    """-> the reference's merge: exit status, header digest and md5 of the body (or of the Jaccard text)"""
    def ask():
        r = subprocess.run([jfutil.REF_JF, "merge", "-o", out] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        if r.returncode == 0 and "-j" in args:
            return {"rc": 0, "md5": jfutil.md5(open(out, "rb").read())}
        return db_answer(r.returncode, out)
    return ref.answer(rel(["merge"] + args), ask)


bad = 0


def report(it, what, args):
    global bad
    bad += 1
    print("MISMATCH #%d %s: %s" % (it, what, " ".join(args)))


with tempfile.TemporaryDirectory() as d:
    for it in range(n_iter):
        k = rng.choice([1, 3, 4, 8, 12, 16, 17, 21, 31, 32, 33, 47, 63, 64])
        size = rng.choice(["1k", "20k", "300k"])
        cargs = ["-m", str(k), "-s", size] + (["-C"] if rng.random() < 0.6 else []) + \
                (["--out-counter-len", str(rng.choice([1, 2, 3, 5]))] if rng.random() < 0.4 else [])
        fas, dbs = [], []
        for j in range(2):
            fa = os.path.join(d, "f%d_%d.fa" % (it, j))
            rand_fasta(fa, rng.choice([2000, 30000]))
            db = os.path.join(d, "db%d_%d.jf" % (it, j))
            ref_count(cargs, db, fa)
            fas.append(fa)
            dbs.append(db)
        db = dbs[0]
        # dump
        for _ in range(3):
            a = ["dump"] + rng.sample(["-c", "-t"], rng.randrange(0, 3)) + \
                (["-L", str(rng.choice([1, 2, 5, 300]))] if rng.random() < 0.4 else []) + \
                (["-U", str(rng.choice([1, 3, 50, 100000]))] if rng.random() < 0.4 else []) + [db]
            x, y = both(a)
            if x != y:
                report(it, "dump", a)
        # histo
        for _ in range(3):
            a = ["histo"] + (["-l", str(rng.choice([0, 1, 2, 10]))] if rng.random() < 0.5 else []) + \
                (["-h", str(rng.choice([1, 5, 100, 100000]))] if rng.random() < 0.5 else []) + \
                (["-i", str(rng.choice([1, 2, 7]))] if rng.random() < 0.4 else []) + (["-f"] if rng.random() < 0.3 else []) + [db]
            x, y = both(a)
            if x != y:
                report(it, "histo", a)
        # stats
        for _ in range(2):
            a = ["stats"] + (["-L", str(rng.choice([1, 2, 5]))] if rng.random() < 0.4 else []) + \
                (["-U", str(rng.choice([1, 3, 1000]))] if rng.random() < 0.4 else []) + [db]
            x, y = both(a)
            if x != y:
                report(it, "stats", a)
        # query: k-mers of the input, random k-mers, lower case, one with an N (both must treat it alike)
        seq = "".join(l.strip() for l in open(fas[0]) if not l.startswith(">"))
        mers = [seq[p:p + k] for p in (rng.randrange(0, max(1, len(seq) - k)) for _ in range(5)) if len(seq) >= k]
        mers += ["".join(rng.choice("ACGT") for _ in range(k)) for _ in range(3)]
        mers += [m.lower() for m in mers[:2]]
        a = ["query", db] + mers
        x, y = both(a)
        if x != y:
            report(it, "query", a)
        a = ["query", "-s", fas[1], db]
        x, y = both(a)
        if x != y:
            report(it, "query -s", a)
        # merge (same -m/-s => same matrix)
        ma, mb = os.path.join(d, "ma.jf"), os.path.join(d, "mb.jf")
        extra = (["-L", str(rng.choice([0, 1, 2, 3]))] if rng.random() < 0.3 else []) + (["-U", str(rng.choice([2, 100]))] if rng.random() < 0.3 else [])
        extra += rng.choice([[], [], ["-m"], ["--max"]])
        x = ref_merge(extra + dbs, ma)
        y = subprocess.run([jfutil.OUR_JF, "merge", "-o", mb] + extra + dbs, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        if x["rc"] != y.returncode:
            report(it, "merge exit %d/%d %s" % (x["rc"], y.returncode, y.stderr[-100:]), extra + dbs)
        elif x != db_answer(y.returncode, mb):
            report(it, "merge output", extra + dbs)
        # jaccard (two text lines instead of a database), three inputs
        ja, jb = os.path.join(d, "ja.txt"), os.path.join(d, "jb.txt")
        three = dbs + [dbs[0]] if rng.random() < 0.5 else dbs
        x = ref_merge(["-j"] + three, ja)
        y = subprocess.run([jfutil.OUR_JF, "merge", "-j", "-o", jb] + three, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        if x["rc"] != y.returncode or (y.returncode == 0 and x["md5"] != jfutil.md5(open(jb, "rb").read())):
            report(it, "merge --jaccard", three)
        # text/sorted databases of the same inputs, merged as text
        tdbs = []
        for j in range(2):
            t = os.path.join(d, "t%d_%d.jf" % (it, j))
            ref_count([c for c in cargs if c not in ("--out-counter-len",)][:4 + ("-C" in cargs)] + ["--text"], t, fas[j])
            tdbs.append(t)
        x = ref_merge(extra + tdbs, ma)
        y = subprocess.run([jfutil.OUR_JF, "merge", "-o", mb] + extra + tdbs, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        if x["rc"] != y.returncode:
            report(it, "text merge exit %d/%d %s" % (x["rc"], y.returncode, y.stderr[-100:]), extra + tdbs)
        elif x != db_answer(y.returncode, mb):
            report(it, "text merge output", extra + tdbs)
        if bad:
            keep = "/tmp/fuzz_readers_fail"
            os.makedirs(keep, exist_ok=True)
            for f in fas + dbs:
                subprocess.run(["cp", f, keep])
            print("   count", " ".join(cargs), "(files kept in %s)" % keep)
            break
if not bad:
    ref.close()
print("%d iterations, %d mismatches" % (it + 1, bad))
sys.exit(1 if bad else 0)
