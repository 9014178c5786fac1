#!/usr/bin/env python
"""Differential fuzz of the C restatement (oracle/_ref/jf_oracle) against the UNMODIFIED reference
(oracle/_ref/jellyfish): random switches and small random inputs, header keys and record bodies
compared byte for byte; failures print the command line so that the case can be added to tests/cases.py.
    python scripts/fuzz_oracle.py [N] [SEED] [--record FILE | --replay FILE]
Without a switch the reference binary is asked directly.  --record also keeps its answers (exit status, header digest, body
md5) in FILE; --replay takes them from FILE instead of the binary, so the comparison runs where the reference does not.
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
n_iter = int(argv[0]) if len(argv) > 0 else 100
rng = random.Random(int(argv[1]) if len(argv) > 1 else 1)
ref = jfutil.RefLog(golden, mode)


def rand_seq(n, alphabet="ACGT"):
    return "".join(rng.choice(alphabet) for _ in range(n))


def rand_fasta(path):
    out = []
    for _ in range(rng.randrange(1, 6)):
        n = rng.choice([0, 1, 5, 40, 200, 3000, 20000])
        alpha = rng.choice(["ACGT", "ACGT", "ACGTacgt", "ACGTN", "AC", "A", "ACGTRYn-"])
        s = rand_seq(n, alpha)
        if rng.random() < 0.3 and n > 100:      # repeats -> big counts
            s = s[:50] * (n // 50)
        w = rng.choice([1, 7, 60, 70, 100000])
        eol = rng.choice(["\n", "\n", "\r\n"])
        out.append(">h%d x" % rng.randrange(1000) + eol + "".join(s[i:i + w] + eol * rng.choice([1, 1, 1, 2]) for i in range(0, len(s), w)))
    data = "".join(out)
    if rng.random() < 0.3:
        data = data.rstrip("\r\n")
    open(path, "w", newline="").write(data)


def rand_fastq(path):
    out = []
    wrap = rng.choice([0, 0, 0, 50])        # multi-line records now and then
    for i in range(rng.randrange(1, 40)):
        n = rng.choice([1, 30, 76, 150, 400])
        s = rand_seq(n, rng.choice(["ACGT", "ACGTN", "ACGTacgt"]))
        q = "".join(chr(rng.randrange(33, 75)) if rng.random() < 0.1 else rng.choice("FGHIJ") for _ in range(n))
        if wrap:
            s = "\n".join(s[j:j + wrap] for j in range(0, n, wrap))
            q = "\n".join(q[j:j + wrap] for j in range(0, n, wrap))
        out.append("@r%d\n%s\n+%s\n%s\n" % (i, s, rng.choice(["", "r%d" % i]), q))
    open(path, "w").write("".join(out))


def db_answer(rc, path):
    """What the comparison needs of a count run: success, and the header digest and body of the database."""
    if rc != 0:
        return {"ok": False}
    h, b = jfutil.split_db(path)
    return {"ok": True, "header": jfutil.semantic_md5(h), "md5": jfutil.md5(b), "len": len(b)}


def run_ref(cmd, out):
    return db_answer(subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE).returncode, out)


bad = 0
with tempfile.TemporaryDirectory() as d:
    def rel(args):
        return " ".join(os.path.relpath(a, d) if a.startswith(d) else a for a in args)

    for it in range(n_iter):
        files = []
        kinds = sorted(rng.random() < 0.3 for _ in range(rng.randrange(1, 4)))   # FASTA files first (see -Q note in tests/cases.py)
        for j, fq in enumerate(kinds):
            p = os.path.join(d, "in%d_%d" % (it, j))
            (rand_fastq if fq else rand_fasta)(p)
            files.append(p)
        k = rng.choice([1, 2, 3, 4, 5, 8, 11, 12, 15, 16, 17, 21, 25, 31, 32, 33, 40, 48, 63, 64, rng.randrange(1, 65)])
        size = rng.choice(["1", "2", "10", "100", "1k", "5k", "64k", "100k", "1M", str(rng.randrange(1, 300000))])
        args = ["-m", str(k), "-s", size]
        if rng.random() < 0.6:
            args.append("-C")
        if rng.random() < 0.3:
            args += ["-c", str(rng.choice([1, 2, 3, 5, 7, 10, 16]))]
        if rng.random() < 0.3:
            args += ["-p", str(rng.choice([1, 2, 5, 10, 30, 62, 126, 200]))]
        if rng.random() < 0.2:
            args += ["--out-counter-len", str(rng.choice([1, 2, 3, 7]))]
        if rng.random() < 0.2:
            args += ["-L", str(rng.choice([1, 2, 5]))]
        if rng.random() < 0.15:
            args += ["-U", str(rng.choice([1, 3, 100]))]
        if rng.random() < 0.1:
            args.append("--text")
        if rng.random() < 0.15:
            args += ["--if", rng.choice(files)]
        if rng.random() < 0.15:
            args += rng.choice([["-Q", rng.choice("#5AF")], ["--min-quality", str(rng.randrange(0, 9)), "--quality-start", "33"]])
        u = rng.random()
        if u < 0.1:
            args += ["--bf-size", rng.choice(["100", "5k", "100k"]), "--bf-fp", rng.choice(["0.01", "0.2", "0.001"])]
        elif u < 0.2:
            bc = os.path.join(d, "f.bc")
            bargs = ["-m", str(k), "-s", rng.choice(["100", "5k", "100k"]), "-f", rng.choice(["0.001", "0.05", "0.3"])] + (["-C"] if "-C" in args else [])
            r1 = ref.answer("bc " + rel(bargs + files[:2]), lambda: run_ref([jfutil.REF_JF, "bc", "-t", "2"] + bargs + ["-o", bc] + files[:2], bc))
            r2 = subprocess.run([jfutil.ORACLE_C, "bc"] + bargs + ["-o", bc + ".o"] + files[:2], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
            if r1["ok"] and r2.returncode == 0:
                if r1["md5"] != jfutil.md5(jfutil.split_db(bc + ".o")[1]):
                    bad += 1
                    print("MISMATCH #%d: bc files differ: bc %s %s" % (it, " ".join(bargs), " ".join(files[:2])))
                if mode == "replay":          # the restatement's file stands in for the reference's: the same counters
                    os.replace(bc + ".o", bc)
                args += ["--bc", bc]
        r_db, o_db = os.path.join(d, "r.jf"), os.path.join(d, "o.jf")
        for f in (r_db, o_db):
            if os.path.exists(f):
                os.remove(f)
        rr = ref.answer("count " + rel(args + files), lambda: run_ref([jfutil.REF_JF, "count", "-t", "1"] + args + ["-o", r_db] + files, r_db))
        ro = subprocess.run([jfutil.ORACLE_C, "count"] + args + ["-o", o_db] + files, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        ok = True
        why = ""
        if rr["ok"] != (ro.returncode == 0):
            ok, why = False, "exit status: ref %s, oracle %d: %s" % ("ok" if rr["ok"] else "failed", ro.returncode, ro.stderr[-200:])
        elif rr["ok"]:
            h2, b2 = jfutil.split_db(o_db)
            if rr["header"] != jfutil.semantic_md5(h2):
                ok, why = False, "semantic header keys differ"
            elif rr["md5"] != jfutil.md5(b2):
                ok, why = False, "bodies differ (%d vs %d bytes)" % (rr["len"], len(b2))
        if not ok:
            bad += 1
            keep = os.path.join("/tmp", "fuzz_fail_%d" % it)
            os.makedirs(keep, exist_ok=True)
            kept = []
            for f in files:
                subprocess.run(["cp", f, keep])
                kept.append(os.path.join(keep, os.path.basename(f)))
            print("MISMATCH #%d: %s\n   count %s %s" % (it, why, " ".join(args), " ".join(kept)))
ref.close()
print("%d iterations, %d mismatches" % (n_iter, bad))
sys.exit(1 if bad else 0)
