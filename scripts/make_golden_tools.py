#!/usr/bin/env python
"""Regenerate tests/golden/golden_tools.json and tests/golden/disk_parts/ from the UNMODIFIED reference (oracle/_ref/jellyfish):
what its own tools answer where the tests compare the project's with them (test_host.py: readers, merge; test_gpu_parity.py:
the 1 Mbp count, the corner cases where the reference loses k-mers).  The inputs the tests feed the reference's tools are
written by the C restatement (oracle/_ref/jf_oracle) at test time; this script checks that the restatement writes the same
databases as the reference and records their md5s, which the tests check in turn.
    python scripts/make_golden_tools.py
"""
import json
import os
import shutil
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)
import gen      # noqa: E402
import jfutil   # noqa: E402
from cases import DISK_PARTS_COUNT, EDGE_CASES, MERGE_COUNTS, MERGE_OPS, READER_COMMANDS  # noqa: E402
from jellyfish_b200.engine import write_header  # noqa: E402

os.environ["SOURCE_DATE_EPOCH"] = "0"
GOLDEN = os.path.join(ROOT, "tests", "golden")
db_digest = jfutil.db_digest


def ref(*args):
    return jfutil.run([jfutil.REF_JF] + list(args)).stdout.decode()


out = {}
with tempfile.TemporaryDirectory() as d:
    files = gen.make_all(d)

    # test_against_reference_binary_1m: the reference's count, and what its stats / histo print of it
    db = os.path.join(d, "ref_1m.jf")
    jfutil.run([jfutil.REF_JF, "count", "-m", "21", "-s", "2M", "-t", "4", "-C", "-o", db, files["plain1m.fa"]])
    out["count_1m"] = dict(db_digest(db), header_keys=sorted(jfutil.split_db(db)[0]), stats=ref("stats", db), histo=ref("histo", db))

    # test_cli_readers_match_reference_tools: the reference's readers on the restatement's database
    db = os.path.join(d, "readers.jf")
    jfutil.run([jfutil.ORACLE_C, "count", "-m", "17", "-s", "1M", "-C", "-o", db, files["multi.fa"], files["repeat.fa"]])
    out["readers"] = {"db_body_md5": jfutil.md5(jfutil.split_db(db)[1]),
                      "stdout_md5": {" ".join(cmd): jfutil.md5(jfutil.run([jfutil.REF_JF] + cmd + [db]).stdout) for cmd in READER_COMMANDS}}

    # test_merge_matches_reference: its inputs (reference = restatement), every merge the test runs, the --disk parts
    dbs, counts = {}, {}
    for name, args, ins in MERGE_COUNTS:
        dbs[name] = os.path.join(d, "m_%s.jf" % name)
        jfutil.run([jfutil.REF_JF, "count"] + args + ["-o", dbs[name]] + [files[i] for i in ins])
        alt = dbs[name] + ".oracle"
        jfutil.run([jfutil.ORACLE_C, "count"] + args + ["-o", alt] + [files[i] for i in ins])
        counts[name] = db_digest(dbs[name])
        assert db_digest(alt) == counts[name], name
    merges = {}
    for tag, switches, names in MERGE_OPS:
        r = os.path.join(d, "m_ref_%s" % tag)
        jfutil.run([jfutil.REF_JF, "merge"] + switches + ["-o", r] + [dbs[n] for n in names])
        merges[tag] = {"text": open(r).read()} if "--jaccard" in switches else db_digest(r)
    # the intermediate files of a --disk run: stored as the reference wrote them, the path of its binary blanked in the header
    parts_dir = os.path.join(GOLDEN, "disk_parts")
    shutil.rmtree(parts_dir, ignore_errors=True)
    os.makedirs(parts_dir)
    cwd = os.getcwd()
    os.chdir(d)
    args, inp = DISK_PARTS_COUNT
    jfutil.run([jfutil.REF_JF, "count"] + args + ["-o", "m_part", inp])
    os.chdir(cwd)
    parts = []
    for i in range(64):
        p = os.path.join(d, "m_part%d" % i)
        if os.path.exists(p):
            h, b = jfutil.split_db(p)
            h["exe_path"] = "jellyfish"
            parts.append(os.path.join(parts_dir, "m_part%d" % i))
            with open(parts[-1], "wb") as f:
                write_header(f, h)
                f.write(b)
    assert len(parts) >= 3
    r = os.path.join(d, "m_ref_disk")
    jfutil.run([jfutil.REF_JF, "merge", "-o", r] + parts)
    merges["disk"] = db_digest(r)
    out["merge"] = {"counts": counts, "merges": merges}

    # test_cli_count_corner_cases_against_reference_golden: the reference's records on the tiny tables, as a digest and the
    # records that differ from the exact counts (the restatement on a roomy table)
    out["edge_losses"] = {}
    for name in sorted(EDGE_CASES):
        args, ins = EDGE_CASES[name]
        tiny = os.path.join(d, "tiny_%s.jf" % name)
        jfutil.run([jfutil.REF_JF, "count"] + list(args) + ["-o", tiny] + [files[i] for i in ins])
        roomy = list(args)
        roomy[roomy.index("-s") + 1] = "4M"
        for sw in ("-p", "-c"):
            if sw in roomy:
                i = roomy.index(sw)
                del roomy[i:i + 2]
        exact = os.path.join(d, "roomy_%s.jf" % name)
        jfutil.run([jfutil.ORACLE_C, "count"] + roomy + ["-o", exact] + [files[i] for i in ins])
        rt = dict(jfutil.records(*jfutil.split_db(tiny)))
        true = dict(jfutil.records(*jfutil.split_db(exact)))
        assert set(rt) <= set(true)
        differs = sorted([k, rt.get(k)] for k in true if rt.get(k) != true[k])
        out["edge_losses"][name] = {"records_md5": jfutil.records_md5(rt.items()), "differs": differs}
        print(name, len(true) - len(rt), sum(1 for k in rt if rt[k] < true[k]))

with open(os.path.join(GOLDEN, "golden_tools.json"), "w") as f:
    json.dump(out, f, indent=1, sort_keys=True)
    f.write("\n")
