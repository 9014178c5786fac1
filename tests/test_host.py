"""CPU tests of the host side: the C-ABI library loads and exports every declared symbol, the
host arithmetic (matrix stream, header format) is right, the CPU readers of the format agree
with the reference's, and the product fails loudly without a GPU (no CPU fallback)."""
import ctypes
import io
import json
import os
import re
import subprocess

import pytest

import jfutil
from cases import CASES, MERGE_COUNTS, MERGE_OPS, READER_COMMANDS

GOLDEN = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))


def test_library_exports_every_declared_symbol(built):
    from jellyfish_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(jfutil.ROOT, "include", "jfgpu.h")).read()
    declared = set(re.findall(r"\b(jfgpu_[a-z_0-9]+)\s*\(", header))
    declared -= {"jfgpu_sink_fn"}
    assert declared == set(_lib.SYMBOLS)
    for name in declared:
        assert getattr(lib, name) is not None
    assert b"sm_100a" in lib.jfgpu_version()


def test_struct_layouts_match_header(built, tmp_path):
    """Every field of every ctypes mirror sits where the C compiler puts the field of the same name in include/jfgpu.h."""
    from jellyfish_b200 import _lib
    structs = {"jfgpu_params": _lib.Params, "jfgpu_stats": _lib.Stats, "jfgpu_table_info": _lib.TableInfo,
               "jfgpu_bloom_info": _lib.BloomInfo, "jfgpu_shard_buffers": _lib.ShardBuffers}
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "jfgpu.h"', "int main(void) {"]
    for cname, st in structs.items():
        lines.append('  printf("%s %%zu\\n", sizeof(%s));' % (cname, cname))
        for f, _ in st._fields_:
            lines.append('  printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (cname, f, cname, f))
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(jfutil.ROOT, "include"), "-o", str(exe), str(src)])
    want = dict(l.split() for l in subprocess.check_output([str(exe)]).decode().splitlines())
    for cname, st in structs.items():
        assert ctypes.sizeof(st) == int(want[cname]), cname
        for f, _ in st._fields_:
            assert getattr(st, f).offset == int(want["%s.%s" % (cname, f)]), (cname, f)


def test_reference_matrix_stream(built):
    import jellyfish_b200 as j
    cols = j.reference_matrix(27, 42)
    assert cols[:3] == [64834949, 57999349, 22595292] and cols[41] == 69326724
    assert j.reference_matrix(21, 42)[:3] == [457302, 1834222, 704443]
    # agrees with the C restatement for other shapes, including later draws of the stream
    for r, c, skip in [(10, 10, 0), (19, 42, 2), (31, 126, 1), (34, 62, 0)]:
        out = subprocess.check_output([jfutil.ORACLE_C, "matrix", str(r), str(c), str(skip)]).split()
        assert j.reference_matrix(r, c, skip) == [int(x) for x in out]


def test_reference_matrix_against_reference_library_golden(built):
    # tests/golden/matrix_golden.json: drawn by the unmodified reference library, shapes with more
    # than 30 rows included (tables of 2^31 slots and more -- BASELINE configs[1] uses 2^32..2^34)
    import json
    import jellyfish_b200 as j
    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "matrix_golden.json")))
    assert any(g["r"] > 30 for g in golden)
    for g in golden:
        assert j.reference_matrix(g["r"], g["c"], g["skip"]) == g["columns"], (g["r"], g["c"], g["skip"])


def test_no_cpu_fallback(built):
    """Without a CUDA device the engine refuses to run (it must never count on the CPU)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import jellyfish_b200 as j
    with pytest.raises(j.JellyfishError) as ei:
        j.HashCounter(1000, 7, k=21)
    assert "no CPU fallback" in str(ei.value)
    r = subprocess.run([jfutil.OUR_JF, "count", "-m", "21", "-s", "1M", "/dev/null"], stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"no CPU fallback" in r.stderr


def test_cli_argument_errors(built):
    r = subprocess.run([jfutil.OUR_JF, "count", "-s", "1M", "x.fa"], stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"--mer-len" in r.stderr
    r = subprocess.run([jfutil.OUR_JF, "count", "-m", "21", "x.fa"], stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"--size" in r.stderr
    r = subprocess.run([jfutil.OUR_JF, "count", "-m", "21", "-s", "1M", "--bc", "a", "--bf-size", "3", "x.fa"], stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"conflict" in r.stderr
    r = subprocess.run([jfutil.OUR_JF, "nonsense"], stderr=subprocess.PIPE)
    assert r.returncode == 1


def test_python_header_writer_round_trip(built, workdir):
    from jellyfish_b200.engine import write_header, ReadMerFile
    hdr = {"alignment": 8, "canonical": True, "cmdline": ["count", "a b"], "counter_len": 4, "format": "binary/sorted",
           "key_len": 42, "matrix1": {"r": 3, "c": 42, "identity": False, "columns": list(range(42))}, "size": 8}
    p = os.path.join(workdir, "hdr.jf")
    with open(p, "wb") as f:
        write_header(f, hdr)
        f.write((5).to_bytes(6, "little") + (9).to_bytes(4, "little"))
    raw = open(p, "rb").read()
    hlen = int(raw[:9])
    assert (9 + hlen) % 8 == 0
    r = ReadMerFile(p)
    assert r.header == hdr
    assert list(r) == [("A" * 19 + "CC", 9)]


@pytest.fixture(scope="module")
def oracle_db(built, workdir, inputs):
    """A database written by the oracle restatement, for the CPU readers to chew on."""
    db = os.path.join(workdir, "readers.jf")
    jfutil.run([jfutil.ORACLE_C, "count", "-m", "17", "-s", "1M", "-C", "-o", db, inputs["multi.fa"], inputs["repeat.fa"]])
    return db


def test_cli_readers_self_consistent(oracle_db, workdir):
    h, body = jfutil.split_db(oracle_db)
    recs = jfutil.records(h, body)
    from jellyfish_b200 import int_to_mer
    col = jfutil.run([jfutil.OUR_JF, "dump", "-c", oracle_db]).stdout.decode().splitlines()
    assert col == ["%s %d" % (int_to_mer(k, 17), c) for k, c in recs]
    fa = jfutil.run([jfutil.OUR_JF, "dump", "-L", "2", oracle_db]).stdout.decode().split()
    assert len(fa) == 2 * sum(1 for _, c in recs if c >= 2)
    st = jfutil.run([jfutil.OUR_JF, "stats", oracle_db]).stdout.decode().split()
    assert int(st[1]) == sum(1 for _, c in recs if c == 1) and int(st[3]) == len(recs)
    assert int(st[5]) == sum(c for _, c in recs) and int(st[7]) == max(c for _, c in recs)
    hist = dict(map(int, line.split()) for line in jfutil.run([jfutil.OUR_JF, "histo", oracle_db]).stdout.decode().splitlines())
    assert hist[1] == sum(1 for _, c in recs if c == 1)
    # query: present, absent, reverse complement of a canonical database
    k0, c0 = recs[len(recs) // 2]
    mer = int_to_mer(k0, 17)
    rc = mer[::-1].translate(str.maketrans("ACGT", "TGCA"))
    out = jfutil.run([jfutil.OUR_JF, "query", oracle_db, mer, rc]).stdout.decode().splitlines()
    assert out == ["%s %d" % (mer, c0)] * 2
    info = jfutil.run([jfutil.OUR_JF, "info", "-j", oracle_db]).stdout
    assert json.loads(info)["key_len"] == 34


def test_cli_readers_match_reference_tools(oracle_db, workdir):
    """Byte for byte what the reference's own dump / histo / stats print of the same database (md5s of their output,
    tests/golden/golden_tools.json, scripts/make_golden_tools.py)."""
    g = jfutil.golden("golden_tools.json")["readers"]
    assert jfutil.md5(jfutil.split_db(oracle_db)[1]) == g["db_body_md5"]
    for cmd in READER_COMMANDS:
        b = jfutil.run([jfutil.OUR_JF] + cmd + [oracle_db]).stdout
        assert jfutil.md5(b) == g["stdout_md5"][" ".join(cmd)], cmd


def test_merge_matches_reference(built, workdir, inputs):
    """merge_files (jellyfish/merge_files.cc:45-176): how per-GPU shard files become one database.  Every merge against the
    reference's merge of the same databases (tests/golden/golden_tools.json); the merged databases are the restatement's,
    which writes the same ones as the reference's count (their md5s are pinned there too)."""
    g = jfutil.golden("golden_tools.json")["merge"]
    # same size and same (first) matrix: both programs start the random stream afresh
    dbs = {}
    for name, args, ins in MERGE_COUNTS:
        dbs[name] = os.path.join(workdir, "m_%s.jf" % name)
        jfutil.run([jfutil.ORACLE_C, "count"] + args + ["-o", dbs[name]] + [inputs[i] for i in ins])
        assert jfutil.db_digest(dbs[name]) == g["counts"][name], name
    # the sum, the other operations (merge_main.cc:31-37, merge_files.cc:63-95): minimum (a k-mer missing from an input counts
    # 0 and is dropped unless -L 0 keeps it), maximum, count filters, three inputs, the Jaccard similarities; text/sorted
    # databases merge as text (merge_files.cc:168-172, text_dumper.hpp:50-80)
    for tag, switches, names in MERGE_OPS:
        out = os.path.join(workdir, "m_our_%s.jf" % tag)
        jaccard = "--jaccard" in switches
        jfutil.run([jfutil.OUR_JF, "merge"] + (["-j"] if jaccard else switches) + ["-o", out] + [dbs[n] for n in names])
        if jaccard:
            assert open(out).read() == g["merges"][tag]["text"] and open(out).read().startswith("Jaccard  "), tag
        else:
            got = jfutil.db_digest(out)
            assert got == g["merges"][tag] and got["body_len"] > 0, tag
    m2 = os.path.join(workdir, "m_our.jf")
    r = subprocess.run([jfutil.OUR_JF, "merge", "-m", "-M", "-o", m2, dbs["a"], dbs["b"]], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode != 0 and b"conflict" in r.stderr
    # formats must agree
    r = subprocess.run([jfutil.OUR_JF, "merge", "-o", m2, dbs["a"], dbs["ta"]], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode != 0 and b"different formats (binary/sorted, text/sorted)" in r.stderr
    # the last step of --disk (count_main.cc:356-371): many intermediate files of one run, written by the reference itself
    # (`count` with the switches of DISK_PARTS_COUNT, tests/golden/disk_parts/)
    part = os.path.join(jfutil.ROOT, "tests", "golden", "disk_parts", "m_part")
    parts = [part + str(i) for i in range(64) if os.path.exists(part + str(i))]
    assert len(parts) >= 3
    jfutil.run([jfutil.OUR_JF, "merge", "-o", m2] + parts)
    got = jfutil.db_digest(m2)
    assert got == g["merges"]["disk"] and got["body_len"] > 0
