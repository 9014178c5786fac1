"""GPU parity tests proper: the CUDA path, called through the C ABI (by the C++ host driver
`jellyfish-b200 count` and by the ctypes mirror), against the committed golden fixtures written by
the unmodified reference (tests/golden/) and the C restatement (oracle/jf_oracle.c).
Integer / byte work: the bar is bit-exact record bodies and equal semantic header keys."""
import json
import os
import random

import pytest

import jfutil
from cases import BC_CASES, BF_CASES, BIG_CASES, CASES, EDGE_CASES

pytestmark = pytest.mark.gpu
GOLDEN = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))


def _count_cli(workdir, inputs, name, args, ins, extra=()):
    db = os.path.join(workdir, "gpu_%s.jf" % name)
    jfutil.run([jfutil.OUR_JF, "count"] + jfutil.subst(list(args), inputs) + list(extra) + ["-o", db] + [inputs[i] for i in ins])
    return jfutil.split_db(db)


@pytest.mark.parametrize("name", sorted(CASES))
def test_cli_count_matches_reference_golden(name, built, workdir, inputs):
    args, ins = CASES[name]
    h, b = _count_cli(workdir, inputs, name, args, ins)
    g = GOLDEN[name]
    assert jfutil.semantic(h) == g["header"]
    assert len(b) == g["body_len"]
    assert jfutil.md5(b) == g["body_md5"]


def test_against_reference_binary_1m(built, workdir, inputs):
    """Same input through both programs, body compared byte for byte (1 Mbp, k=21 canonical,
    the shape of BASELINE configs[0]); the reference's `count -t 4` is in tests/golden/golden_tools.json."""
    g = jfutil.golden("golden_tools.json")["count_1m"]
    h2, b2 = _count_cli(workdir, inputs, "ours_1m", ["-m", "21", "-s", "2M", "-C"], ["plain1m.fa"])
    assert g["header"] == jfutil.semantic(h2)
    assert g["body_len"] == len(b2) and g["body_md5"] == jfutil.md5(b2)
    # and our file carries the reference's header keys; stats and histo print of it what the reference's print of its own
    assert sorted(h2) == g["header_keys"]
    ours = os.path.join(workdir, "gpu_ours_1m.jf")
    assert jfutil.run([jfutil.OUR_JF, "stats", ours]).stdout.decode() == g["stats"]
    assert jfutil.run([jfutil.OUR_JF, "histo", ours]).stdout.decode() == g["histo"]


def test_python_api_chunked_feeds(built, workdir, inputs):
    """Feeding a file in arbitrary pieces (state carried on the device) and with tiny device
    batches gives the same database as one feed."""
    from jellyfish_b200 import HashCounter
    data = open(inputs["multi.fa"], "rb").read() + b""
    g = GOLDEN["multi"]
    rng = random.Random(3)
    for batch in (0, 4096 + 16, 70000):
        with HashCounter(1000000, 7, k=17, canonical=True, max_batch_bytes=batch) as hc:
            if batch == 0:
                hc.add_text(data)
            else:
                off, first = 0, True
                while off < len(data):
                    n = rng.choice([1, 3, 17, 100, 5000, 33333, 200000])
                    hc.add_text(data[off:off + n], begin=first, end=off + n >= len(data))
                    first = False
                    off += n
            st = hc.done()
            body = hc.dump_records()
            assert jfutil.md5(body) == g["body_md5"], batch
            hdr = hc.header()
            assert {k: hdr[k] for k in jfutil.SEMANTIC_KEYS} == g["header"]
            assert st["kmers"] == st["inserted"] and st["distinct"] * (3 + 4) <= len(body) + 7 * st["distinct"]


def test_split_anywhere_including_cr(built, inputs):
    """Every split point of a small DOS/CR-laden file, two feeds each."""
    from jellyfish_b200 import HashCounter
    data = open(inputs["cr_mid.fa"], "rb").read()
    g = GOLDEN["cr_mid"]
    for cut in range(1, len(data)):
        if data[cut - 1:cut] == b"\r":
            continue   # contract of jfgpu_feed: the host never ends a non-final piece on '\r'
        with HashCounter(1000, 7, k=4, canonical=True) as hc:
            hc.add_text(data[:cut], begin=True, end=False)
            hc.add_text(data[cut:], begin=False, end=True)
            hc.done()
            assert jfutil.md5(hc.dump_records()) == g["body_md5"], cut


def test_lookup_histogram_and_stats(built, inputs):
    from jellyfish_b200 import HashCounter, ReadMerFile, mer_to_int
    import tempfile
    with HashCounter(100000, 7, k=14, canonical=True) as hc:
        hc.add_files([inputs["repeat.fa"], inputs["polya.fa"]])
        st = hc.done()
        assert st["kmers"] == (500 * 400 - 13) + (100000 - 13)
        assert st["overflowed"] > 0            # counts far beyond the in-slot counter field
        with tempfile.TemporaryDirectory() as d:
            p = os.path.join(d, "x.jf")
            nrec = hc.dump(p)
            recs = list(ReadMerFile(p))
        assert nrec == len(recs) == st["distinct"]
        assert sum(c for _, c in recs) == st["kmers"]
        mers = [m for m, _ in recs[:100]] + ["A" * 14, "ACGTACGTACGTAC"]
        vals = hc.get_many(mers)
        want = dict(recs)
        assert vals == [want.get(m, 0) for m in mers]
        assert hc.get("T" * 14) == want["A" * 14] == 100000 - 13       # canonical lookup
        assert hc["ACGTACGTACGTAC"] is None
        hist = hc.histogram(200)
        for c in range(1, 199):
            assert hist[c] == sum(1 for _, v in recs if v == c)
        assert hist[199] == sum(1 for _, v in recs if v >= 199)


def test_non_canonical_and_filters_via_api(built, inputs):
    from jellyfish_b200 import HashCounter
    with HashCounter(600000, 7, k=21, canonical=False) as hc:
        hc.add_files([inputs["plain.fa"]])
        hc.done()
        assert jfutil.md5(hc.dump_records()) == GOLDEN["k21"]["body_md5"]
    with HashCounter(10000, 7, k=21, canonical=True) as hc:
        hc.add_files([inputs["repeat.fa"]])
        hc.done()
        assert jfutil.md5(hc.dump_records(out_counter_len=1)) == GOLDEN["repeat_ocl1"]["body_md5"]
        assert jfutil.md5(hc.dump_records(lower=300, upper=400)) == GOLDEN["repeat_LU"]["body_md5"]


def test_errors(built, workdir, inputs):
    import subprocess
    from jellyfish_b200 import HashCounter, JellyfishError
    bad = os.path.join(workdir, "bad.txt")
    open(bad, "w").write("hello\nACGT\n")
    r = subprocess.run([jfutil.OUR_JF, "count", "-m", "5", "-s", "1k", "-o", os.path.join(workdir, "x.jf"), bad], stderr=subprocess.PIPE)
    assert r.returncode != 0 and b"Unsupported format" in r.stderr
    r = subprocess.run([jfutil.OUR_JF, "count", "-m", "5", "-s", "1k", "-o", os.path.join(workdir, "x.jf"), "/nonexistent.fa"], stderr=subprocess.PIPE)
    assert r.returncode != 0 and b"Can't open file" in r.stderr
    # table full and doubling disabled -> "Hash full" (hash_counter.hpp:194-195)
    with HashCounter(1000, 7, k=21, canonical=True, allow_regrow=False) as hc:
        with pytest.raises(JellyfishError) as ei:
            hc.add_files([inputs["plain.fa"]])
            hc.done()
        assert "Hash full" in str(ei.value)


def test_large_scale_properties(built):
    """At a size the CPU reference does not finish in seconds: device-generated FASTA,
    size-independent properties (total = number of windows, idempotence of a second pass
    doubling every count, stats consistency)."""
    import torch
    from jellyfish_b200 import HashCounter, _lib
    lib = _lib.load()
    n_bases = 200_000_000
    nbytes = lib.jfgpu_synth_fasta_bytes(n_bases)
    buf = torch.empty(nbytes + 64, dtype=torch.uint8, device="cuda")
    import ctypes as C
    got = C.c_uint64(0)
    assert lib.jfgpu_synth_fasta_device(0, C.c_void_p(buf.data_ptr()), nbytes + 64, n_bases, 42, C.byref(got), None) == 0
    torch.cuda.synchronize()
    with HashCounter(400_000_000, 7, k=21, canonical=True) as hc:
        hc.add_device_text(buf.data_ptr(), got.value)
        st1 = hc.done()
        assert st1["kmers"] == n_bases - 20 == st1["inserted"]
        h1 = hc.histogram(64)
        assert sum(i * h for i, h in enumerate(h1)) == st1["kmers"]
        assert sum(h1) == st1["distinct"]
        hc.add_device_text(buf.data_ptr(), got.value)
        st2 = hc.done()
        assert st2["kmers"] == 2 * st1["kmers"] and st2["distinct"] == st1["distinct"]
        h2 = hc.histogram(64)
        assert all(h2[2 * i] == h1[i] for i in range(1, 31)) and all(h2[2 * i + 1] == 0 for i in range(0, 31))


@pytest.mark.parametrize("name", ["k21C", "multi_files", "k63_multi", "k31C", "ovf32", "ovf128", "polya", "repeat", "grow2", "grow_k40", "c3", "one_per_line",
                                  "fq_long", "fq_fa_mixed"])
def test_partitioned_insertion_matches_golden(name, built, inputs):
    """The region-by-region path (records staged per table region, then inserted region by region)
    forced on small tables, including table doubling in the middle of a drain."""
    from jellyfish_b200 import HashCounter
    args, ins = CASES[name]
    opt = dict(zip(args[::2], args[1::2])) if False else {}
    it = iter(args)
    kw = {"canonical": False, "val_len": 7, "reprobes": 126}
    ocl, lower, upper = 4, 0, (1 << 64) - 1
    for a in it:
        if a == "-m": k = int(next(it))
        elif a == "-s":
            v = next(it); size = int(v[:-1]) * {"k": 10**3, "M": 10**6, "G": 10**9}[v[-1]] if v[-1] in "kMG" else int(v)
        elif a == "-C": kw["canonical"] = True
        elif a == "-c": kw["val_len"] = int(next(it))
        elif a == "-p": kw["reprobes"] = int(next(it))
        elif a == "--out-counter-len": ocl = int(next(it))
        elif a == "-L": lower = int(next(it))
        elif a == "-U": upper = int(next(it))
    g = GOLDEN[name]
    for pool in (0, 64 << 20):
        with HashCounter(size, kw["val_len"], k=k, canonical=kw["canonical"], reprobes=kw["reprobes"], part_min_mb=1,
                         pool_bytes=pool, max_batch_bytes=1 << 20) as hc:
            hc.add_files([inputs[i] for i in ins])
            st = hc.done()
            assert st["kmers"] == st["inserted"]
            body = hc.dump_records(lower, upper, ocl)
            hdr = hc.header(ocl)
            assert {x: hdr[x] for x in jfutil.SEMANTIC_KEYS} == g["header"], (name, pool)
            assert jfutil.md5(body) == g["body_md5"], (name, pool)


@pytest.mark.parametrize("name,world,part", [("k21C", 2, 0), ("multi_files", 4, 0), ("k63_multi", 2, 0), ("k31C", 8, 0),
                                             ("k21C", 2, 1), ("k63_multi", 4, 1), ("multi_files", 2, 1), ("ovf32", 2, 1)])
def test_route_and_shards_on_one_gpu(name, world, part, built, workdir, inputs):
    """The multi-GPU data path without NCCL: one engine per shard on the same device; keys bucketed
    by `jfgpu_extract_route`, handed to their owner's `jfgpu_insert_keys`, shard dumps concatenated."""
    import torch
    from jellyfish_b200 import HashCounter
    from jellyfish_b200.distributed import concat_shards
    args, ins = CASES[name]
    k = int(args[args.index("-m") + 1])
    v = args[args.index("-s") + 1]
    size = int(v[:-1]) * {"k": 10**3, "M": 10**6, "G": 10**9}[v[-1]] if v[-1] in "kMG" else int(v)
    # part=1: the owner turns the received keys into region records (K1c) and inserts them region by region
    shards = [HashCounter(size, 7, k=k, canonical="-C" in args, shard_index=r, n_shards=world, allow_regrow=False, max_batch_bytes=200000,
                          part_min_mb=part, pool_bytes=(256 << 20) if part else 0)
              for r in range(world)]
    kw = shards[0].key_words
    cap = 400000
    keys = torch.zeros((world, cap * kw), dtype=torch.int64, device="cuda")
    counts = torch.zeros(world, dtype=torch.int64, device="cuda")
    total = 0
    for i, f in enumerate(ins):
        data = open(inputs[f], "rb").read()
        buf = torch.zeros(len(data) + 256, dtype=torch.uint8, device="cuda")
        if data:
            buf[:len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        router = shards[i % world]            # any shard can do the routing: same matrix everywhere
        off = 0
        while True:
            ln = min(150000, len(data) - off)
            counts.zero_()
            torch.cuda.synchronize()
            router.extract_route(buf.data_ptr() + off, ln, keys.data_ptr(), cap, counts.data_ptr(), begin=off == 0, end=off + ln >= len(data))
            c = counts.tolist()
            assert max(c) <= cap
            for d in range(world):
                shards[d].insert_keys(keys[d].data_ptr(), c[d])
            total += sum(c)
            off += ln
            if off >= len(data):
                break
    out = os.path.join(workdir, "route1_%s_%d_%d" % (name, world, part))
    n_ins = 0
    for r, hc in enumerate(shards):
        st = hc.done()
        n_ins += st["inserted"]
        hc.dump("%s.%d" % (out, r))
        hc.close()
    assert n_ins == total
    h, b = jfutil.split_db(concat_shards(out, world, out + ".jf"))
    g = GOLDEN[name]
    assert jfutil.semantic(h) == g["header"]
    assert jfutil.md5(b) == g["body_md5"]


def test_fastq_without_final_newline(built, workdir, inputs):
    """Deliberate divergence from a reference bug: when a FASTQ file lacks the final newline the
    reference throws inside skip_quals (mer_overlap_sequence_parser.hpp:290-307), the exception is
    swallowed by the producer (cooperative_pool2.hpp:252) and the last buffer of reads is silently
    lost (an 2-read file gives an EMPTY database).  The engine counts every read; the checker here is
    the C restatement, which implements the documented semantics without that loss."""
    from jellyfish_b200 import HashCounter
    db = os.path.join(workdir, "noeol_oracle.jf")
    jfutil.run([jfutil.ORACLE_C, "count", "-m", "31", "-s", "600k", "-o", db, inputs["reads_noeol.fq"]])
    h, b = jfutil.split_db(db)
    with HashCounter(600000, 7, k=31, canonical=False) as hc:
        hc.add_files([inputs["reads_noeol.fq"]])
        hc.done()
        assert hc.dump_records() == b
        hdr = hc.header()
        assert {x: hdr[x] for x in jfutil.SEMANTIC_KEYS} == jfutil.semantic(h)


def test_fastq_format_errors(built, workdir):
    """Not 4-line FASTQ -> loud failure ("Invalid fastq sequence"), never a silent miscount."""
    from jellyfish_b200 import HashCounter, JellyfishError
    bad = b"@r1\nACGTACGTAC\nACGTACGTAA\n+\nIIIIIIIIIIIIIIIIIIII\n@r2\nACGT\n+\nIIII\n"     # two sequence lines
    with HashCounter(1000, 7, k=4, canonical=True) as hc:
        with pytest.raises(JellyfishError) as ei:
            hc.add_text(bad)
            hc.done()
        assert "fastq" in str(ei.value).lower()


def test_skewed_input_in_region_mode(built, workdir):
    """20 Mbp with long low-complexity stretches (poly-A, short tandem repeats) through the default
    region-by-region path (table >= 256 MB): hot regions overflow their chunks within one iteration,
    so the spill list and the direct-insertion fallback are exercised under load.  Checked against the
    C restatement (sort-based, so independent of any table)."""
    import gen
    from jellyfish_b200 import HashCounter
    parts = [gen._seq(5000000, 71), b"A" * 4000000, b"ACG" * 1500000, gen._seq(3000000, 72), b"AT" * 1000000, gen._seq(1500000, 73)]
    fa = os.path.join(workdir, "skew.fa")
    with open(fa, "wb") as f:
        f.write(gen.fasta(b"".join(parts)))
    db = os.path.join(workdir, "skew_oracle.jf")
    jfutil.run([jfutil.ORACLE_C, "count", "-m", "21", "-s", "64M", "-C", "-o", db, fa])
    h, b = jfutil.split_db(db)
    with HashCounter(64000000, 7, k=21, canonical=True) as hc:
        assert hc.info()["part_regions"] > 0
        hc.add_files([fa])
        st = hc.done()
        assert st["kmers"] == st["inserted"]
        assert hc.dump_records() == b
        hdr = hc.header()
        assert {x: hdr[x] for x in jfutil.SEMANTIC_KEYS} == jfutil.semantic(h)


@pytest.mark.parametrize("part", [0, 1])
def test_if_passes_via_api(part, built, inputs):
    """`count --if`: PRIME the keys of one file (count 0), then UPDATE with the others -- through the
    Python mirror, in both insertion modes (direct / region by region)."""
    from jellyfish_b200 import HashCounter
    g = GOLDEN["if_sub"]
    with HashCounter(1000000, 7, k=17, canonical=True, part_min_mb=part, pool_bytes=(128 << 20) if part else 0, max_batch_bytes=1 << 20) as hc:
        hc.set_op(HashCounter.OP_PRIME)
        hc.add_files([inputs["multi2.fa"]])
        hc.set_op(HashCounter.OP_UPDATE)
        hc.add_files([inputs["multi.fa"], inputs["multi2.fa"], inputs["dangling.fa"]])
        hc.done()
        assert jfutil.md5(hc.dump_records()) == g["body_md5"]
        hdr = hc.header()
        assert {x: hdr[x] for x in jfutil.SEMANTIC_KEYS} == g["header"]


@pytest.mark.parametrize("name", sorted(BIG_CASES))
def test_cli_count_matches_reference_golden_large_table(name, built, workdir, inputs):
    """A table of 2^31 slots (8 GB of 32-bit slots): the matrix has 31 rows, where the reference's
    random_bits() overlaps its draws (lib/misc.cc:66-72); header and body against the reference's golden."""
    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_big.json")))
    args, ins = BIG_CASES[name]
    db = os.path.join(workdir, "gpu_%s.jf" % name)
    jfutil.run([jfutil.OUR_JF, "count"] + list(args) + ["-o", db] + [inputs[i] for i in ins], timeout=600)
    h, b = jfutil.split_db(db)
    g = golden[name]
    assert jfutil.semantic(h) == g["header"]
    assert len(b) == g["body_len"]
    assert jfutil.md5(b) == g["body_md5"]


# Corner cases where the REFERENCE loses k-mers or occurrences (tiny tables that double many times with a clipped reprobe
# limit, counts beyond val_len in tiny / direct-indexed tables): its own count on a roomy table disagrees with its count
# on the tiny one.  name -> (k-mers missing from the reference's output, k-mers whose count it reports too low).
# The engine is held to the reference's HEADER (final size, carried reprobe limit, matrix, val_len) and to the exact counts.
EDGE_REFERENCE_LOSES = {
    "edge_c1_p2": (1, 1), "edge_k5_s10_c1": (0, 11), "edge_k5_s2_p10": (0, 2), "edge_s2_k31_p62": (7, 0), "edge_s2_ties": (6, 0),
}


@pytest.mark.parametrize("name", sorted(EDGE_CASES))
def test_cli_count_corner_cases_against_reference_golden(name, built, workdir, inputs):
    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_edge.json")))
    args, ins = EDGE_CASES[name]
    h, b = _count_cli(workdir, inputs, name, args, ins)
    g = golden[name]
    assert jfutil.semantic(h) == g["header"]
    if name not in EDGE_REFERENCE_LOSES:
        assert len(b) == g["body_len"]
        assert jfutil.md5(b) == g["body_md5"]
        return
    # documented divergence (DESIGN.md section 7a): exact counts, in (position, key) order
    missing, low = EDGE_REFERENCE_LOSES[name]
    rec = (h["key_len"] + 7) // 8 + h["counter_len"]
    assert len(b) == g["body_len"] + missing * rec and jfutil.md5(b) != g["body_md5"]
    roomy = [a for a in args]
    roomy[roomy.index("-s") + 1] = "4M"
    for sw in ("-p", "-c"):
        if sw in roomy:
            i = roomy.index(sw); del roomy[i:i + 2]
    ref = os.path.join(workdir, "roomy_%s.jf" % name)
    jfutil.run([jfutil.ORACLE_C, "count"] + roomy + ["-o", ref] + [inputs[i] for i in ins])
    hr, br = jfutil.split_db(ref)
    got = jfutil.records(h, b)
    assert dict(got) == dict(jfutil.records(hr, br)) and len(got) == len(dict(got))
    order = [(jfutil.hash_pos(h, k), k) for k, _ in got]
    assert order == sorted(order)
    # the reference itself, on this tiny table, against the exact counts: the losses named above.  Its records are the
    # exact ones but for those listed in tests/golden/golden_tools.json (count None: missing), held to its digest there.
    e = jfutil.golden("golden_tools.json")["edge_losses"][name]
    true = dict(got)
    rt = dict(true)
    for key, v in e["differs"]:
        if v is None:
            del rt[key]
        else:
            rt[key] = v
    assert jfutil.records_md5(rt.items()) == e["records_md5"]
    assert len(true) - len(rt) == missing and sum(1 for k in rt if rt[k] < true[k]) == low


GOLDEN_BC = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_bc.json")))
GOLDEN_BF = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_bf.json")))


@pytest.mark.parametrize("name", sorted(BC_CASES))
def test_bloom_counter_matches_reference_golden(name, built, workdir, inputs):
    """`jellyfish bc` on the device (file byte for byte: the counter does not depend on the insertion order), then
    `count --bc FILE` (bc_main.cc:84-161, count_main.cc:110-120,191-206) against the reference's goldens."""
    bargs, bins, cargs, cins = BC_CASES[name]
    g = GOLDEN_BC[name]
    bc = os.path.join(workdir, "gpu_%s.bc" % name)
    jfutil.run([jfutil.OUR_JF, "bc"] + bargs + ["-o", bc] + [inputs[i] for i in bins])
    hb, bb = jfutil.split_db(bc)
    assert {k: hb.get(k) for k in g["bc_header"]} == g["bc_header"]
    assert len(bb) == g["bc_len"] and jfutil.md5(bb) == g["bc_md5"]
    db = os.path.join(workdir, "gpu_%s_bc.jf" % name)
    jfutil.run([jfutil.OUR_JF, "count"] + cargs + ["--bc", bc, "-o", db] + [inputs[i] for i in cins])
    h, b = jfutil.split_db(db)
    assert jfutil.semantic(h) == g["header"]
    assert len(b) == g["body_len"] and jfutil.md5(b) == g["body_md5"]


def test_bloom_counter_python_api(built, workdir, inputs):
    from jellyfish_b200 import BloomCounter, HashCounter
    bargs, bins, cargs, cins = BC_CASES["bc_k21C"]
    g = GOLDEN_BC["bc_k21C"]
    bc = os.path.join(workdir, "api.bc")
    with BloomCounter(400000, 0.001, k=21, canonical=True) as b:
        b.add_files([inputs[i] for i in bins])
        b.dump(bc)
    hb, bb = jfutil.split_db(bc)
    assert {k: hb.get(k) for k in g["bc_header"]} == g["bc_header"] and jfutil.md5(bb) == g["bc_md5"]
    with HashCounter(1000000, 7, k=21, canonical=True) as hc:
        hc.load_bloom_counter(bc)
        hc.add_files([inputs[i] for i in cins])
        st = hc.done()
        assert st["inserted"] < st["kmers"]
        assert jfutil.md5(hc.dump_records()) == g["body_md5"]


@pytest.mark.parametrize("name", sorted(n for n in BF_CASES if "-Q" not in BF_CASES[n][0]))
def test_bloom_prefilter_against_reference_golden(name, built, workdir, inputs):
    """count --bf-size (count_main.cc:122-133,317-321).  Which first occurrences pass as false positives depends on the
    insertion order (the reference's own output changes with -t), so the device path is held to: the same header as
    the reference's -t 1 run, every count in {occ - 1, occ}, and a false-positive rate of the order asked for."""
    args, ins = BF_CASES[name]
    g = GOLDEN_BF[name]
    db = os.path.join(workdir, "gpu_%s.jf" % name)
    jfutil.run([jfutil.OUR_JF, "count"] + args + ["-o", db] + [inputs[i] for i in ins])
    h, b = jfutil.split_db(db)
    assert jfutil.semantic(h) == g["header"]
    # occurrences: the same switches without the filter, through the restatement
    plain = [a for a in args]
    for sw in ("--bf-size", "--bf-fp"):
        if sw in plain:
            i = plain.index(sw); del plain[i:i + 2]
    ref = os.path.join(workdir, "occ_%s.jf" % name)
    jfutil.run([jfutil.ORACLE_C, "count"] + plain + ["-o", ref] + [inputs[i] for i in ins])
    hr, br = jfutil.split_db(ref)
    occ = dict(jfutil.records(hr, br))
    got = dict(jfutil.records(h, b))
    assert set(got) <= set(occ)
    cap = (1 << (8 * h["counter_len"])) - 1
    bad = [k for k, v in got.items() if v not in (min(occ[k], cap), min(occ[k] - 1, cap))]
    assert not bad, "counts outside {occ-1, occ}: %d" % len(bad)
    missing = [k for k in occ if k not in got and occ[k] > 1]
    assert not missing, "k-mers seen more than once must be present: %d missing" % len(missing)
    # false positives = singletons that got through.  The yardstick is the reference's own -t 1 run (golden body length):
    # an undersized filter (bf_fp10_grow: 200k for 585k distinct mers) passes far more than --bf-fp, in the reference too
    singles = [k for k in occ if occ[k] == 1]
    passed = sum(1 for k in singles if k in got)
    rec = (h["key_len"] + 7) // 8 + h["counter_len"]
    ref_passed = g["body_len"] // rec - (len(occ) - len(singles))
    assert 0 <= ref_passed <= len(singles)
    assert abs(passed - ref_passed) <= 50 + 0.05 * ref_passed + 4 * ref_passed ** 0.5, "false positives: %d of %d singletons, reference %d" % (passed, len(singles), ref_passed)


def test_baseline_config0_100mbp_body_md5(built, workdir):
    """BASELINE configs[0]: `count -m 21 -s 100M -C` on `generate_sequence -s 3141592653 100000000`.  The body md5 is the
    one the reference produced for -t 1 and -t 8 (SURVEY.md section 8c); input md5 pins the generator (tests/gen.py)."""
    fa, = jfutil.generate(os.path.join(workdir, "seq100m"), 3141592653, 100000000)
    assert os.path.getsize(fa) == 101428586 and jfutil.md5(open(fa, "rb").read()) == "94b718fdd506b6528bd574818bb753ea"
    db = os.path.join(workdir, "gpu_cfg0.jf")
    jfutil.run([jfutil.OUR_JF, "count", "-m", "21", "-s", "100M", "-C", "-o", db, fa], timeout=600)
    h, b = jfutil.split_db(db)
    assert h["size"] == 134217728 and h["key_len"] == 42 and h["max_reprobe"] == 126 and h["val_len"] == 7
    assert h["matrix1"]["r"] == 27 and h["matrix1"]["c"] == 42
    assert h["matrix1"]["columns"][:3] == [64834949, 57999349, 22595292] and h["matrix1"]["columns"][41] == 69326724
    assert len(b) == 99997658 * 10
    assert jfutil.md5(b) == "63058a336e1d9431eb6618d4a4f4deed"


@pytest.mark.parametrize("name,world", [("multi_files", 2), ("multi_files", 4), ("k15C", 2), ("fq_dos", 2), ("c3", 2), ("x17_4M", 8)])
def test_record_exchange_on_one_gpu(name, world, built, workdir, inputs):
    """The record form of the multi-GPU data path without NCCL: one engine per shard on the same device.  K1 files 4-byte
    records of the GLOBAL regions by owning shard (jfgpu_shard_extract / _pack), the chunks are copied into the owners'
    receive pools the way the all-to-all would, the owners re-file them under their own regions (jfgpu_shard_unpack) and
    drain them; the concatenated shard dumps must be the reference's database."""
    import torch
    from jellyfish_b200 import HashCounter
    from jellyfish_b200.distributed import CHUNK, concat_shards
    # (x17_4M: no golden of that size -- eight shards need a table of 4M slots to be filled region by region; the yardstick
    # is the single-GPU engine, itself held to the goldens above)
    args, ins = CASES[name] if name in CASES else (["-m", "17", "-s", "4M", "-C"], ["plain1m.fa"])
    k = int(args[args.index("-m") + 1])
    v = args[args.index("-s") + 1]
    size = int(v[:-1]) * {"k": 10**3, "M": 10**6, "G": 10**9}[v[-1]] if v[-1] in "kMG" else int(v)
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    arena = 2 * n_sm * max(1, 1024 // world) + 64
    shards, bufs = [], []
    for r in range(world):
        hc = HashCounter(size, int(args[args.index("-c") + 1]) if "-c" in args else 7, k=k, canonical="-C" in args, shard_index=r, n_shards=world,
                         allow_regrow=False, part_min_mb=1, pool_bytes=4 << 30)      # (an arena must take a batch of 1024 chunks)
        send = torch.empty(2 * world * arena * CHUNK, dtype=torch.uint8, device="cuda")
        send_dir = torch.empty(2 * world * arena * 8, dtype=torch.uint8, device="cuda")
        recv = torch.empty(world * arena * CHUNK, dtype=torch.uint8, device="cuda")
        recv_dir = torch.empty(world * arena * 8, dtype=torch.uint8, device="cuda")
        assert hc.shard_setup(send.data_ptr(), send_dir.data_ptr(), arena, recv.data_ptr(), recv_dir.data_ptr(), arena), "geometry not covered"
        assert hc.shard_round_bytes() >= 1 << 20
        shards.append(hc)
        bufs.append((send, send_dir, recv, recv_dir))
    n_round = 0
    for i, f in enumerate(ins):
        data = open(inputs[f], "rb").read()
        buf = torch.zeros(len(data) + 256, dtype=torch.uint8, device="cuda")
        if data:
            buf[:len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        src = i % world
        router = shards[src]
        off = 0
        while True:
            ln = min(170000, len(data) - off)
            bank = n_round & 1
            n_round += 1
            router.shard_extract(buf.data_ptr() + off, ln, bank, begin=off == 0, end=off + ln >= len(data))
            counts = router.shard_pack(bank)
            assert max(counts) <= arena
            send, send_dir = bufs[src][0], bufs[src][1]
            for d in range(world):
                c = counts[d]
                recv, recv_dir = bufs[d][2], bufs[d][3]
                a0 = (bank * world + d) * arena
                recv[src * arena * CHUNK:(src * arena + c) * CHUNK] = send[a0 * CHUNK:(a0 + c) * CHUNK]
                recv_dir[src * arena * 8:(src * arena + c) * 8] = send_dir[a0 * 8:(a0 + c) * 8]
                torch.cuda.synchronize()
                got = [0] * world
                got[src] = c
                shards[d].shard_unpack(got)
                torch.cuda.synchronize()
            off += ln
            if off >= len(data):
                break
    out = os.path.join(workdir, "recx_%s_%d" % (name, world))
    n_kmers = n_ins = 0
    for r, hc in enumerate(shards):
        st = hc.done()
        n_kmers += st["kmers"]
        n_ins += st["inserted"]
        hc.dump("%s.%d" % (out, r))
        hc.close()
    assert n_ins == n_kmers > 0
    h, b = jfutil.split_db(concat_shards(out, world, out + ".jf"))
    if name in GOLDEN:
        g = GOLDEN[name]
        assert jfutil.semantic(h) == g["header"]
        assert jfutil.md5(b) == g["body_md5"]
    else:
        with HashCounter(size, 7, k=k, canonical="-C" in args, allow_regrow=False) as one:
            one.add_files([inputs[f] for f in ins])
            one.done()
            assert jfutil.md5(one.dump_records()) == jfutil.md5(b) and len(b) > 0
            hdr = one.header()
            assert {x: hdr[x] for x in jfutil.SEMANTIC_KEYS} == jfutil.semantic(h)


GOLDEN_QUAL = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_qual.json")))
QUAL_MULTILINE = ("q_ml", "q_mixed")       # inputs with FASTQ records wrapped over several lines


@pytest.mark.parametrize("name", sorted(n for n in __import__("cases").QUAL_CASES))
def test_quality_filter_matches_reference_golden(name, built, workdir, inputs):
    """-Q / --min-quality on the device (count_main.cc:234-256,326-329; whole_sequence_parser.hpp:137-193;
    mer_qual_iterator.hpp:64-92): 4-line FASTQ records and FASTA, byte for byte against the reference's goldens.
    FASTQ records wrapped over several lines are rejected loudly (DESIGN.md section 7a)."""
    import subprocess
    from cases import QUAL_CASES
    args, ins = QUAL_CASES[name]
    if name in QUAL_MULTILINE:
        r = subprocess.run([jfutil.OUR_JF, "count"] + jfutil.subst(list(args), inputs) + ["-o", os.path.join(workdir, "q.jf")] + [inputs[i] for i in ins],
                           stderr=subprocess.PIPE)
        assert r.returncode != 0 and b"Invalid fastq" in r.stderr
        return
    h, b = _count_cli(workdir, inputs, name, args, ins)
    g = GOLDEN_QUAL[name]
    assert jfutil.semantic(h) == g["header"]
    assert len(b) == g["body_len"]
    assert jfutil.md5(b) == g["body_md5"]


def test_quality_filter_python_api_split_feeds(built, inputs):
    """The same through the ctypes mirror with the file fed in arbitrary pieces: the engine keeps the incomplete last read of a
    feed for the next one."""
    from jellyfish_b200 import HashCounter
    from cases import QUAL_CASES
    args, ins = QUAL_CASES["q_fq"]
    data = open(inputs[ins[0]], "rb").read()
    g = GOLDEN_QUAL["q_fq"]
    rng = random.Random(11)
    with HashCounter(1000000, 7, k=21, canonical=True, min_qual="5", max_batch_bytes=70000) as hc:
        off, first = 0, True
        while off < len(data):
            n = rng.choice([1, 7, 300, 5000, 44444, 200000])
            hc.add_text(data[off:off + n], begin=first, end=off + n >= len(data))
            first = False
            off += n
        hc.done()
        assert jfutil.md5(hc.dump_records()) == g["body_md5"]


def test_shard_records_of_a_2_to_37_slot_table_match_the_host_hash(built, inputs):
    """The send side of the record exchange at the bench's 8-GPU geometry (global table 2^37 slots, five position bits
    beyond the 32 the table-driven hash produces: parity rows): every record K1 files -- (global region, position in the
    region, explicit key bits) -- against the position computed on the host from the hash matrix the header would carry."""
    import numpy as np
    import torch
    from jellyfish_b200 import HashCounter, canonical_int, mer_to_int
    from jellyfish_b200.distributed import CHUNK
    world, k = 8, 21
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    arena = 2 * n_sm * (1024 // world) + 64
    with HashCounter(1 << 37, 7, k=k, canonical=True, shard_index=3, n_shards=world, allow_regrow=False) as hc:
        info = hc.info()
        assert info["lsize"] == 37 and info["matrix_r"] == 37
        send = torch.zeros(2 * world * arena * CHUNK, dtype=torch.uint8, device="cuda")
        send_dir = torch.zeros(2 * world * arena * 8, dtype=torch.uint8, device="cuda")
        recv = torch.zeros(world * arena * CHUNK, dtype=torch.uint8, device="cuda")
        recv_dir = torch.zeros(world * arena * 8, dtype=torch.uint8, device="cuda")
        assert hc.shard_setup(send.data_ptr(), send_dir.data_ptr(), arena, recv.data_ptr(), recv_dir.data_ptr(), arena)
        data = open(inputs["plain.fa"], "rb").read()
        buf = torch.zeros(len(data) + 256, dtype=torch.uint8, device="cuda")
        buf[:len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        hc.shard_extract(buf.data_ptr(), len(data), 0)
        counts = hc.shard_pack(0)
        torch.cuda.synchronize()
        got = []
        for d in range(world):
            c = counts[d]
            dirs = send_dir[d * arena * 8:(d * arena + c) * 8].cpu().numpy().view(np.uint32).reshape(-1, 2)
            chunks = send[d * arena * CHUNK:(d * arena + c) * CHUNK].cpu().numpy().view(np.uint32).reshape(-1, CHUNK // 4)
            for (region, n), recs in zip(dirs, chunks):
                assert region // (1024 // world) == d            # the chunk sits in its owner's arena
                got.extend((int(region) << 32) | int(x) for x in recs[:n])
        # the host's version: canonical 21-mers of the sequence, position = matrix x key, region = top 10 bits of the 37
        seq = "".join(l.strip() for l in data.decode().splitlines() if not l.startswith(">"))
        cols, c = info["matrix_columns"], info["matrix_c"]
        hb = 2 * k - 37
        want = []
        for i in range(len(seq) - k + 1):
            key = canonical_int(mer_to_int(seq[i:i + k]), k)
            h, x, j = 0, key, 0
            while x:
                if x & 1:
                    h ^= cols[c - 1 - j]
                x >>= 1
                j += 1
            pos = h & ((1 << 37) - 1)
            want.append(((pos >> 27) << 32) | ((pos & ((1 << 27) - 1)) << hb) | (key >> 37))
        assert sorted(got) == sorted(want)


@pytest.mark.parametrize("name", sorted(__import__("cases").DISK_CASES))
def test_disk_spill_and_merge_matches_reference_golden(name, built, workdir, inputs):
    """--disk: the table does not double; when it is full the engine calls the spill hook (jfgpu_set_spill), the driver writes
    <output>0, <output>1, ... and merges them at the end (count_main.cc:346-371).  Header and body against the reference's."""
    from cases import DISK_CASES
    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_disk.json")))
    args, ins = DISK_CASES[name]
    db = os.path.join(workdir, "gpu_%s.jf" % name)
    jfutil.run([jfutil.OUR_JF, "count"] + list(args) + ["-o", db] + [inputs[i] for i in ins])
    h, b = jfutil.split_db(db)
    g = golden[name]
    assert jfutil.semantic(h) == g["header"]
    assert len(b) == g["body_len"] and jfutil.md5(b) == g["body_md5"]
    assert not os.path.exists(db + "0")              # intermediate files are unlinked after the merge
    # --no-merge leaves the intermediate files, each a valid database of the same geometry
    db2 = os.path.join(workdir, "gpu_%s_parts.jf" % name)
    jfutil.run([jfutil.OUR_JF, "count"] + list(args) + ["--no-merge", "-o", db2] + [inputs[i] for i in ins])
    parts = [db2 + str(i) for i in range(64) if os.path.exists(db2 + str(i))]
    assert len(parts) >= 2
    total = {}
    for part in parts:
        hp, bp = jfutil.split_db(part)
        assert hp["size"] == h["size"] and hp["matrix1"] == h["matrix1"]
        for key, v in jfutil.records(hp, bp):
            total[key] = total.get(key, 0) + v
    lo = int(args[args.index("-L") + 1]) if "-L" in args else 0
    cap = (1 << (8 * h["counter_len"])) - 1
    assert {key: min(v, cap) for key, v in total.items() if v >= lo} == dict(jfutil.records(h, b))


def _generator_file(workdir, inputs, tag, names):
    """A -g file whose commands write the given inputs on their standard output, every second one through gunzip when
    gzip is here (the reference's own use: tests/multi_file.sh:16-23); blank lines and comments in between."""
    import shlex
    import shutil
    import subprocess
    lines = ["", "   ", "# generator commands of " + tag]
    for i, n in enumerate(names):
        path = inputs[n]
        if i % 2 == 1 and shutil.which("gzip") and shutil.which("gunzip"):
            gz = os.path.join(workdir, "%s_%d.gz" % (tag, i))
            with open(gz, "wb") as f:
                subprocess.run(["gzip", "-c", path], stdout=f, check=True)
            lines.append("  gunzip -c %s" % shlex.quote(gz))
        else:
            lines.append("cat %s" % shlex.quote(path))
        lines.append("")
    cmds = os.path.join(workdir, tag + "_cmds")
    with open(cmds, "w") as f:
        f.write("\n".join(lines) + "\n")
    return cmds


@pytest.mark.parametrize("name,width", [("multi_files", 2), ("fq_fa_mixed", 3), ("k63_multi", 1)])
def test_generator_commands_count_like_files(name, width, built, workdir, inputs):
    """-g / -G / -S (lib/generator_manager.cc, count_main.cc:260-267,297-303): the first input as a file, the others as the
    outputs of generator commands run `width` at a time -- every output one input file of its own -- against the reference's
    golden for the same inputs given as files (the database does not depend on how or in which order the inputs arrive)."""
    args, ins = CASES[name]
    cmds = _generator_file(workdir, inputs, "gen_" + name, ins[1:])
    h, b = _count_cli(workdir, inputs, "gen_" + name, args, ins[:1], extra=["-g", cmds, "-G", str(width), "-S", "/bin/sh"])
    g = GOLDEN[name]
    assert jfutil.semantic(h) == g["header"]
    assert len(b) == g["body_len"] and jfutil.md5(b) == g["body_md5"]


def test_bloom_counter_from_generator_commands(built, workdir, inputs):
    """`bc -g` (bc_main.cc:95-103,127-143; tests/bloom_counter.sh:11-15): no file argument at all, the file byte for byte"""
    bargs, bins, _, _ = BC_CASES["bc_k21C"]
    g = GOLDEN_BC["bc_k21C"]
    cmds = _generator_file(workdir, inputs, "gen_bc", bins)
    bc = os.path.join(workdir, "gpu_gen_bc.bc")
    jfutil.run([jfutil.OUR_JF, "bc"] + bargs + ["-g", cmds, "-G", "2", "-o", bc])
    hb, bb = jfutil.split_db(bc)
    assert {k: hb.get(k) for k in g["bc_header"]} == g["bc_header"]
    assert len(bb) == g["bc_len"] and jfutil.md5(bb) == g["bc_md5"]


def test_failing_generator_command_fails_the_count(built, workdir, inputs):
    """tests/multi_file.sh:25-33"""
    import subprocess
    cmds = os.path.join(workdir, "gen_fail_cmds")
    with open(cmds, "w") as f:
        f.write("cat %s\nfalse\n" % inputs["plain.fa"])
    r = subprocess.run([jfutil.OUR_JF, "count", "-m", "21", "-s", "600k", "-C", "-g", cmds, "-G", "2", "-o", os.path.join(workdir, "gen_fail.jf")],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode != 0
    assert b"Command 'false' exited with error status 1" in r.stderr and b"Some generator commands failed" in r.stderr
