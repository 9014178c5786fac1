"""Parity cases: name -> (count switches, input files of tests/gen.py).

Configurations follow the reference's own integration tests (tests/parallel_hashing.sh,
merge.sh, multi_file.sh, small_mers.sh, large_key.sh) scaled to inputs that the CPU reference
counts in seconds, plus the edge cases of SURVEY.md section 8a.
"""
CASES = {
    # geometry sweep: slot widths 32 / 64 / 128, one- and two-word keys
    "k21C":         (["-m", "21", "-s", "600k", "-C"], ["plain.fa"]),
    "k21":          (["-m", "21", "-s", "600k"], ["plain.fa"]),
    "k15C":         (["-m", "15", "-s", "1M", "-C"], ["plain.fa"]),
    "k31C":         (["-m", "31", "-s", "600k", "-C"], ["plain.fa"]),
    "k32C":         (["-m", "32", "-s", "600k", "-C"], ["plain.fa"]),
    "k33C":         (["-m", "33", "-s", "600k", "-C"], ["plain.fa"]),
    "k40":          (["-m", "40", "-s", "600k"], ["plain.fa"]),
    "k63C":         (["-m", "63", "-s", "700k", "-C"], ["plain.fa"]),
    "k64C":         (["-m", "64", "-s", "700k", "-C"], ["plain.fa"]),
    "k24_tiny":     (["-m", "24", "-s", "300k", "-C", "-p", "30"], ["plain.fa"]),
    # small mers / direct indexing (tests/small_mers.sh)
    "k2C":          (["-m", "2", "-s", "1M", "-C"], ["plain.fa"]),
    "k5_1k":        (["-m", "5", "-s", "1k", "-C"], ["plain.fa"]),
    "k8":           (["-m", "8", "-s", "10M"], ["plain.fa"]),
    "k10C":         (["-m", "10", "-s", "1M", "-C"], ["plain.fa"]),
    # input text semantics
    "dos":          (["-m", "21", "-s", "600k", "-C"], ["dos.fa"]),
    "noeol":        (["-m", "21", "-s", "600k", "-C"], ["noeol.fa"]),
    "lower":        (["-m", "21", "-s", "600k", "-C"], ["lower.fa"]),
    "multi":        (["-m", "17", "-s", "1M", "-C"], ["multi.fa"]),
    "multi_files":  (["-m", "17", "-s", "1M", "-C"], ["multi.fa", "empty.fa", "multi2.fa", "header_only.fa", "dangling.fa"]),
    "one_per_line": (["-m", "25", "-s", "100k", "-C"], ["one_per_line.fa"]),
    "blank_runs":   (["-m", "31", "-s", "100k", "-C"], ["blank_runs.fa"]),
    "long_header":  (["-m", "21", "-s", "100k"], ["long_header.fa"]),
    "cr_mid":       (["-m", "4", "-s", "1k", "-C"], ["cr_mid.fa"]),
    "oneline":      (["-m", "21", "-s", "300k", "-C"], ["oneline.fa"]),
    "k63_multi":    (["-m", "63", "-s", "1M", "-C"], ["multi.fa", "dos.fa"]),
    # FASTQ, default path (no -Q): mer_overlap_sequence_parser.hpp:187-217,290-307
    # (a FASTQ file WITHOUT a final newline is not a golden case: the reference silently drops the
    #  last buffer of such a file -- see tests/test_gpu_parity.py::test_fastq_without_final_newline)
    "fq":           (["-m", "21", "-s", "1M", "-C"], ["reads.fq"]),
    "fq_dos":       (["-m", "17", "-s", "600k", "-C"], ["reads_dos.fq"]),
    "fq_long":      (["-m", "25", "-s", "2M", "-C"], ["reads_long.fq"]),
    "fq_k63":       (["-m", "63", "-s", "1M", "-C"], ["reads.fq", "one_read.fq"]),
    "fq_fa_mixed":  (["-m", "21", "-s", "2M", "-C"], ["reads.fq", "multi.fa", "reads_dos.fq", "plain.fa", "one_read.fq"]),
    # counters: large counts, output clipping, count filters
    "polya":        (["-m", "21", "-s", "1k", "-C"], ["polya.fa"]),
    "repeat":       (["-m", "21", "-s", "10k", "-C"], ["repeat.fa"]),
    "repeat_ocl1":  (["-m", "21", "-s", "10k", "-C", "--out-counter-len", "1"], ["repeat.fa"]),
    "repeat_LU":    (["-m", "21", "-s", "10k", "-C", "-L", "300", "-U", "400"], ["repeat.fa"]),
    # counter-field carries in each slot width (14-, 8- and 15-bit in-slot counters)
    "ovf32":        (["-m", "14", "-s", "100k", "-C"], ["polya.fa", "repeat.fa"]),
    "ovf64":        (["-m", "32", "-s", "30k", "-C"], ["polya.fa", "repeat.fa"]),
    "ovf128":       (["-m", "63", "-s", "700k", "-C"], ["polya.fa", "repeat.fa"]),
    "text":         (["-m", "21", "-s", "600k", "-C", "--text"], ["plain.fa"]),
    "text_k40_LU":  (["-m", "40", "-s", "10k", "--text", "-L", "2"], ["repeat.fa", "polya.fa"]),
    # --if: count only the k-mers of the given files (PRIME then UPDATE, tests/subset_hashing.sh)
    "if_sub":       (["-m", "17", "-s", "1M", "-C", "--if", "@multi2.fa"], ["multi.fa", "multi2.fa", "dangling.fa"]),
    "if_zeros":     (["-m", "21", "-s", "600k", "--if", "@plain.fa", "--if", "@dangling.fa"], ["multi.fa", "dangling.fa"]),
    "if_k40_rep":   (["-m", "40", "-s", "10k", "-C", "--if", "@repeat.fa"], ["repeat.fa", "polya.fa", "repeat.fa"]),
    "c3":           (["-m", "12", "-s", "300k", "-C", "-c", "3"], ["plain.fa"]),
    # size doubling with new matrix draws (hash_counter.hpp:200-238)
    "grow2":        (["-m", "21", "-s", "100k", "-C"], ["plain.fa"]),
    "grow_k40":     (["-m", "40", "-s", "50k"], ["plain.fa"]),
    "grow_to_full": (["-m", "8", "-s", "10k", "-C"], ["plain.fa"]),
}

# -Q / --min-quality (count_main.cc:326-329: whole_sequence_parser + mer_qual_iterator). The
# restatement is pinned against these; the device path for them is a round-2 row, so they are
# kept apart from CASES (which the GPU parity tests iterate). FASTA files come before FASTQ files in
# a case: read_fasta (whole_sequence_parser.hpp:137-152) never clears the record's quality string,
# so a FASTA record read into a buffer slot that held a FASTQ read is filtered with that read's
# stale qualities -- which slot depends on thread timing; not reproduced (DESIGN.md section 7a).
QUAL_CASES = {
    "q_fq":        (["-m", "21", "-s", "1M", "-C", "-Q", "5"], ["reads_q.fq"]),
    "q_fq_hi":     (["-m", "17", "-s", "1M", "-Q", "G"], ["reads_q.fq"]),
    "q_minq":      (["-m", "17", "-s", "1M", "-C", "--min-quality", "20", "--quality-start", "33"], ["reads_q.fq"]),
    "q_minq_dflt": (["-m", "15", "-s", "1M", "-C", "--min-quality", "6"], ["reads_q.fq"]),
    "q_all_pass":  (["-m", "21", "-s", "1M", "-C", "-Q", "!"], ["reads.fq"]),
    "q_uniform":   (["-m", "12", "-s", "1M", "-C", "-Q", "#"], ["reads.fq"]),
    "q_dos":       (["-m", "17", "-s", "600k", "-C", "-Q", "5"], ["reads_q_dos.fq"]),
    "q_noeol":     (["-m", "21", "-s", "1M", "-C", "-Q", "\""], ["reads_noeol.fq"]),
    "q_long":      (["-m", "25", "-s", "2M", "-C", "-Q", "\""], ["reads_long.fq"]),
    "q_ml":        (["-m", "21", "-s", "1M", "-C", "-Q", "$"], ["reads_ml.fq"]),
    "q_fa":        (["-m", "21", "-s", "1M", "-C", "-Q", "5"], ["multi.fa", "dos.fa", "cr_mid.fa", "noeol.fa", "blank_runs.fa"]),
    "q_mixed":     (["-m", "25", "-s", "4M", "-C", "-Q", "4"], ["multi.fa", "empty.fa", "reads_q.fq", "reads_ml.fq", "one_read.fq", "reads_q_dos.fq"]),
    "q_k40_if":    (["-m", "40", "-s", "1M", "-Q", "3", "--if", "@reads_q.fq"], ["reads_q.fq", "reads_q_dos.fq"]),
}

# Tables of 2^31 slots and more: the hash matrix has more than 30 rows, where the reference's
# random_bits() overlaps its 31-bit draws by one bit (lib/misc.cc:66-72). The reference needs
# ~7 GB and ~1.5 min for this golden (scripts/make_golden.py --big); the restatement does not
# materialise the table. Kept apart from CASES: the device table is 8 GB.
BIG_CASES = {
    "big_l31": (["-m", "21", "-s", "2G", "-C"], ["plain.fa"]),
    # the bench's own table geometry (BASELINE configs[1] after its two doublings): 2^34 slots, a 34-row
    # matrix; the reference needs 50 GB and 7 min for it, the device table is 68.7 GB of 32-bit slots
    "big_l34": (["-m", "21", "-s", "16G", "-C"], ["plain.fa"]),
    # BASELINE configs[4] geometry: k=63 (two key words, 128-bit device slots), 2^31 slots
    "big_k63_l31": (["-m", "63", "-s", "2G", "-C"], ["plain.fa"]),
    # k=31 with a 2^33-slot table (64-bit device slots; the largest k=31 table the reference fits in this container's RAM)
    "big_k31_l33": (["-m", "31", "-s", "8G", "-C"], ["plain.fa"]),
}

# --bf-size / --bf-fp: one-pass Bloom prefilter (count_main.cc:317-321, bloom_filter.hpp:40-63).
# Which first occurrences are false positives depends on the insertion ORDER, so these goldens are
# the reference with -t 1 (input order) and pin the restatement only; a device path can be held to
# count(x) in {occ(x) - 1, occ(x)} (DESIGN.md, next rows). Restatement-only for now.
BF_CASES = {
    "bf_twice":    (["-m", "21", "-s", "1M", "-C", "--bf-size", "1M"], ["plain.fa", "plain.fa"]),
    "bf_small":    (["-m", "21", "-s", "1M", "-C", "--bf-size", "300k"], ["repeat.fa", "multi.fa", "multi.fa"]),
    "bf_fp10_grow": (["-m", "17", "-s", "100k", "--bf-size", "200k", "--bf-fp", "0.1"], ["plain.fa", "multi.fa", "plain.fa"]),
    "bf_k40":      (["-m", "40", "-s", "100k", "--bf-size", "500k", "--bf-fp", "0.001"], ["plain.fa", "multi.fa", "plain.fa"]),
    "bf_fq":       (["-m", "21", "-s", "1M", "-C", "--bf-size", "100k"], ["reads.fq", "reads.fq"]),
    "bf_q":        (["-m", "17", "-s", "1M", "-C", "--bf-size", "400k", "-Q", "5"], ["reads_q.fq", "reads_q.fq", "reads_q_dos.fq"]),
    "bf_k63":      (["-m", "63", "-s", "700k", "-C", "--bf-size", "700k", "--bf-fp", "0.05"], ["plain.fa", "dos.fa", "plain.fa"]),
}

# `jellyfish bc` (bc_main.cc) then `count --bc FILE` (count_main.cc:110-120,191-206): two-pass Bloom
# counter. Both outputs are independent of insertion order and thread count (every position of the
# counter ends at min(2, hits)), so a device path can be held to these byte for byte.
# name -> (bc switches, bc inputs, count switches (--bc FILE is appended), count inputs)
BC_CASES = {
    "bc_k21C":  (["-m", "21", "-s", "400k", "-C"], ["plain.fa", "multi.fa", "plain.fa"],
                 ["-m", "21", "-s", "1M", "-C"], ["plain.fa", "multi.fa", "plain.fa"]),
    "bc_k40":   (["-m", "40", "-s", "100k", "-f", "0.05"], ["plain.fa", "dos.fa", "reads.fq"],
                 ["-m", "40", "-s", "100k"], ["plain.fa", "dos.fa", "dos.fa", "reads.fq"]),
    "bc_k63C":  (["-m", "63", "-s", "700k", "-C", "-f", "0.01"], ["plain.fa", "repeat.fa"],
                 ["-m", "63", "-s", "700k", "-C"], ["repeat.fa", "plain.fa", "plain.fa"]),
    "bc_tiny":  (["-m", "12", "-s", "20k", "-C"], ["multi.fa"],
                 ["-m", "12", "-s", "300k", "-C", "-L", "2"], ["multi.fa", "multi2.fa"]),
}

# Corners found by scripts/fuzz_oracle.py (differential fuzz of the restatement against the reference):
# tables that start with a few slots keep their CLIPPED reprobe limit through every doubling
# (hash_counter.hpp:205-209 passes ary_->max_reprobe()); counts beyond 2^val_len occupy continuation
# slots that count towards fullness; with a limit of 1 the dumper's heap cannot reorder equal positions;
# a direct-indexed table (size = 4^k) grows val_len only when a continuation entry finds no slot.
# The restatement reproduces all of these (reference run with -t 1); the device engine does not yet
# (DESIGN.md section 7a), so these stay out of CASES.
EDGE_CASES = {
    "edge_s100_k48":   (["-m", "48", "-s", "100", "-C"], ["multi.fa"]),
    "edge_s10_k54":    (["-m", "54", "-s", "10"], ["multi2.fa"]),
    "edge_s2_ties":    (["-m", "25", "-s", "2", "-C"], ["dangling.fa", "cr_mid.fa", "one_read.fq"]),
    "edge_s2_k31_p62": (["-m", "31", "-s", "2", "-C", "-p", "62"], ["multi2.fa"]),
    "edge_direct_sparse": (["-m", "4", "-s", "100k", "-C"], ["polya.fa", "dangling.fa"]),
    "edge_c1_p2":      (["-m", "17", "-s", "10", "-C", "-c", "1", "-p", "2"], ["repeat.fa", "multi2.fa"]),
    "edge_k5_s10_c1":  (["-m", "5", "-s", "10", "-c", "1"], ["multi.fa", "polya.fa"]),
    "edge_k5_s2_p10":  (["-m", "5", "-s", "2", "-C", "-p", "10"], ["repeat.fa", "polya.fa"]),
    "edge_rep_c2":     (["-m", "21", "-s", "2k", "-C", "-c", "2"], ["repeat.fa", "polya.fa", "multi2.fa"]),
}

# --disk (count_main.cc:277,346-371; hash_counter.hpp:187-192): no size doubling -- a full table is written to an
# intermediate file and zeroed, the files are merged at the end.  The merged database keeps the ORIGINAL size and matrix,
# so its body does not depend on when the table filled up.
DISK_CASES = {
    "disk_k40":    (["-m", "40", "-s", "50k", "--disk", "-C"], ["plain.fa"]),
    "disk_k21_LU": (["-m", "21", "-s", "100k", "--disk", "-C", "-L", "2"], ["plain.fa", "multi.fa", "plain.fa"]),
    "disk_k17_c3": (["-m", "17", "-s", "30k", "--disk", "-c", "3", "--out-counter-len", "2"], ["multi.fa", "multi2.fa"]),
}

# The host-side readers (dump, histo, stats) against the reference's on one database (test_host.py), and the merges
# (merge_main.cc:31-37, merge_files.cc:45-176) of test_host.py::test_merge_matches_reference: name -> count switches and inputs
# of the merged databases; (tag, merge switches, databases) of every merge; the --disk run whose intermediate files the
# reference wrote (tests/golden/disk_parts/).  The reference's answers: tests/golden/golden_tools.json.
READER_COMMANDS = (["dump", "-c"], ["dump"], ["dump", "-c", "-t", "-L", "2", "-U", "50"], ["histo"], ["histo", "-l", "2", "-h", "20", "-i", "3", "-f"],
                   ["stats"], ["stats", "-L", "2"])
MERGE_COUNTS = (("a", ["-m", "17", "-s", "1M", "-C"], ["multi.fa"]),
                ("b", ["-m", "17", "-s", "1M", "-C"], ["multi2.fa"]),
                ("c", ["-m", "17", "-s", "1M", "-C"], ["multi.fa", "dangling.fa"]),
                ("ta", ["-m", "17", "-s", "1M", "-C", "--text"], ["multi.fa"]),
                ("tb", ["-m", "17", "-s", "1M", "-C", "--text"], ["multi2.fa", "dangling.fa"]))
MERGE_OPS = (("sum", [], ["a", "b"]), ("min", ["--min"], ["a", "c"]), ("min0", ["-m", "-L", "0"], ["a", "b"]), ("max", ["--max"], ["a", "b", "c"]),
             ("maxLU", ["-M", "-L", "2", "-U", "3"], ["a", "c"]), ("sum3", ["-L", "2"], ["a", "b", "c"]), ("min3", ["-m"], ["c", "a", "c"]),
             ("jaccard_ac", ["--jaccard"], ["a", "c"]), ("jaccard_ab", ["--jaccard"], ["a", "b"]), ("jaccard_abc", ["--jaccard"], ["a", "b", "c"]),
             ("tsum", [], ["ta", "tb"]), ("tmin", ["-m"], ["ta", "tb"]), ("tmaxL", ["-M", "-L", "2"], ["ta", "tb"]))
DISK_PARTS_COUNT = (["-m", "21", "-s", "1k", "-C", "--disk", "--no-merge", "-t", "2"], "dangling.fa")
