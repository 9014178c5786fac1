"""Deterministic test inputs (pure Python, independent of any binary)."""
import os
import random


_QUAD = [bytes(b"ACGT"[(v >> (2 * j)) & 3] for j in range(4)) for v in range(256)]


def _seq(n, seed):
    """n iid bases; base i = bits (2i, 2i+1) of one big random integer (linear time: the integer is
    turned into little-endian bytes, every byte yields 4 bases)."""
    rng = random.Random(seed)
    bits = rng.getrandbits(2 * n)
    raw = bits.to_bytes((2 * n + 7) // 8, "little")
    return b"".join(_QUAD[v] for v in raw)[:n]


def fasta(seq, line=70, name=b"read1", eol=b"\n"):
    out = [b">" + name + eol]
    for i in range(0, len(seq), line):
        out.append(seq[i:i + line] + eol)
    return b"".join(out)


def generate_sequence(prefix, seed, *lengths):
    """The FASTA files of the reference's `generate_sequence -o PREFIX -s SEED LEN...`, byte for byte: one MT19937 stream
    (seeded as init_genrand, its first 37 words skipped), 16 bases per 32-bit word from the low bits up (A, C, G, T), one
    record '>read1' in 70-column lines followed by an empty record '>read2'.  Several lengths -> PREFIX_0.fa, PREFIX_1.fa, ...
    from the same stream, each file starting on a fresh word.  -> list of paths."""
    import numpy as np
    rs = np.random.RandomState(seed & 0xFFFFFFFF)
    rs.randint(0, 1 << 32, size=37, dtype=np.uint64)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    paths = []
    for i, n in enumerate(lengths):
        path = "%s_%d.fa" % (prefix, i) if len(lengths) > 1 else prefix + ".fa"
        words = rs.randint(0, 1 << 32, size=(n + 15) // 16, dtype=np.uint64).astype(np.uint32)
        shifts = np.arange(0, 32, 2, dtype=np.uint32)
        seq = lut[((words[:, None] >> shifts) & 3).reshape(-1)[:n]]
        full = n // 70
        with open(path, "wb") as f:
            f.write(b">read1\n")
            body = np.empty((full, 71), dtype=np.uint8)
            body[:, :70] = seq[:full * 70].reshape(-1, 70)
            body[:, 70] = 10
            f.write(body.tobytes())
            if n > full * 70:
                f.write(seq[full * 70:].tobytes() + b"\n")
            if n:
                f.write(b">read2\n")
        paths.append(path)
    return paths


def make_all(d):
    """-> dict name -> path.  Sizes are small so that the CPU reference runs in seconds."""
    f = {}

    def w(name, data):
        p = os.path.join(d, name)
        with open(p, "wb") as fh:
            fh.write(data)
        f[name] = p
        return p

    s300 = _seq(300000, 1)
    w("plain.fa", fasta(s300))
    w("dos.fa", fasta(s300, eol=b"\r\n"))
    w("noeol.fa", fasta(s300)[:-1])
    w("lower.fa", fasta(s300.lower()))
    # several records, some short, N's and IUPAC codes, blank lines, '>' inside a line, spaces
    rng = random.Random(7)
    recs = []
    for i in range(200):
        s = bytearray(_seq(rng.randrange(1, 3000), 100 + i))
        for _ in range(rng.randrange(0, 4)):
            s[rng.randrange(len(s))] = rng.choice(b"NnRYKMSWBDHVU-. >\t")
        body = fasta(bytes(s), line=rng.choice([1, 7, 60, 70, 200]), name=b"r%d some description" % i)
        if rng.random() < 0.3:
            body = body.replace(b"\n", b"\n\n", 2)
        recs.append(body)
    w("multi.fa", b"".join(recs))
    w("multi2.fa", b"".join(reversed(recs[:50])))
    w("empty.fa", b"")
    w("header_only.fa", b">just a header\n")
    w("dangling.fa", fasta(_seq(5000, 3)) + b">read2\n")
    # pathological line structure: one base per line, runs of blank lines, very long header
    s2 = _seq(20000, 5)
    w("one_per_line.fa", fasta(s2, line=1))
    w("blank_runs.fa", b">x\n" + b"".join(s2[i:i + 50] + b"\n" * (1 + (i // 50) % 400) for i in range(0, 5000, 50)))
    w("long_header.fa", b">" + b"h" * 70000 + b"\n" + s2[:3000] + b"\n>" + b"ACGT" * 300 + b"\n" + s2[3000:6000] + b"\n")
    w("cr_mid.fa", b">x\nACGTACGTAC\rGTACGTTGCA\r\r\nACGTAGCTAGCTAGCTAGGGATCGATCGACTAGCTA\r\n\r\nACGATCGATCGTTTAGC\r")
    w("oneline.fa", b">x\n" + _seq(100000, 9) + b"\n")
    # repetitive: counts far beyond 2^val_len
    w("polya.fa", fasta(b"A" * 100000))
    w("repeat.fa", fasta(_seq(500, 11) * 400))
    w("plain1m.fa", fasta(_seq(1000000, 2)))
    # FASTQ (4-line records): ragged read lengths, N's and lower case, quality strings that begin
    # with '@' or '+', DOS line ends, a missing final newline, reads longer than a device tile
    rng = random.Random(11)

    def fastq(n_reads, seed, eol=b"\n", lens=(36, 76, 101, 150, 151, 250), long_read=0, final_eol=True):
        r = random.Random(seed)
        out = []
        for i in range(n_reads):
            ln = long_read if (long_read and i % 7 == 3) else r.choice(lens)
            sq = bytearray(_seq(ln, seed * 100003 + i))
            for _ in range(r.randrange(0, 3)):
                sq[r.randrange(ln)] = r.choice(b"NnRacgt")
            q = bytearray(r.randrange(33, 75) for _ in range(ln))
            if i % 5 == 0:
                q[0] = ord("@")
            if i % 5 == 1:
                q[0] = ord("+")
            out.append(b"@read_%d/1 len=%d" % (i, ln) + eol + bytes(sq) + eol + (b"+" if i % 2 else b"+read_%d/1" % i) + eol + bytes(q) + eol)
        data = b"".join(out)
        return data if final_eol else data[:-len(eol)]

    w("reads.fq", fastq(3000, 21))
    w("reads_dos.fq", fastq(1500, 22, eol=b"\r\n"))
    w("reads_noeol.fq", fastq(1500, 23, final_eol=False))
    w("reads_long.fq", fastq(40, 24, long_read=40000))
    w("one_read.fq", b"@r\nACGTACGTACGTACGTTTGCAAGCATCGAT\n+\nIIIIIIIIIIIIIIIIIIIIIIIIIIIIII\n")
    # multi-line FASTQ (sequence and qualities wrapped at 60), an empty read, no final newline
    r = random.Random(31)
    ml = []
    for i in range(400):
        ln = r.choice((0, 59, 60, 61, 150, 400)) if i % 50 == 7 else r.choice((59, 60, 61, 150, 400))
        sq = _seq(ln, 777000 + i) if ln else b""
        q = bytes(r.randrange(35, 74) for _ in range(ln))
        wrap = lambda x: b"".join(x[j:j + 60] + b"\n" for j in range(0, len(x), 60)) if x else b"\n"
        ml.append(b"@ml_%d\n" % i + wrap(sq) + b"+\n" + wrap(q))
    w("reads_ml.fq", b"".join(ml)[:-1])

    # realistic qualities for -Q: mostly high, ~4% low bases, low tails, a few bytes >= 0x80
    # (negative as a char: always below the threshold)
    def fastq_q(n_reads, seed, eol=b"\n"):
        r = random.Random(seed)
        out = []
        for i in range(n_reads):
            ln = r.choice((50, 76, 101, 151))
            sq = bytearray(_seq(ln, seed * 7919 + i))
            if i % 9 == 0:
                sq[r.randrange(ln)] = ord("N")
            q = bytearray(r.choice(b"FGHIIIIJ") if r.random() > 0.04 else r.randrange(33, 60) for _ in range(ln))
            tail = r.randrange(0, 12)
            for j in range(ln - tail, ln):
                q[j] = r.randrange(33, 45)
            if i % 37 == 5:
                q[r.randrange(ln)] = r.randrange(128, 256)
            out.append(b"@q%d" % i + eol + bytes(sq) + eol + b"+" + eol + bytes(q) + eol)
        return b"".join(out)

    w("reads_q.fq", fastq_q(3000, 41))
    w("reads_q_dos.fq", fastq_q(1000, 42, eol=b"\r\n"))
    return f
