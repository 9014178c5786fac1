"""Helpers shared by the tests: locate binaries, run them, split jellyfish databases."""
import json
import os
import subprocess
import hashlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
REF_JF = os.path.join(REF_DIR, "jellyfish")            # the unmodified reference, built by oracle/Makefile
REF_GEN = os.path.join(REF_DIR, "generate_sequence")
ORACLE_C = os.path.join(REF_DIR, "jf_oracle")          # the independent C restatement
OUR_JF = os.path.join(ROOT, "jellyfish_b200", "lib", "jellyfish-b200")
LIB = os.path.join(ROOT, "jellyfish_b200", "lib", "libjfgpu.so")

SEMANTIC_KEYS = ("size", "key_len", "val_len", "max_reprobe", "reprobes", "counter_len", "format",
                 "canonical", "matrix1", "alignment")


def run(cmd, **kw):
    env = dict(os.environ, SOURCE_DATE_EPOCH="0")
    env.update(kw.pop("env", {}))
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env, **kw)
    if r.returncode != 0:
        raise RuntimeError("command failed (%d): %s\nstdout: %s\nstderr: %s" % (
            r.returncode, " ".join(map(str, cmd)), r.stdout.decode(errors="replace")[-2000:],
            r.stderr.decode(errors="replace")[-2000:]))
    return r


def split_db(path):
    """-> (header dict, body bytes) of a jellyfish database."""
    with open(path, "rb") as f:
        data = f.read()
    hlen = int(data[:9])
    raw = data[9:9 + hlen].rstrip(b"\0")
    return json.loads(raw.decode()), data[9 + hlen:]


def semantic(header):
    return {k: header.get(k) for k in SEMANTIC_KEYS}


def md5(b):
    return hashlib.md5(b).hexdigest()


def records(header, body):
    """-> list of (key int, count int)"""
    kb = (header["key_len"] + 7) // 8
    cl = header["counter_len"]
    rec = kb + cl
    out = []
    for i in range(0, len(body) - rec + 1, rec):
        out.append((int.from_bytes(body[i:i + kb], "little"), int.from_bytes(body[i + kb:i + rec], "little")))
    return out


def generate(prefix, seed, *lengths):
    """The files of the reference's `generate_sequence -o PREFIX -s SEED LEN...` (restated in tests/gen.py)."""
    import gen
    return gen.generate_sequence(prefix, seed, *lengths)


def golden(name):
    with open(os.path.join(ROOT, "tests", "golden", name)) as f:
        return json.load(f)


def db_digest(path):
    """What a comparison of two databases looks at: the semantic header keys and the record body."""
    h, b = split_db(path)
    return {"header": semantic(h), "body_md5": md5(b), "body_len": len(b)}


def semantic_md5(header):
    """Digest of the semantic header keys (stored in place of the keys where a golden file holds many headers)."""
    return md5(json.dumps(semantic(header), sort_keys=True).encode())


def records_md5(recs):
    """Digest of a set of (key, count) records, independent of their order in the file."""
    return md5(json.dumps(sorted(recs)).encode())


class RefLog(object):
    """The answers of the reference binary, in the order they were asked for.  live: ask the binary; record: ask it and keep
    the answers in `path`; replay: read them back from `path` (a golden file), so that a comparison with the reference runs
    where the reference does not.  `what` names the question (paths relative to the run's directory); a replayed answer to
    another question means the golden file no longer matches the cases and raises."""

    def __init__(self, path=None, mode="live"):
        assert mode in ("live", "record", "replay")
        self.path, self.mode, self.i = path, mode, 0
        self.items = json.load(open(path)) if mode == "replay" else []

    def answer(self, what, ask):
        if self.mode != "replay":
            v = ask()
            if self.mode == "record":
                self.items.append([what, v])
            return v
        if self.i >= len(self.items) or self.items[self.i][0] != what:
            raise RuntimeError("%s out of step at answer %d: golden %r, asked %r" % (
                self.path, self.i, self.items[self.i][0] if self.i < len(self.items) else None, what))
        self.i += 1
        return self.items[self.i - 1][1]

    def close(self):
        if self.mode == "record":
            with open(self.path, "w") as f:
                json.dump(self.items, f, separators=(",", ":"))
                f.write("\n")
        elif self.mode == "replay" and self.i != len(self.items):
            raise RuntimeError("%s: %d answers recorded, %d asked for" % (self.path, len(self.items), self.i))


def subst(args, files):
    """'@name' in a case's switches stands for the path of that generated input (e.g. --if @multi2.fa)."""
    return [files[a[1:]] if a.startswith("@") else a for a in args]


def hash_pos(header, key):
    """Original position of a key: RectangularBinaryMatrix::times (bit i of the key selects columns[c-1-i],
    rectangular_binary_matrix.hpp:223-261) modulo the table size."""
    m = header["matrix1"]
    size = header["size"]
    if m.get("identity"):
        return key & (size - 1)
    cols, c = m["columns"], m["c"]
    h, i = 0, 0
    while key:
        if key & 1:
            h ^= cols[c - 1 - i]
        key >>= 1
        i += 1
    return h & (size - 1)
