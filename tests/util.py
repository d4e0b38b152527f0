"""Test helpers: tiny FASTA/FASTQ readers (gz-aware) and batch packing."""
import gzip
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _open(p):
    return gzip.open(p, "rb") if p.endswith(".gz") else open(p, "rb")


def read_fasta(path):
    names, seqs, cur = [], [], []
    with _open(path) as f:
        for line in f:
            line = line.rstrip(b"\r\n")
            if line.startswith(b">"):
                if names:
                    seqs.append(np.frombuffer(b"".join(cur), dtype=np.uint8))
                names.append(line[1:].split()[0].decode())
                cur = []
            else:
                cur.append(line)
    seqs.append(np.frombuffer(b"".join(cur), dtype=np.uint8))
    return names, seqs


def read_fastq(path):
    seqs = []
    with _open(path) as f:
        for i, line in enumerate(f):
            if i % 4 == 1:
                seqs.append(line.rstrip(b"\r\n"))
    return seqs


def read_fastq_records(path):
    """[(name, sequence, quality)] of a 4-line FASTQ; name = header up to the first whitespace (kseq)."""
    out = []
    with _open(path) as f:
        lines = [l.rstrip(b"\r\n") for l in f]
    for i in range(0, len(lines) - 3, 4):
        out.append((lines[i][1:].split()[0] if lines[i][1:].split() else b"", lines[i + 1], lines[i + 3]))
    return out


def pack(reads):
    off = np.zeros(len(reads) + 1, dtype=np.uint32)
    off[1:] = np.cumsum([len(r) for r in reads])
    return np.frombuffer(b"".join(reads), dtype=np.uint8), off


def load_pairs(d, r1="read1.fq.gz", r2="read2.fq.gz"):
    a, b = read_fastq(os.path.join(d, r1)), read_fastq(os.path.join(d, r2))
    s1, o1 = pack(a)
    s2, o2 = pack(b)
    return s1, o1, s2, o2


def planted_repeat_reference():
    """4 x 5 Mbp of random bases (seed 3) with planted 5 kb segmental repeats, a 300 bp family and N runs: (names, seqs)."""
    rng = np.random.default_rng(3)
    seqs = []
    fam = rng.integers(0, 4, 300)
    for si in range(4):
        s = rng.integers(0, 4, 5000000)
        seg = rng.integers(0, 4, 5000)
        for st in rng.integers(0, len(s) - 5000, 30):
            s[st:st + 5000] = seg
        for st in rng.integers(0, len(s) - 300, 800):
            s[st:st + 300] = fam
        a = np.frombuffer(b"ACGT", dtype=np.uint8)[s].copy()
        for st in rng.integers(0, len(a) - 200, 40):
            a[st:st + int(rng.integers(1, 200))] = ord("N")
        seqs.append(a)
    return ["s%d" % i for i in range(len(seqs))], seqs


def write_fasta(path, names, seqs):
    with open(path, "wb") as f:
        for n, a in zip(names, seqs):
            f.write(b">%s\n" % n.encode()); a.tofile(f); f.write(b"\n")


def index_digest(a):
    """What an index (n_buckets / flags / keys / vals / occ arrays in khash's layout) holds, independent of the bucket order
    inside khash's arrays (a function of its resize history, not of the content): the bucket count, the key -> value map and the
    occurrence table, each as a sha256 with its size."""
    import hashlib
    nb = int(a["n_buckets"])
    b = np.arange(nb)
    occupied = ((a["flags"][b >> 4] >> ((b & 15) << 1)) & 3) == 0
    keys, vals = a["keys"][occupied].astype("<u8"), a["vals"][occupied].astype("<u8")
    o = np.argsort(keys)
    return dict(n_buckets=nb, n_keys=int(len(keys)), n_occ=int(len(a["occ"])),
                keys_vals_sha256=hashlib.sha256(keys[o].tobytes() + vals[o].tobytes()).hexdigest(),
                occ_sha256=hashlib.sha256(np.ascontiguousarray(a["occ"], dtype="<u8").tobytes()).hexdigest())
