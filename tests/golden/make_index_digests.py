"""Records what the UNMODIFIED reference binary's `chromap -i` writes, for the tests that compare the index this project builds
with it without running the reference binary: the file's header and length, the digests of tests/util.index_digest and a seeded
sample of (key, value) pairs.  Needs oracle/_ref/chromap (oracle/Makefile); called by make_golden.sh.  Outputs are committed:
  synth_small/ref_index.json   the index of synth_small/ref.fa.gz
  planted_20mbp_index.json     the index of tests/util.planted_repeat_reference() (20 Mbp, written as a FASTA first)
"""
import gzip
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import oracle_py as orc  # noqa: E402
from tests.util import index_digest, planted_repeat_reference, write_fasta  # noqa: E402

REF_BIN = os.path.join(ROOT, "oracle", "_ref", "chromap")


def describe(fasta, work):
    idx = os.path.join(work, "ref.index")
    subprocess.run([REF_BIN, "-i", "-r", fasta, "-o", idx], check=True, capture_output=True)
    raw = open(idx, "rb").read()
    a = orc.Index(idx).arrays()
    out = dict(header=[int(x) for x in np.frombuffer(raw[:8], "<i4")] + [int(x) for x in np.frombuffer(raw[8:28], "<u4")],
               file_bytes=len(raw), **index_digest(a))
    b = np.arange(a["n_buckets"])
    occupied = np.nonzero(((a["flags"][b >> 4] >> ((b & 15) << 1)) & 3) == 0)[0]
    pick = np.sort(np.random.default_rng(7).choice(occupied, size=min(256, len(occupied)), replace=False))
    out["sample_keys"] = [int(x) for x in a["keys"][pick]]
    out["sample_vals"] = [int(x) for x in a["vals"][pick]]
    return out


def main():
    with tempfile.TemporaryDirectory() as work:
        fa = os.path.join(work, "synth_small.fa")
        open(fa, "wb").write(gzip.open(os.path.join(HERE, "synth_small", "ref.fa.gz")).read())
        with open(os.path.join(HERE, "synth_small", "ref_index.json"), "w") as f:
            json.dump(describe(fa, work), f, indent=1)
            f.write("\n")
        names, seqs = planted_repeat_reference()
        fa = os.path.join(work, "planted.fa")
        write_fasta(fa, names, seqs)
        d = describe(fa, work)
        d["fasta_sha256"] = hashlib.sha256(open(fa, "rb").read()).hexdigest()
        with open(os.path.join(HERE, "planted_20mbp_index.json"), "w") as f:
            json.dump(d, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
