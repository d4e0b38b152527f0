"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle and the golden vectors made by
the reference binary.  Run with `-m gpu` on the B200 box."""
import gzip
import os

import numpy as np
import pytest

import chromap_b200 as cb
from oracle import oracle_py as orc
import ctypes as C

from tests.util import load_pairs, read_fasta, read_fastq_records

pytestmark = pytest.mark.gpu


def assert_same_records(a, b):
    """Field-wise equality (the 2 padding bytes of the 24-byte record are not part of the contract)."""
    assert len(a) == len(b)
    for f in a.dtype.names:
        bad = np.nonzero(a[f] != b[f])[0]
        assert len(bad) == 0, (f, bad[:5], a[bad[:5]], b[bad[:5]])

CASES = {
    "chip": dict(preset="chip"),
    "atac": dict(preset="atac"),
    "default": dict(preset=""),
    "q0dedup": dict(preset="", remove_pcr_duplicates=1, mapq_threshold=0),
    "e5": dict(preset="", error_threshold=5, mapq_threshold=10, tn5_shift=1, remove_pcr_duplicates=1),
    "e12l300": dict(preset="", error_threshold=12, max_insert_size=300, mapq_threshold=0),
    "n3q0": dict(preset="", max_num_best_mappings=3, mapq_threshold=0),
}


@pytest.fixture(scope="module")
def synth(golden_dir):
    d = os.path.join(golden_dir, "synth_small")
    names, seqs = read_fasta(os.path.join(d, "ref.fa.gz"))
    oref = orc.Reference(os.path.join(d, "ref.fa.gz"))
    oidx = orc.Index(ref=oref, k=17, w=7)
    return dict(d=d, names=names, seqs=seqs, oref=oref, oidx=oidx, pairs=load_pairs(d))


def _mapper(synth, kw, build_on_device=False):
    kw = dict(kw)
    p = cb.make_params(kw.pop("preset"), max_read_length=64, **kw)
    m = cb.Mapper(p)
    m.upload_reference(synth["seqs"], synth["names"])
    if build_on_device:
        m.build_index(17, 7)
    else:
        a = synth["oidx"].arrays()
        m.upload_index(17, 7, a["n_buckets"], a["flags"], a["keys"], a["vals"], a["occ"])
    return m


def _oparams(kw):
    kw = dict(kw)
    return orc.make_params(kw.pop("preset"), **kw)


def test_stage_minimizers_equal_oracle(synth):
    m = _mapper(synth, CASES["default"])
    s1, o1, s2, o2 = synth["pairs"]
    n = 1500
    h, p, cnt = m.stage_minimizers(s1[:o1[n]], o1[:n + 1], s2[:o2[n]], o2[:n + 1], 64)
    for i in range(n):
        for mate, (s, o) in enumerate(((s1, o1), (s2, o2))):
            oh, ot = orc.minimizers(s[o[i]:o[i + 1]], 17, 7)
            r = 2 * i + mate
            assert cnt[r] == len(oh)
            assert np.array_equal(h[r, :cnt[r]], oh)
            assert np.array_equal(p[r, :cnt[r]].astype(np.uint64), ot & np.uint64(0xFFFFFFFF))


@pytest.mark.parametrize("k,w", [(19, 10), (23, 11), (15, 5), (28, 20)])
def test_stage_minimizers_other_k_w(synth, k, w):
    p = cb.make_params("", max_read_length=64)
    m = cb.Mapper(p)
    m.upload_reference([synth["seqs"][0][:50000]], ["chr1"])
    m.build_index(k, w)
    s1, o1, s2, o2 = synth["pairs"]
    n = 400
    h, pos, cnt = m.stage_minimizers(s1[:o1[n]], o1[:n + 1], s2[:o2[n]], o2[:n + 1], 64)
    for i in range(n):
        for mate, (s, o) in enumerate(((s1, o1), (s2, o2))):
            oh, ot = orc.minimizers(s[o[i]:o[i + 1]], k, w)
            r = 2 * i + mate
            assert cnt[r] == len(oh)
            assert np.array_equal(h[r, :cnt[r]], oh)
            assert np.array_equal(pos[r, :cnt[r]].astype(np.uint64), ot & np.uint64(0xFFFFFFFF))
    # the device index builder uses the same generator on reference chunks: compare with the oracle's index
    oref = orc.Reference(seqs=[synth["seqs"][0][:50000]])
    oidx = orc.Index(ref=oref, k=k, w=w)
    assert np.array_equal(m.download_index()["occ"], oidx.arrays()["occ"])
    assert m.index_info()["n_keys"] == int((((oidx.arrays()["flags"][np.arange(oidx.arrays()["n_buckets"]) >> 4] >> ((np.arange(oidx.arrays()["n_buckets"]) & 15) << 1)) & 3) == 0).sum())


def test_stage_probe_equals_khash_lookup(synth):
    import ctypes as C
    m = _mapper(synth, CASES["default"])
    rng = np.random.default_rng(5)
    hs = [orc.minimizers(synth["seqs"][0][:200000], 17, 7)[0][::3]]
    hs.append(rng.integers(0, 1 << 34, 5000, dtype=np.uint64))  # mostly absent
    hashes = np.concatenate(hs)
    f, k, v = m.stage_probe(hashes)
    L = orc.lib()
    for i in range(0, len(hashes), 5):
        kk, vv = C.c_uint64(), C.c_uint64()
        found = L.orc_index_lookup(synth["oidx"].h, int(hashes[i]), C.byref(kk), C.byref(vv))
        assert found == f[i]
        if found:
            assert (kk.value, vv.value) == (int(k[i]), int(v[i]))


@pytest.mark.parametrize("e,L", [(8, 50), (4, 150), (15, 36), (1, 30)])
def test_stage_banded_align_equals_oracle(synth, e, L):
    import ctypes as C
    m = _mapper(synth, CASES["default"])
    rng = np.random.default_rng(e * 1000 + L)
    n = 3000
    acgt = np.frombuffer(b"ACGTN", dtype=np.uint8)
    pats = acgt[rng.integers(0, 4, (n, L + 2 * e))].copy()
    texts = np.zeros((n, L), dtype=np.uint8)
    for i in range(n):  # read = window shifted by up to +-e, with substitutions / an indel
        sh = int(rng.integers(0, 2 * e + 1))
        t = pats[i, sh:sh + L].copy()
        if len(t) < L:
            t = np.concatenate([t, acgt[rng.integers(0, 4, L - len(t))]])
        nsub = int(rng.integers(0, e + 3))
        t[rng.integers(0, L, nsub)] = acgt[rng.integers(0, 5, nsub)]
        if rng.random() < 0.3:
            p = int(rng.integers(1, L - 1))
            t = np.concatenate([t[:p], t[p + 1:], acgt[rng.integers(0, 4, 1)]])
        texts[i] = t
    err, endp = m.stage_banded_align(e, L, pats, texts)
    Lb = orc.lib()
    for i in range(n):
        ep = C.c_int(0)
        oe = Lb.orc_banded_align(e, pats[i].ctypes.data, texts[i].ctypes.data, L, C.byref(ep))
        assert oe == err[i]
        if oe <= e:
            assert ep.value == endp[i]


@pytest.mark.parametrize("n,cap", [(1, 64), (2, 64), (63, 64), (64, 64), (65, 64), (1000, 256), (4096, 4096), (4097, 4096), (20000, 1024), (65536, 4096), (50001, 2048)])
def test_cta_sort_matches_numpy(n, cap):
    m = cb.Mapper(cb.make_params("", max_read_length=64))
    rng = np.random.default_rng(n)
    keys = rng.integers(0, 1 << 62, n, dtype=np.uint64)
    keys[rng.integers(0, n, n // 3)] = keys[0]  # duplicates
    got, _ = m.stage_cta_sort(keys, sm_cap=cap)
    assert np.array_equal(got, np.sort(keys))
    tags = rng.integers(1, 6, n).astype(np.uint8)
    gk, gt = m.stage_cta_sort(keys, tags, sm_cap=cap)
    order = np.lexsort((keys, 255 - tags.astype(np.int64)))  # count descending, then position ascending
    assert np.array_equal(gk, keys[order]) and np.array_equal(gt, tags[order])


@pytest.mark.parametrize("case", sorted(CASES))
def test_map_batch_records_equal_oracle_and_golden(synth, case):
    kw = CASES[case]
    m = _mapper(synth, kw)
    s1, o1, s2, o2 = synth["pairs"]
    recs, stats = m.map_batch(s1, o1, s2, o2)
    orecs, otrace = orc.map_pairs(_oparams(kw), synth["oidx"], synth["oref"], s1, o1, s2, o2, trace=True)
    tr = m.trace(len(o1) - 1)
    def same(f, mask):
        a, b = tr[f][mask], otrace[f][mask]
        if not np.array_equal(a, b):
            bad = np.nonzero(np.any(np.atleast_2d((a != b).T).T.reshape(len(a), -1), axis=1))[0][:5]
            raise AssertionError("%s differs at pairs %s: gpu %s oracle %s" % (f, np.nonzero(mask)[0][bad], a[bad], b[bad]))
    both = (otrace["n_minimizers"] > 0).all(axis=1)
    same("n_minimizers", both)
    for f in ("trimmed_len", "n_pos_candidates_gen", "n_neg_candidates_gen", "supplement_result"):
        same(f, both)
    alive = otrace["n_records"] > 0
    for f in ("n_pos_candidates", "n_neg_candidates", "n_pos_mappings", "n_neg_mappings", "min_errors", "n_best",
              "min_sum_errors", "n_best_pairs", "n_second_best_pairs", "repetitive_seed_length", "trimmed_len"):
        same(f, alive)
    assert len(recs) == len(orecs)
    assert_same_records(recs, orecs)
    assert stats["n_overflow_pairs"] == 0
    bed = m.format_bed(m.postprocess(recs))
    want = gzip.open(os.path.join(synth["d"], case + ".bed.gz")).read()
    assert bed == want


def test_pipelined_host_batches_equal_per_batch_oracle(synth):
    """Host buffers spanning several reference batches take the copy/compute-overlapped path; every reference
    batch restarts the taskloop chunking, exactly like consecutive batches of the reference."""
    kw = dict(preset="", remove_pcr_duplicates=1, mapq_threshold=0)
    p = cb.make_params(kw["preset"], max_read_length=64, batch_size=1700, remove_pcr_duplicates=1, mapq_threshold=0)
    m = cb.Mapper(p)
    m.upload_reference(synth["seqs"], synth["names"])
    a = synth["oidx"].arrays()
    m.upload_index(17, 7, a["n_buckets"], a["flags"], a["keys"], a["vals"], a["occ"])
    s1, o1, s2, o2 = synth["pairs"]
    n = len(o1) - 1
    recs, stats = m.map_batch(s1, o1, s2, o2, first_read_id=100)
    want = []
    op = _oparams(kw)
    for b0 in range(0, n, 1700):
        b1 = min(n, b0 + 1700)
        r, _ = orc.map_pairs(op, synth["oidx"], synth["oref"], s1[o1[b0]:o1[b1]], o1[b0:b1 + 1] - o1[b0], s2[o2[b0]:o2[b1]], o2[b0:b1 + 1] - o2[b0],
                             first_read_id=100 + b0)
        want.append(r)
    want = np.concatenate(want)
    assert len(recs) == len(want)
    assert_same_records(recs, want)


def test_index_built_on_device_equals_reference_semantics(synth):
    m = _mapper(synth, CASES["default"], build_on_device=True)
    a = synth["oidx"].arrays()
    info = m.index_info()
    assert info["n_occ"] == len(a["occ"])
    d = m.download_index()
    assert np.array_equal(d["occ"], a["occ"])
    assert d["n_buckets"] == a["n_buckets"] and d["n_keys"] == info["n_keys"]
    # every key of the oracle's table is found with the same value, and nothing else is present
    occupied = ((a["flags"][np.arange(a["n_buckets"]) >> 4] >> ((np.arange(a["n_buckets"]) & 15) << 1)) & 3) == 0
    keys, vals = a["keys"][occupied], a["vals"][occupied]
    assert len(keys) == info["n_keys"]
    f, k, v = m.stage_probe(keys >> np.uint64(1))
    assert f.all() and np.array_equal(k, keys) and np.array_equal(v, vals)
    # and mapping through the device-built index gives the golden BED
    s1, o1, s2, o2 = synth["pairs"]
    recs, _ = m.map_batch(s1, o1, s2, o2)
    bed = m.format_bed(m.postprocess(recs))
    assert bed == gzip.open(os.path.join(synth["d"], "default.bed.gz")).read()


def test_device_built_index_has_the_content_of_the_reference_binarys_index(tmp_path, golden_dir):
    """`chromap -i` (the unmodified reference binary) and cmx_build_index on the same 20 Mbp reference with planted repeats and
    N runs: same k / w, same bucket count, the SAME occurrence table byte for byte, and the same key -> value map (no other key),
    every key found by the device's probe with its value.  The reference binary's side is stored as digests plus a sample of its
    (key, value) pairs (tests/golden/planted_20mbp_index.json, written by tests/golden/make_index_digests.py).  Only the bucket
    ORDER inside khash's arrays is not compared: it is a function of khash's resize history (kh_resize re-inserts in bucket
    order), not of the content; lookups do not depend on it.  This is what lets bench.py's reference arm run on an index
    written by cmx_download_index."""
    import hashlib
    import json
    from tests.util import index_digest, planted_repeat_reference, write_fasta
    want = json.load(open(os.path.join(golden_dir, "planted_20mbp_index.json")))
    names, seqs = planted_repeat_reference()
    fa = tmp_path / "ref.fa"
    write_fasta(fa, names, seqs)
    assert hashlib.sha256(fa.read_bytes()).hexdigest() == want["fasta_sha256"], "not the reference the digests were made from"
    k_mer, window = want["header"][:2]
    m = cb.Mapper(cb.make_params("", max_read_length=64))
    m.upload_reference(seqs, names)
    m.build_index(k_mer, window)
    info = m.index_info()
    d = m.download_index()
    got = index_digest(d)
    assert got == {f: want[f] for f in got}
    assert info["n_occ"] == want["n_occ"] and info["n_keys"] == d["n_keys"] == want["n_keys"]
    sk, sv = np.array(want["sample_keys"], dtype=np.uint64), np.array(want["sample_vals"], dtype=np.uint64)
    f, k, v = m.stage_probe(sk >> np.uint64(1))
    assert f.all() and np.array_equal(k, sk) and np.array_equal(v, sv)
    nb = d["n_buckets"]
    occ_d = ((d["flags"][np.arange(nb) >> 4] >> ((np.arange(nb) & 15) << 1)) & 3) == 0
    keys, vals = d["keys"][occ_d], d["vals"][occ_d]
    f, k, v = m.stage_probe(keys >> np.uint64(1))
    assert f.all() and np.array_equal(k, keys) and np.array_equal(v, vals)


def test_reference_quickstart_golden(golden_dir):
    """BASELINE config 1 (reference test/ data): md5 e311f0a0… / 63b977e6…"""
    import hashlib
    d = os.path.join(golden_dir, "ref_test")
    names, seqs = read_fasta(os.path.join(d, "ref.fa.gz"))
    oidx = orc.Index(os.path.join(d, "ref.index"))  # the index file the reference binary wrote
    a = oidx.arrays()
    s1, o1, s2, o2 = load_pairs(d, "read1.fq", "read2.fq")
    for preset, md5 in (("", "e311f0a0848edca7196d839f47b3e007"), ("chip", "e311f0a0848edca7196d839f47b3e007"),
                        ("atac", "63b977e6e8af35be7861f35b6163f714")):
        m = cb.Mapper(cb.make_params(preset, max_read_length=128))
        m.upload_reference(seqs, names)
        m.upload_index(oidx.k, oidx.w, a["n_buckets"], a["flags"], a["keys"], a["vals"], a["occ"])
        recs, _ = m.map_batch(s1, o1, s2, o2)
        assert hashlib.md5(m.format_bed(m.postprocess(recs))).hexdigest() == md5


def test_bigger_synthetic_with_heavy_repeats_equals_oracle(tmp_path):
    """100k pairs on 4 x 2 Mbp with planted repeats: exercises every scratch tier and the sampling chunks."""
    import subprocess
    import sys
    d = str(tmp_path)
    subprocess.check_call([sys.executable, os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools", "gen_synth.py"),
                           "--out", d, "--n-seq", "4", "--seq-len", "2000000", "--n-pairs", "100000", "--short-frac", "0.2"])
    names, seqs = read_fasta(os.path.join(d, "ref.fa"))
    oref = orc.Reference(os.path.join(d, "ref.fa"))
    s1, o1, s2, o2 = load_pairs(d, "read1.fq", "read2.fq")
    for preset, kw in (("atac", {}), ("", dict(mapq_threshold=0, remove_pcr_duplicates=1))):
        m = cb.Mapper(cb.make_params(preset, max_read_length=64, **kw))
        m.upload_reference(seqs, names)
        m.build_index(17, 7)
        d_idx = m.download_index()
        oidx_path = os.path.join(d, "dev.index")
        # write the device-built index in the reference's file format and let the ORACLE load it
        with open(oidx_path, "wb") as f:
            np.array([17, 7], dtype=np.int32).tofile(f)
            np.array([d_idx["n_keys"], d_idx["n_buckets"], d_idx["n_keys"], d_idx["n_keys"],
                      int(d_idx["n_buckets"] * 0.77 + 0.5)], dtype=np.uint32).tofile(f)
            d_idx["flags"].tofile(f); d_idx["keys"].tofile(f); d_idx["vals"].tofile(f)
            np.array([len(d_idx["occ"])], dtype=np.uint32).tofile(f)
            d_idx["occ"].tofile(f)
        oidx = orc.Index(oidx_path)
        recs, stats = m.map_batch(s1, o1, s2, o2)
        orecs, _ = orc.map_pairs(orc.make_params(preset, **kw), oidx, oref, s1, o1, s2, o2, n_threads=8)
        assert stats["n_overflow_pairs"] == 0
        assert_same_records(recs, orecs)
        obed = orc.format_bed(oref, orc.postprocess(orc.make_params(preset, **kw), orecs))
        assert m.format_bed(m.postprocess(recs)) == obed


HIC_CASES = {
    "hic": dict(),
    "hic_q0": dict(mapq_threshold=0),
    "hic_e6dedup": dict(mapq_threshold=0, error_threshold=6, remove_pcr_duplicates=1),
}


def _read_names(path):
    import gzip as gz
    names = []
    with gz.open(path, "rb") as f:
        for i, line in enumerate(f):
            if i % 4 == 0:
                names.append(line[1:].split()[0])
    return names


@pytest.mark.parametrize("case", sorted(HIC_CASES))
def test_hic_split_alignment_equals_oracle_and_golden(case, golden_dir):
    """--preset hic: split alignment, four pairing directions, pairs output (BASELINE config 5 semantics)."""
    d = os.path.join(golden_dir, "synth_hic")
    names, seqs = read_fasta(os.path.join(d, "ref.fa.gz"))
    oref = orc.Reference(os.path.join(d, "ref.fa.gz"))
    oidx = orc.Index(ref=oref, k=17, w=7)
    s1, o1, s2, o2 = load_pairs(d)
    kw = HIC_CASES[case]
    m = cb.Mapper(cb.make_params("hic", max_read_length=160, **kw))
    m.upload_reference(seqs, names)
    a = oidx.arrays()
    m.upload_index(17, 7, a["n_buckets"], a["flags"], a["keys"], a["vals"], a["occ"])
    recs, stats = m.map_batch(s1, o1, s2, o2)
    orecs, otrace = orc.map_pairs(orc.make_params("hic", **kw), oidx, oref, s1, o1, s2, o2, trace=True)
    tr = m.trace(len(o1) - 1)
    alive = otrace["n_records"] > 0
    for f in ("n_minimizers", "n_pos_candidates", "n_neg_candidates", "n_pos_mappings", "n_neg_mappings", "min_errors", "n_best", "n_best_pairs"):
        bad = np.nonzero((tr[f][alive] != otrace[f][alive]).reshape(alive.sum(), -1).any(axis=1))[0]
        assert len(bad) == 0, (f, np.nonzero(alive)[0][bad[:5]], tr[f][alive][bad[:5]], otrace[f][alive][bad[:5]])
    assert_same_records(recs, orecs)
    assert stats["n_overflow_pairs"] == 0
    rn = _read_names(os.path.join(d, "read1.fq.gz"))
    text = m.format_pairs(m.postprocess_pairs(recs), rn, [len(s) for s in seqs])
    assert text == gzip.open(os.path.join(d, case + ".pairs.gz")).read()
    assert m.format_pairs_gpu(m.postprocess_gpu(recs), rn, [len(s) for s in seqs]) == text  # sort / dedup and text on the device


def test_hic_reference_quickstart_golden(golden_dir):
    import hashlib
    d = os.path.join(golden_dir, "ref_test")
    names, seqs = read_fasta(os.path.join(d, "ref.fa.gz"))
    oidx = orc.Index(os.path.join(d, "ref.index"))
    a = oidx.arrays()
    s1, o1, s2, o2 = load_pairs(d, "read1.fq", "read2.fq")
    m = cb.Mapper(cb.make_params("hic", max_read_length=128))
    m.upload_reference(seqs, names)
    m.upload_index(oidx.k, oidx.w, a["n_buckets"], a["flags"], a["keys"], a["vals"], a["occ"])
    recs, _ = m.map_batch(s1, o1, s2, o2)
    rn = [l[1:].split()[0] for i, l in enumerate(open(os.path.join(d, "read1.fq"), "rb")) if i % 4 == 0]
    text = m.format_pairs(m.postprocess_pairs(recs), rn, [len(s) for s in seqs])
    assert hashlib.md5(text).hexdigest() == "fc844a251ebdcec0f641b59fef804d0f"


def _read_barcodes(path):
    import gzip as gz
    seqs, quals = [], []
    with gz.open(path, "rb") as f:
        for i, line in enumerate(f):
            if i % 4 == 1:
                seqs.append(line.rstrip(b"\r\n"))
            elif i % 4 == 3:
                quals.append(line.rstrip(b"\r\n"))
    return np.frombuffer(b"".join(seqs), dtype=np.uint8), np.frombuffer(b"".join(quals), dtype=np.uint8), len(seqs[0])


@pytest.mark.parametrize("case,use_wl", [("sc_whitelist", True), ("sc_nowhitelist", False)])
def test_scatac_barcodes_equal_oracle_and_golden(case, use_wl, golden_dir):
    """BASELINE config 4 semantics: cell barcodes, whitelist correction on the device, cell-level duplicate removal."""
    d = os.path.join(golden_dir, "synth_sc")
    names, seqs = read_fasta(os.path.join(d, "ref.fa.gz"))
    oref = orc.Reference(os.path.join(d, "ref.fa.gz"))
    oidx = orc.Index(ref=oref, k=17, w=7)
    s1, o1, s2, o2 = load_pairs(d)
    bcs, quals, bc_len = _read_barcodes(os.path.join(d, "barcode.fq.gz"))
    m = cb.Mapper(cb.make_params("atac", max_read_length=64))
    m.upload_reference(seqs, names)
    a = oidx.arrays()
    m.upload_index(17, 7, a["n_buckets"], a["flags"], a["keys"], a["vals"], a["occ"])
    wl = None
    if use_wl:
        wl = orc.Whitelist(os.path.join(d, "whitelist.txt"), bc_len)
        wl.sample(bcs)   # host pre-pass of the reference (ComputeBarcodeAbundance); the product CLI has its own
        keys, counts, ns = wl.arrays()
        m.upload_barcode_whitelist(keys, counts, ns, bc_len)
    recs, stats = m.map_batch(s1, o1, s2, o2, barcodes=bcs, barcode_quals=quals, bc_len=bc_len)
    orecs, obc, ost = orc.map_pairs_bc(orc.make_params("atac"), oidx, oref, s1, o1, s2, o2, bcs, quals, bc_len, whitelist=wl)
    assert_same_records(recs, orecs)
    assert np.array_equal(stats["barcode_keys"], obc)
    if use_wl:
        assert (stats["n_barcodes_in_whitelist"], stats["n_barcodes_corrected"]) == (int(ost[0]), int(ost[1]))
    r2, b2 = m.postprocess_bc(recs, stats["barcode_keys"])
    assert m.format_bed_bc(r2, b2, bc_len) == gzip.open(os.path.join(d, case + ".bed.gz")).read()


def _random_records(rng, n, pairs):
    """Records with many equal fragments, equal MAPQs and ties down to the last key field."""
    if pairs:
        r = np.zeros(n, dtype=cb.PAIRS_RECORD)
        r["read_id"] = rng.permutation(n).astype(np.uint32)
        r["rid1"] = rng.integers(0, 3, n); r["rid2"] = np.maximum(r["rid1"], rng.integers(0, 3, n))
        r["pos1"] = rng.integers(0, 40, n) * 7; r["pos2"] = rng.integers(0, 40, n) * 7
        r["strand1"] = rng.integers(0, 2, n); r["strand2"] = rng.integers(0, 2, n)
        r["mapq"] = rng.choice([0, 1, 13, 60], n); r["is_unique"] = rng.integers(0, 2, n)
        return r
    r = np.zeros(n, dtype=cb.PE_RECORD)
    r["read_id"] = rng.permutation(n).astype(np.uint32)
    r["rid"] = rng.integers(0, 3, n)
    r["fragment_start"] = rng.integers(0, 60, n) * 11
    r["fragment_length"] = rng.choice([60, 61, 200, 65535], n)
    r["mapq"] = rng.choice([0, 3, 30, 60], n); r["direction"] = rng.integers(0, 2, n); r["is_unique"] = rng.integers(0, 2, n)
    r["num_dups"] = 1
    r["positive_alignment_length"] = rng.choice([48, 50, 51], n); r["negative_alignment_length"] = rng.choice([49, 50], n)
    return r


@pytest.mark.parametrize("kind", ["bed", "bed_bc", "pairs"])
@pytest.mark.parametrize("low_mem,dedup,tn5,q", [(1, 1, 0, 30), (1, 1, 1, 0), (1, 0, 1, 3), (0, 1, 1, 0), (0, 1, 0, 30), (0, 0, 0, 1)])
def test_postprocess_on_device_equals_host(kind, low_mem, dedup, tn5, q):
    rng = np.random.default_rng(7 + low_mem * 8 + dedup * 4 + tn5 * 2 + q)
    pairs = kind == "pairs"
    kw = dict(low_memory_mode=low_mem, remove_pcr_duplicates=dedup, mapq_threshold=q)
    if pairs:
        p = cb.make_params("hic", max_read_length=64, **kw)
    else:
        p = cb.make_params("", max_read_length=64, tn5_shift=tn5, **kw)
    if pairs and dedup and not low_mem:
        # RemovePCRDuplicate keeps the LAST record of a run (mapping_processor.h:181-197); the pairs path only has the low-memory
        # rule, so the combination is refused, not approximated
        with pytest.raises(cb.CmxError):
            cb.Mapper(p)
        return
    m = cb.Mapper(p)
    for n in (1, 2, 1000, 200000):
        recs = _random_records(rng, n, pairs)
        if n >= 1000:  # a long run of duplicates (num_dups saturates at 255)
            recs[: n // 3] = recs[0]
            recs["read_id"][: n // 3] = np.arange(n // 3, dtype=np.uint32) + 7 * n
            recs["mapq"][: n // 3] = rng.choice([0, 30, 60], n // 3)
        if kind == "bed_bc":
            bcs = rng.integers(0, 5, n).astype(np.uint64) * 0x123456789
            want, wbc = m.postprocess_bc(recs, bcs)
            got, gbc = m.postprocess_gpu(recs, bcs)
            assert np.array_equal(wbc, gbc)
        elif pairs:
            want, got = m.postprocess_pairs(recs), m.postprocess_gpu(recs)
        else:
            want, got = m.postprocess(recs), m.postprocess_gpu(recs)
        assert_same_records(got, want)


@pytest.mark.parametrize("bc", [False, True])
@pytest.mark.parametrize("dedup,tn5,q", [(1, 0, 30), (1, 1, 0), (0, 1, 3)])
def test_native_dedup_exchange_world_of_one_equals_host_postprocess(bc, dedup, tn5, q):
    """cmx_dedup_exchange (tuple pack, ncclAllGather, radix sort, survivor rule on the GPU) with a communicator of one rank +
    cmx_exchange_finish == the host low-memory post-processing.  The N > 1 run is tools/multi_gpu_map.py under torchrun."""
    rng = np.random.default_rng(31 + dedup * 4 + tn5 * 2 + q + (8 if bc else 0))
    p = cb.make_params("", max_read_length=64, tn5_shift=tn5, low_memory_mode=1, remove_pcr_duplicates=dedup, mapq_threshold=q)
    m = cb.Mapper(p)
    m.comm_init(1, 0, m.comm_unique_id())
    for n in (0, 1, 1000, 200000):
        recs = _random_records(rng, n, False)
        if n >= 1000:
            recs[: n // 3] = recs[0]
            recs["read_id"][: n // 3] = np.arange(n // 3, dtype=np.uint32) + 7 * n
            recs["mapq"][: n // 3] = rng.choice([0, 30, 60], n // 3)
        if bc:
            bcs = rng.integers(0, 5, n).astype(np.uint64) * 0x123456789
            want, wbc = m.postprocess_bc(recs, bcs)
            surv, sbc, st = m.dedup_exchange(recs, bcs)
            got, gbc = cb.exchange_finish(p, surv, sbc)
            assert np.array_equal(wbc, gbc)
        else:
            want = m.postprocess(recs)
            surv, st = m.dedup_exchange(recs)
            got = cb.exchange_finish(p, surv)
        assert st["n_global"] == n and st["n_ranks"] == 1
        assert_same_records(got, want)
        # the range-shuffle form (cmx_dedup_shuffle): with one rank the whole key range is this rank's
        if bc:
            part, pbc, sst = m.dedup_shuffle(recs, bcs)
            assert np.array_equal(wbc, pbc)
        else:
            part, sst = m.dedup_shuffle(recs)
        assert sst["n_global"] == n and sst["n_received"] == n and sst["n_ranks"] == 1 and sst["bytes_sent"] == 0
        assert_same_records(part, want)
        if n >= 1000:  # too small an output buffer is refused, with the needed capacity
            with pytest.raises(cb.CmxError):
                m.dedup_shuffle(recs, bcs if bc else None, capacity=len(want) - 1)
    m.comm_destroy()


@pytest.mark.parametrize("bc", [False, True])
def test_bed_text_on_device_equals_host(synth, bc):
    m = _mapper(synth, CASES["default"])
    rng = np.random.default_rng(5)
    for n in (0, 1, 999, 300000):
        recs = _random_records(rng, n, False)
        recs["rid"] = rng.integers(0, len(synth["names"]), n)
        recs["fragment_start"] = rng.choice([0, 9, 10, 99999, 4294967295, 1000000000], n)
        recs["num_dups"] = rng.choice([1, 9, 10, 255], n)
        recs["mapq"] = rng.choice([0, 9, 10, 60], n)
        if bc:
            bcs = rng.integers(0, 1 << 32, n).astype(np.uint64)
            assert m.format_bed_gpu(recs, bcs, 16) == m.format_bed_bc(recs, bcs, 16)
        else:
            assert m.format_bed_gpu(recs) == m.format_bed(recs)


SE_CASES = {
    "se_default": dict(preset=""),
    "se_chip": dict(preset="chip"),
    "se_q0dedup_tn5": dict(preset="", mapq_threshold=0, remove_pcr_duplicates=1, tn5_shift=1),
    "se_n3q0": dict(preset="", max_num_best_mappings=3, mapq_threshold=0),
    "se_lowmem_q0": dict(preset="", low_memory_mode=1, mapq_threshold=0, remove_pcr_duplicates=1, tn5_shift=1),
}


@pytest.mark.parametrize("case", sorted(SE_CASES))
def test_single_end_records_equal_oracle_and_golden(synth, case):
    """chromap -1 only (MapSingleEndReads): records == oracle, BED == the reference binary's, host and device post-processing."""
    kw = dict(SE_CASES[case])
    m = _mapper(synth, dict(kw, single_end=1))
    s1, o1, _, _ = synth["pairs"]
    recs, stats = m.map_batch(s1, o1, None, None)
    orecs = orc.map_reads_se(_oparams(kw), synth["oidx"], synth["oref"], s1, o1)
    assert len(recs) == len(orecs)
    assert_same_records(recs, orecs)
    assert stats["n_overflow_pairs"] == 0
    want = gzip.open(os.path.join(synth["d"], case + ".bed.gz")).read()
    assert m.format_bed(m.postprocess(recs)) == want
    assert m.format_bed_gpu(m.postprocess_gpu(recs)) == want


def test_single_end_heavy_repeats_through_all_tiers(tmp_path):
    """Reads from repeat families (hundreds to thousands of hits): single-end through the CTA tiers == oracle."""
    import subprocess
    import sys
    d = str(tmp_path)
    subprocess.check_call([sys.executable, os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools", "gen_synth.py"),
                           "--out", d, "--seed", "23", "--n-seq", "2", "--seq-len", "400000", "--n-pairs", "20000", "--repeat-copies", "60",
                           "--repeat-len", "3000", "--fam-copies", "3000"])
    names, seqs = read_fasta(os.path.join(d, "ref.fa"))
    oref = orc.Reference(os.path.join(d, "ref.fa"))
    oidx = orc.Index(ref=oref, k=17, w=7)
    kw = dict(preset="", mapq_threshold=0, max_num_best_mappings=2)
    p = cb.make_params("", max_read_length=64, single_end=1, mapq_threshold=0, max_num_best_mappings=2)
    m = cb.Mapper(p)
    m.upload_reference(seqs, names)
    a = oidx.arrays()
    m.upload_index(17, 7, a["n_buckets"], a["flags"], a["keys"], a["vals"], a["occ"])
    s1, o1, _, _ = load_pairs(d, "read1.fq", "read2.fq")
    recs, stats = m.map_batch(s1, o1, None, None)
    orecs = orc.map_reads_se(_oparams(kw), oidx, oref, s1, o1, n_threads=8)
    assert stats["n_overflow_pairs"] == 0
    tm = m.timing()
    assert tm["tier_pairs"][1] > 0
    assert len(recs) == len(orecs)
    assert_same_records(recs, orecs)


def _d2h(ptr, nbytes):
    rt = C.CDLL("libcudart.so.12")
    rt.cudaMemcpy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
    out = np.empty(nbytes, dtype=np.uint8)
    assert rt.cudaMemcpy(out.ctypes.data, ptr, nbytes, 2) == 0
    return out


def test_fastq_ingest_on_device_equals_host_reader(synth):
    """cmx_fastq_cut + cmx_ingest_fastq: packed bases / qualities / name spans == the host FASTQ reader; mapping the
    device-resident batch gives the same records as mapping the host batch."""
    m = _mapper(synth, CASES["default"])
    d = synth["d"]
    t1 = gzip.open(os.path.join(d, "read1.fq.gz")).read()
    t2 = gzip.open(os.path.join(d, "read2.fq.gz")).read()
    s1, o1, s2, o2 = synth["pairs"]
    n = len(o1) - 1
    # record-boundary cuts
    b, k = m.fastq_cut(t1, 1000)
    assert k == 1000 and t1[:b].count(b"\n") == 4000 and t1[b - 1:b] == b"\n"
    b_all, k_all = m.fastq_cut(t1 + b"@partial\nACGT\n+", 10 ** 9)
    assert k_all == n and b_all == len(t1)
    g1, spans = m.ingest_fastq(0, t1, want_qual=True, want_names=True)
    g2, _ = m.ingest_fastq(1, t2)
    assert g1.n_reads == n and g2.n_reads == n
    off = _d2h(g1.off, 4 * (n + 1)).view(np.uint32)
    assert np.array_equal(off, o1)
    assert np.array_equal(_d2h(g1.seq, int(off[-1])), s1)
    recs = read_fastq_records(os.path.join(d, "read1.fq.gz"))
    assert _d2h(g1.qual, int(off[-1])).tobytes() == b"".join(q for _, _, q in recs)
    names = [t1[a:a + l] for a, l in spans]
    assert names == [nm for nm, _, _ in recs]
    assert g1.min_len == min(len(s) for _, s, _ in recs) and g1.max_len == max(len(s) for _, s, _ in recs)
    want, _ = m.map_batch(s1, o1, s2, o2)
    got, _ = m.map_batch(g1.seq, g1.off, g2.seq, g2.off, on_device=True, n_pairs=n)
    assert_same_records(got, want)
    # CRLF line ends and a final chunk are handled like kseq does; anything else is refused, not guessed at
    crlf = t1[:b].replace(b"\n", b"\r\n")
    gc, _ = m.ingest_fastq(2, crlf)
    assert gc.n_reads == 1000 and np.array_equal(_d2h(gc.off, 4 * 1001).view(np.uint32), o1[:1001])
    for bad in (b">r\nACGT\n+\nIIII\n", b"@r\nACGT\nIIII\nIIII\n", b"@r\n\n+\n\n", b"@r\nACGT\n+\nIII\n"):
        with pytest.raises(cb.CmxError):
            m.ingest_fastq(2, bad)


def test_scatac_large_whitelist_equals_oracle(golden_dir, tmp_path):
    """A 300 000-entry whitelist (BASELINE config 4 uses 737 k): device hash table and 1-substitution correction == oracle."""
    d = os.path.join(golden_dir, "synth_sc")
    names, seqs = read_fasta(os.path.join(d, "ref.fa.gz"))
    oref = orc.Reference(os.path.join(d, "ref.fa.gz"))
    oidx = orc.Index(ref=oref, k=17, w=7)
    s1, o1, s2, o2 = load_pairs(d)
    n, bc_len = len(o1) - 1, 16
    rng = np.random.default_rng(99)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    wl_codes = np.unique(rng.integers(0, 1 << 32, 300000, dtype=np.uint64))
    wl_seq = acgt[(wl_codes[:, None] >> (2 * np.arange(bc_len - 1, -1, -1, dtype=np.uint64))[None, :]) & np.uint64(3)]
    wl_path = str(tmp_path / "wl.txt")
    with open(wl_path, "wb") as f:
        f.write(b"\n".join(r.tobytes() for r in wl_seq) + b"\n")
    cells = wl_seq[rng.integers(0, len(wl_seq), 800)]
    bcs = cells[rng.integers(0, len(cells), n)].copy()
    sub = rng.random(n) < 0.08
    pos = rng.integers(0, bc_len, n)
    bcs[sub, pos[sub]] = acgt[rng.integers(0, 4, int(sub.sum()))]
    bcs[rng.random(n) < 0.02, rng.integers(0, bc_len)] = ord("N")
    junk = rng.random(n) < 0.03
    bcs[junk] = acgt[rng.integers(0, 4, (int(junk.sum()), bc_len))]
    quals = (rng.integers(2, 41, (n, bc_len)) + 33).astype(np.uint8)
    bcs, quals = bcs.reshape(-1), quals.reshape(-1)
    m = cb.Mapper(cb.make_params("atac", max_read_length=64))
    m.upload_reference(seqs, names)
    a = oidx.arrays()
    m.upload_index(17, 7, a["n_buckets"], a["flags"], a["keys"], a["vals"], a["occ"])
    wl = orc.Whitelist(wl_path, bc_len)
    wl.sample(bcs)
    keys, counts, ns = wl.arrays()
    m.upload_barcode_whitelist(keys, counts, ns, bc_len)
    recs, stats = m.map_batch(s1, o1, s2, o2, barcodes=bcs, barcode_quals=quals, bc_len=bc_len)
    orecs, obc, ost = orc.map_pairs_bc(orc.make_params("atac"), oidx, oref, s1, o1, s2, o2, bcs, quals, bc_len, whitelist=wl)
    assert int(ost[1]) > 50  # corrections did happen
    assert_same_records(recs, orecs)
    assert np.array_equal(stats["barcode_keys"], obc)
    assert (stats["n_barcodes_in_whitelist"], stats["n_barcodes_corrected"]) == (int(ost[0]), int(ost[1]))
    r2, b2 = m.postprocess_gpu(recs, stats["barcode_keys"])
    w2, wb2 = m.postprocess_bc(recs, stats["barcode_keys"])
    assert_same_records(r2, w2) and np.array_equal(b2, wb2)


def test_reads_longer_than_max_read_length_escalate_and_ragged_lengths(golden_dir):
    """2x150 bp reads, randomly cut to 20..150 bases, through a context sized for 64-base reads: too-short reads are
    dropped, long ones climb the scratch tiers (their minimizer capacity grows 2x / 4x); records == oracle.  Reads
    beyond the largest tier are reported (CMX_ERR_OVERFLOW), never mapped wrongly."""
    d = os.path.join(golden_dir, "synth_hic")
    names, seqs = read_fasta(os.path.join(d, "ref.fa.gz"))
    oref = orc.Reference(os.path.join(d, "ref.fa.gz"))
    oidx = orc.Index(ref=oref, k=17, w=7)
    s1, o1, s2, o2 = load_pairs(d)
    rng = np.random.default_rng(3)

    def cut(s, o):
        lens = np.minimum(np.diff(o.astype(np.int64)), rng.integers(20, 151, len(o) - 1))
        parts = [s[o[i]:o[i] + lens[i]] for i in range(len(lens))]
        off = np.zeros(len(o), dtype=np.uint32)
        off[1:] = np.cumsum(lens)
        return np.concatenate(parts), off

    s1, o1 = cut(s1, o1)
    s2, o2 = cut(s2, o2)
    kw = dict(preset="", mapq_threshold=0)
    m = cb.Mapper(cb.make_params("", max_read_length=64, mapq_threshold=0))
    m.upload_reference(seqs, names)
    a = oidx.arrays()
    m.upload_index(17, 7, a["n_buckets"], a["flags"], a["keys"], a["vals"], a["occ"])
    recs, stats = m.map_batch(s1, o1, s2, o2)
    orecs, _ = orc.map_pairs(_oparams(kw), oidx, oref, s1, o1, s2, o2)
    assert stats["n_overflow_pairs"] == 0
    tm = m.timing()
    assert tm["tier_pairs"][1] > 0 and tm["tier_pairs"][2] > 0
    assert len(recs) == len(orecs) and len(recs) > 500
    assert_same_records(recs, orecs)
    m2 = cb.Mapper(cb.make_params("", max_read_length=32, mapq_threshold=0, min_read_length=20))  # largest tier: 128 bases
    m2.upload_reference(seqs, names)
    m2.upload_index(17, 7, a["n_buckets"], a["flags"], a["keys"], a["vals"], a["occ"])
    with pytest.raises(cb.CmxError) as ei:
        m2.map_batch(s1, o1, s2, o2)
    assert "scratch tier" in str(ei.value)


def test_bench_sized_batch_properties_and_sampled_oracle():
    """One bench-sized step (2 M pairs, four reference batches) on a 300 Mbp synthetic reference: size-independent
    properties of the whole path, plus the oracle on a contiguous sample that includes a taskloop-chunk boundary."""
    torch = pytest.importorskip("torch")
    import bench
    dev = torch.device("cuda", 0)
    n_seq, n, L = 6, 2000000, 50
    ref, offsets, seq_len = bench.gen_reference(torch, dev, 300000000, n_seq, 11)
    p = cb.make_params("", max_read_length=64, mapq_threshold=0, remove_pcr_duplicates=1, low_memory_mode=1)
    m = cb.Mapper(p, device=0)
    m.upload_reference_ptr(ref.data_ptr(), offsets)
    m.names = ["chr%d" % (i + 1) for i in range(n_seq)]
    m.build_index(17, 7)
    r1, r2, off = bench.gen_pairs(torch, ref, n_seq, seq_len, n, L, 424242, dev)
    h1, h2, ho = r1.cpu().numpy(), r2.cpu().numpy(), off.cpu().numpy().view(np.uint32)
    out_dev = torch.empty(n * 24, dtype=torch.uint8, device=dev)
    # (a) the same records whatever the path: device-resident input with 4 lanes / 1 lane, host input (piecewise upload)
    m.set_lanes(4)
    _, st4 = m.map_batch(r1, off, r2, off, on_device=True, n_pairs=n, out=out_dev, out_on_device=True)
    rec4 = out_dev.cpu().numpy()[:st4["n_records"] * 24].view(cb.PE_RECORD).copy()
    m.set_lanes(1)
    _, st1 = m.map_batch(r1, off, r2, off, on_device=True, n_pairs=n, out=out_dev, out_on_device=True)
    rec1 = out_dev.cpu().numpy()[:st1["n_records"] * 24].view(cb.PE_RECORD).copy()
    m.set_lanes(4)
    rech, sth = m.map_batch(h1, ho, h2, ho)
    assert st4["n_overflow_pairs"] == 0 and st4["n_records"] == st1["n_records"] == sth["n_records"] > 0.9 * n
    assert_same_records(rec4, rec1)
    assert_same_records(rec4, rech)
    # (b) records come back in read order, one per mapped pair, inside their sequences
    assert np.all(np.diff(rec4["read_id"].astype(np.int64)) > 0)
    assert np.all(rec4["rid"] < n_seq) and np.all(rec4["fragment_start"].astype(np.int64) + rec4["fragment_length"] <= seq_len)
    assert np.all(rec4["mapq"] <= 60)
    # (c) post-processing: device == host; output sorted by the reference's key, no duplicate fragment left, counts add up
    pg, ph = m.postprocess_gpu(rec4), m.postprocess(rec4)
    assert_same_records(pg, ph)
    key = (pg["rid"].astype(np.uint64) << np.uint64(48)) | (pg["fragment_start"].astype(np.uint64) << np.uint64(16)) | pg["fragment_length"].astype(np.uint64)
    assert np.all(np.diff(key.astype(np.int64)) > 0)
    assert int(pg["num_dups"].astype(np.int64).sum()) == len(rec4)  # no run longer than 255 here, MAPQ threshold 0
    assert m.format_bed_gpu(pg) == m.format_bed(pg)
    # (d) the oracle on pairs [495000, 505000): the end of reference batch 0 and the start of batch 1
    idx = m.download_index()
    oidx = orc.Index(arrays=idx, k=17, w=7)
    href = ref.cpu().numpy()
    oref = orc.Reference(seqs=[href[int(offsets[i]):int(offsets[i + 1])] for i in range(n_seq)])
    op = orc.make_params("", mapq_threshold=0, remove_pcr_duplicates=1, low_memory_mode=1)
    for b0, lo, hi in ((0, 495000, 500000), (500000, 500000, 505000)):
        # the sampling generator restarts per taskloop chunk of a batch: map whole chunks -> the batch's last / first 5000 pairs
        s1, s2 = h1[lo * L:hi * L], h2[lo * L:hi * L]
        o = (np.arange(hi - lo + 1, dtype=np.uint32) * L)
        orecs, _ = orc.map_pairs(op, oidx, oref, s1, o, s2, o, first_read_id=lo, n_threads=8)
        got = rec4[(rec4["read_id"] >= lo) & (rec4["read_id"] < hi)]
        assert len(got) == len(orecs) > 4000
        assert_same_records(got, orecs)


@pytest.mark.parametrize("case,kw,use_wl", [("se_sc_whitelist", dict(preset="atac"), True), ("se_sc_nowhitelist", dict(preset="atac"), False),
                                            ("se_sc_inmem", dict(preset="", mapq_threshold=0, remove_pcr_duplicates=1, tn5_shift=1), True)])
def test_single_end_barcoded_equals_oracle_and_golden(case, kw, use_wl, golden_dir):
    """Single-end reads with cell barcodes (MappingWithBarcode): device correction + mapping == oracle; post-processing on the
    host and on the device reproduce the reference binary's BED (duplicates = same barcode and start, consecutive in order)."""
    d = os.path.join(golden_dir, "synth_sc")
    names, seqs = read_fasta(os.path.join(d, "ref.fa.gz"))
    oref = orc.Reference(os.path.join(d, "ref.fa.gz"))
    oidx = orc.Index(ref=oref, k=17, w=7)
    s1, o1, _, _ = load_pairs(d)
    bcs, quals, bc_len = _read_barcodes(os.path.join(d, "barcode.fq.gz"))
    kw = dict(kw)
    preset = kw.pop("preset")
    m = cb.Mapper(cb.make_params(preset, max_read_length=64, single_end=1, **kw))
    m.upload_reference(seqs, names)
    a = oidx.arrays()
    m.upload_index(17, 7, a["n_buckets"], a["flags"], a["keys"], a["vals"], a["occ"])
    wl = None
    if use_wl:
        wl = orc.Whitelist(os.path.join(d, "whitelist.txt"), bc_len)
        wl.sample(bcs)
        keys, counts, ns = wl.arrays()
        m.upload_barcode_whitelist(keys, counts, ns, bc_len)
    recs, stats = m.map_batch(s1, o1, None, None, barcodes=bcs, barcode_quals=quals, bc_len=bc_len)
    orecs, obc, ost = orc.map_reads_se_bc(orc.make_params(preset, single_end=1, **kw), oidx, oref, s1, o1, bcs, quals, bc_len, whitelist=wl)
    assert_same_records(recs, orecs)
    assert np.array_equal(stats["barcode_keys"], obc)
    want = gzip.open(os.path.join(d, case + ".bed.gz")).read()
    r2, b2 = m.postprocess_bc(recs, stats["barcode_keys"])
    assert m.format_bed_bc(r2, b2, bc_len) == want
    r3, b3 = m.postprocess_gpu(recs, stats["barcode_keys"])
    assert m.format_bed_gpu(r3, b3, bc_len) == want


@pytest.mark.parametrize("case,kw,paired", [("pe_chip", dict(preset="chip"), True), ("pe_q0d", dict(preset="", mapq_threshold=0, remove_pcr_duplicates=1), True),
                                            ("pe_n3", dict(preset="", max_num_best_mappings=3, mapq_threshold=0), True),
                                            ("se_n3", dict(preset="", max_num_best_mappings=3, mapq_threshold=0), False)])
def test_sam_cores_equal_oracle_and_text_equals_reference(synth, case, kw, paired):
    """output_format 4: the device computes, per reported mapping, the ksw_semi_global3 span and CIGAR (sam_kernels.cuh) and
    MAPQ from those spans; cores == oracle, and the host writer turns them into the reference binary's SAM file."""
    from tests.util import read_fastq_records
    extra = dict(output_format=4) if paired else dict(output_format=4, single_end=1)
    m = _mapper(synth, dict(kw, **extra))
    s1, o1, s2, o2 = synth["pairs"]
    recs, stats = m.map_batch(s1, o1, s2 if paired else None, o2 if paired else None)
    assert recs.dtype == cb.SAM_RECORD and stats["n_overflow_pairs"] == 0
    cores = orc.map_sam_cores(_oparams(kw), synth["oidx"], synth["oref"], s1, o1, s2 if paired else None, o2 if paired else None)
    assert len(recs) == len(cores) > 1000
    for f in ("read_id", "rid", "mapq", "is_unique", "secondary", "overflow"):
        assert np.array_equal(recs[f], cores[f]), f
    for q in range(2 if paired else 1):
        for f in ("pos", "end", "strand", "n_cigar"):
            bad = np.nonzero(recs[f][:, q] != cores[f][:, q])[0]
            assert len(bad) == 0, (f, q, bad[:5], recs[f][bad[:5], q], cores[f][bad[:5], q])
        for i in range(len(recs)):
            k = recs["n_cigar"][i, q]
            assert np.array_equal(recs["cigar"][i, q, :k], cores["cigar"][i, q, :k]), (i, q)
    if case in ("pe_chip", "pe_q0d", "se_n3"):
        d = synth["d"]
        split = lambda r: ([a for a, _, _ in r], [b for _, b, _ in r], [c for _, _, c in r])
        r1 = split(read_fastq_records(os.path.join(d, "read1.fq.gz")))
        r2 = split(read_fastq_records(os.path.join(d, "read2.fq.gz"))) if paired else None
        text = cb.format_sam(m.params, synth["names"], synth["seqs"], recs, r1, r2)
        assert text == gzip.open(os.path.join(d, case + ".sam.gz")).read()
