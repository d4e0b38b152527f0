"""CPU-only checks of the product boundary: the C-ABI library loads and exports every symbol that
include/chromap_b200.h declares; without a GPU the product refuses to run (no CPU fallback)."""
import ctypes
import os
import re

import pytest

import chromap_b200 as cb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "chromap_b200.h")).read()
    return sorted(set(re.findall(r"\b(cmx_[a-z_0-9]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    if not os.path.exists(cb.lib_path()):
        import __graft_entry__
        __graft_entry__.build()
    lib = ctypes.CDLL(cb.lib_path())
    names = _declared()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), n


def test_presets_match_reference_driver():
    for preset, want in (("chip", dict(max_insert_size=2000, remove_pcr_duplicates=1, low_memory_mode=1, trim_adapters=0)),
                         ("atac", dict(max_insert_size=2000, remove_pcr_duplicates=1, low_memory_mode=1, trim_adapters=1, tn5_shift=1)),
                         ("", dict(max_insert_size=1000, error_threshold=8, mapq_threshold=30, low_memory_mode=0))):
        p = cb.make_params(preset)
        for k, v in want.items():
            assert getattr(p, k) == v
    with pytest.raises(cb.CmxError):
        cb.make_params("nope")


def test_no_gpu_means_loud_failure():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(cb.CmxError):
        cb.Mapper(cb.make_params("chip"))


def test_taskloop_chunks_match_libgomp_probe():
    # measured with a stand-alone OpenMP probe on this image's libgomp (see DESIGN.md)
    assert cb.taskloop_chunks(23459) == [0, 5865, 11730, 17595]
    assert cb.taskloop_chunks(9999) == [0]
    assert cb.taskloop_chunks(10001) == [0, 5001]
    assert len(cb.taskloop_chunks(500000)) == 100


def test_fastq_cut_finds_record_boundaries():
    """cmx_fastq_cut is host code: whole 4-line records only, at most max_records of them."""
    import ctypes as C
    import chromap_b200 as cb
    L = cb.load_library()
    text = b"@a 1\nACGT\n+\nIIII\n@b\nAC\n+\nII\n@c\nA"
    n = C.c_uint32()
    assert L.cmx_fastq_cut(text, len(text), 10, C.byref(n)) == len(b"@a 1\nACGT\n+\nIIII\n@b\nAC\n+\nII\n") and n.value == 2
    assert L.cmx_fastq_cut(text, len(text), 1, C.byref(n)) == len(b"@a 1\nACGT\n+\nIIII\n") and n.value == 1
    assert L.cmx_fastq_cut(text, 5, 10, C.byref(n)) == 0 and n.value == 0
    assert L.cmx_fastq_cut(b"", 0, 10, C.byref(n)) == 0 and n.value == 0


@pytest.mark.parametrize("case,kw,paired", [("pe_chip", dict(preset="chip"), True), ("pe_q0d", dict(preset="", mapq_threshold=0, remove_pcr_duplicates=1), True),
                                            ("se_n3", dict(preset="", max_num_best_mappings=3, mapq_threshold=0), False)])
def test_host_sam_writer_reproduces_reference_text(golden_dir, case, kw, paired):
    """cmx_format_sam is host code: fed with the oracle's SAM cores (the device emits the same cores, checked in the gpu
    tests) it writes the reference binary's SAM file byte for byte - flags, mate fields, TLEN, order, dedup, NM / MD."""
    import gzip
    import os
    import chromap_b200 as cb
    from oracle import oracle_py as orc
    from tests.util import load_pairs, read_fasta, read_fastq_records
    d = os.path.join(golden_dir, "synth_small")
    names, seqs = read_fasta(os.path.join(d, "ref.fa.gz"))
    ref = orc.Reference(os.path.join(d, "ref.fa.gz"))
    idx = orc.Index(ref=ref, k=17, w=7)
    s1, o1, s2, o2 = load_pairs(d)
    kw = dict(kw)
    preset = kw.pop("preset")
    cores = orc.map_sam_cores(orc.make_params(preset, **kw), idx, ref, s1, o1, s2 if paired else None, o2 if paired else None)
    r1 = read_fastq_records(os.path.join(d, "read1.fq.gz"))
    r2 = read_fastq_records(os.path.join(d, "read2.fq.gz")) if paired else None
    split = lambda r: ([a for a, _, _ in r], [b for _, b, _ in r], [c for _, _, c in r])
    p = cb.make_params(preset, max_read_length=64, output_format=4, single_end=0 if paired else 1, **kw)
    text = cb.format_sam(p, names, seqs, cores.view(cb.SAM_RECORD), split(r1), split(r2) if paired else None)
    assert text == gzip.open(os.path.join(d, case + ".sam.gz")).read()


def test_integration_stub_compiles_against_the_reference_headers():
    """The bridge shown in INTEGRATION.md is real code: it type-checks against the reference's own headers.  Those headers cannot
    be stored here, so the check runs where build() compiles the reference binary (oracle/Makefile, target ref) and records its
    result in oracle/_ref/integration_bridge.txt; this test holds the current INTEGRATION.md and include/chromap_b200.h to it."""
    from oracle import integration_bridge
    p = os.path.join(ROOT, "oracle", "_ref", "integration_bridge.txt")
    if not os.path.exists(p):
        pytest.skip("the reference's headers were absent when the project was built (oracle/Makefile, target ref)")
    head, _, diagnostics = open(p).read().partition("\n")
    checked, rc = head.split()
    assert checked == integration_bridge.digest(), "INTEGRATION.md or include/chromap_b200.h changed since the check: run build() again"
    assert rc == "0", diagnostics


@pytest.mark.parametrize("kw,paired", [(dict(preset="", max_num_best_mappings=3, mapq_threshold=0), True), (dict(preset="atac"), True),
                                       (dict(preset="", low_memory_mode=1, mapq_threshold=0, remove_pcr_duplicates=1), True),
                                       (dict(preset="", low_memory_mode=1, mapq_threshold=0, remove_pcr_duplicates=1), False), (dict(preset="chip"), False)])
def test_host_sam_writer_equals_oracle_writer_on_more_parameter_sets(golden_dir, tmp_path, kw, paired):
    """More parameter sets than there are committed SAM files: the library's writer against the oracle's (which reproduced the
    reference binary on all of them): secondary flags (-n 3), trimmed reads (atac), both duplicate rules."""
    import chromap_b200 as cb
    from oracle import oracle_py as orc
    from tests.util import load_pairs, read_fasta, read_fastq_records
    d = os.path.join(golden_dir, "synth_small")
    names, seqs = read_fasta(os.path.join(d, "ref.fa.gz"))
    ref = orc.Reference(os.path.join(d, "ref.fa.gz"))
    idx = orc.Index(ref=ref, k=17, w=7)
    ip = str(tmp_path / "ref.index")
    idx.save(ip)
    s1, o1, s2, o2 = load_pairs(d)
    kw = dict(kw)
    preset = kw.pop("preset")
    op = orc.make_params(preset, **kw)
    out = str(tmp_path / "o.sam")
    orc.run_files_sam(op, ip, os.path.join(d, "ref.fa.gz"), os.path.join(d, "read1.fq.gz"), os.path.join(d, "read2.fq.gz") if paired else None, out)
    cores = orc.map_sam_cores(op, idx, ref, s1, o1, s2 if paired else None, o2 if paired else None)
    split = lambda r: ([a for a, _, _ in r], [b for _, b, _ in r], [c for _, _, c in r])
    r1 = split(read_fastq_records(os.path.join(d, "read1.fq.gz")))
    r2 = split(read_fastq_records(os.path.join(d, "read2.fq.gz"))) if paired else None
    p = cb.make_params(preset, max_read_length=64, output_format=4, single_end=0 if paired else 1, **kw)
    assert cb.format_sam(p, names, seqs, cores.view(cb.SAM_RECORD), r1, r2) == open(out, "rb").read()


@pytest.mark.parametrize("case,kw,paired", [("pe_chip", dict(preset="chip"), True), ("pe_q0d", dict(preset="", mapq_threshold=0, remove_pcr_duplicates=1, tn5_shift=1), True),
                                            ("se_q0d", dict(preset="", mapq_threshold=0, remove_pcr_duplicates=1, tn5_shift=1), False)])
def test_host_paf_writer_reproduces_reference_text(golden_dir, tmp_path, case, kw, paired):
    """cmx_format_paf is host code over the BED-path records (the device's == the oracle's, checked in the gpu tests): with the
    read names and lengths it writes the reference binary's --PAF file byte for byte, field quirks included; the oracle's own PAF
    writer (orc_run_files_paf) agrees."""
    import gzip
    import numpy as np
    import chromap_b200 as cb
    from oracle import oracle_py as orc
    from tests.util import load_pairs, read_fasta, read_fastq_records
    d = os.path.join(golden_dir, "synth_small")
    names, seqs = read_fasta(os.path.join(d, "ref.fa.gz"))
    ref = orc.Reference(os.path.join(d, "ref.fa.gz"))
    idx = orc.Index(ref=ref, k=17, w=7)
    s1, o1, s2, o2 = load_pairs(d)
    kw = dict(kw)
    preset = kw.pop("preset")
    op = orc.make_params(preset, **kw)
    recs = orc.map_pairs(op, idx, ref, s1, o1, s2, o2)[0] if paired else orc.map_reads_se(op, idx, ref, s1, o1)
    r1 = read_fastq_records(os.path.join(d, "read1.fq.gz"))
    r2 = read_fastq_records(os.path.join(d, "read2.fq.gz")) if paired else None
    p = cb.make_params(preset, max_read_length=64, single_end=0 if paired else 1, **kw)
    text = cb.format_paf(p, names, [len(s) for s in seqs], recs.view(cb.PE_RECORD), [a for a, _, _ in r1], [len(b) for _, b, _ in r1],
                         [a for a, _, _ in r2] if paired else None, [len(b) for _, b, _ in r2] if paired else None)
    want = gzip.open(os.path.join(d, case + ".paf.gz")).read()
    assert text == want
    ip = str(tmp_path / "ref.index")
    idx.save(ip)
    out = str(tmp_path / "o.paf")
    orc.run_files_paf(op, ip, os.path.join(d, "ref.fa.gz"), os.path.join(d, "read1.fq.gz"), os.path.join(d, "read2.fq.gz") if paired else None, out)
    assert open(out, "rb").read() == want
