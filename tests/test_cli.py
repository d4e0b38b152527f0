"""The C++ front end (chromap_b200/bin/chromap-b200): reference CLI names, presets, index file format."""
import gzip
import hashlib
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "chromap_b200", "bin", "chromap-b200")


def _ensure_cli():
    if not os.path.exists(CLI):
        import __graft_entry__
        __graft_entry__.build()
    return CLI


def test_cli_rejects_unsupported_and_missing_gpu():
    cli = _ensure_cli()
    r = subprocess.run([cli, "--preset", "nope"], capture_output=True, text=True)
    assert r.returncode != 0 and "Unrecognized preset" in r.stderr
    r = subprocess.run([cli, "--summary", "-x", "a", "-r", "b"], capture_output=True, text=True)
    assert r.returncode != 0 and "not on the GPU path" in r.stderr
    import torch
    if not torch.cuda.is_available():
        d = os.path.join(ROOT, "tests", "golden", "ref_test")
        r = subprocess.run([cli, "-x", os.path.join(d, "ref.index"), "-r", os.path.join(d, "ref.fa.gz"), "-1", os.path.join(d, "read1.fq"),
                            "-2", os.path.join(d, "read2.fq"), "-o", "/tmp/never.bed"], capture_output=True, text=True)
        assert r.returncode != 0 and "no CPU fallback" in r.stderr
        for fmt in ("--SAM", "--PAF", "--TagAlign"):  # the other output formats parse and reach the same gate
            r = subprocess.run([cli, fmt, "-x", os.path.join(d, "ref.index"), "-r", os.path.join(d, "ref.fa.gz"), "-1", os.path.join(d, "read1.fq"),
                                "-2", os.path.join(d, "read2.fq"), "-o", "/tmp/never.out"], capture_output=True, text=True)
            assert r.returncode != 0 and "no CPU fallback" in r.stderr, (fmt, r.stderr)
        r = subprocess.run([cli, "--PAF", "--preset", "atac", "-x", os.path.join(d, "ref.index"), "-r", os.path.join(d, "ref.fa.gz"), "-1", os.path.join(d, "read1.fq"),
                            "-2", os.path.join(d, "read2.fq"), "-o", "/tmp/never.out"], capture_output=True, text=True)
        assert r.returncode != 0 and "adapter trimming" in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("case,args", [("chip", ["--preset", "chip"]), ("atac", ["--preset", "atac"]), ("default", []),
                                       ("q0dedup", ["--remove-pcr-duplicates", "-q", "0"]),
                                       ("e5", ["-e", "5", "-q", "10", "--Tn5-shift", "--remove-pcr-duplicates"]),
                                       ("e12l300", ["-e", "12", "-l", "300", "-q", "0"])])
def test_cli_end_to_end_equals_reference_binary_output(case, args, tmp_path, golden_dir):
    cli = _ensure_cli()
    d = os.path.join(golden_dir, "synth_small")
    idx = str(tmp_path / "ref.index")
    subprocess.check_call([cli, "-i", "-r", os.path.join(d, "ref.fa.gz"), "-o", idx], stderr=subprocess.DEVNULL)
    out = str(tmp_path / "out.bed")
    subprocess.check_call([cli] + args + ["-x", idx, "-r", os.path.join(d, "ref.fa.gz"), "-1", os.path.join(d, "read1.fq.gz"),
                                         "-2", os.path.join(d, "read2.fq.gz"), "-o", out], stderr=subprocess.DEVNULL)
    assert open(out, "rb").read() == gzip.open(os.path.join(d, case + ".bed.gz")).read()


@pytest.mark.gpu
def test_index_file_written_by_cli_is_loadable_by_the_reference_binary(tmp_path, golden_dir):
    """The file we write is what the unmodified reference's `chromap -i` writes for the same FASTA, up to the bucket order inside
    khash's arrays: the same header (k, w, kh_size, n_buckets, size, n_occupied, upper_bound), the same length, the same key ->
    value map and occurrence table (synth_small/ref_index.json holds the reference's side, tests/golden/make_index_digests.py).
    A reader of the format (the oracle's restatement of Index::Load) maps through it to the reference binary's BED."""
    import json
    import numpy as np
    from oracle import oracle_py as orc
    from tests.util import index_digest
    cli = _ensure_cli()
    d = os.path.join(golden_dir, "synth_small")
    want = json.load(open(os.path.join(d, "ref_index.json")))
    ref = str(tmp_path / "ref.fa")
    open(ref, "wb").write(gzip.open(os.path.join(d, "ref.fa.gz")).read())
    idx = str(tmp_path / "ref.index")
    subprocess.check_call([cli, "-i", "-r", ref, "-o", idx], stderr=subprocess.DEVNULL)
    raw = open(idx, "rb").read()
    assert len(raw) == want["file_bytes"]
    assert [int(x) for x in np.frombuffer(raw[:8], "<i4")] + [int(x) for x in np.frombuffer(raw[8:28], "<u4")] == want["header"]
    got = index_digest(orc.Index(idx).arrays())
    assert got == {f: want[f] for f in got}
    out = str(tmp_path / "ref_out.bed")
    orc.run_files(orc.make_params(""), idx, ref, os.path.join(d, "read1.fq.gz"), os.path.join(d, "read2.fq.gz"), out, n_threads=2)
    assert open(out, "rb").read() == gzip.open(os.path.join(d, "default.bed.gz")).read()


@pytest.mark.gpu
def test_cli_hic_preset_pairs_output(tmp_path, golden_dir):
    cli = _ensure_cli()
    d = os.path.join(golden_dir, "synth_hic")
    idx = str(tmp_path / "ref.index")
    subprocess.check_call([cli, "-i", "-r", os.path.join(d, "ref.fa.gz"), "-o", idx], stderr=subprocess.DEVNULL)
    for case, args in (("hic", []), ("hic_q0", ["-q", "0"]), ("hic_e6dedup", ["-q", "0", "-e", "6", "--remove-pcr-duplicates"])):
        out = str(tmp_path / (case + ".pairs"))
        subprocess.check_call([cli, "--preset", "hic"] + args + ["-x", idx, "-r", os.path.join(d, "ref.fa.gz"), "-1", os.path.join(d, "read1.fq.gz"),
                                                                "-2", os.path.join(d, "read2.fq.gz"), "-o", out], stderr=subprocess.DEVNULL)
        assert open(out, "rb").read() == gzip.open(os.path.join(d, case + ".pairs.gz")).read()


@pytest.mark.gpu
def test_cli_scatac_barcodes(tmp_path, golden_dir):
    cli = _ensure_cli()
    d = os.path.join(golden_dir, "synth_sc")
    idx = str(tmp_path / "ref.index")
    subprocess.check_call([cli, "-i", "-r", os.path.join(d, "ref.fa.gz"), "-o", idx], stderr=subprocess.DEVNULL)
    for case, extra in (("sc_whitelist", ["--barcode-whitelist", os.path.join(d, "whitelist.txt"), "--cache-size", "1000", "--debug-cache", "-A", "1"]),
                        ("sc_nowhitelist", [])):
        out = str(tmp_path / (case + ".bed"))
        r = subprocess.run([cli, "--preset", "atac", "-x", idx, "-r", os.path.join(d, "ref.fa.gz"), "-1", os.path.join(d, "read1.fq.gz"),
                            "-2", os.path.join(d, "read2.fq.gz"), "-b", os.path.join(d, "barcode.fq.gz"), "-o", out] + extra, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert open(out, "rb").read() == gzip.open(os.path.join(d, case + ".bed.gz")).read()
        if extra:
            for line in open(os.path.join(d, "sc_stats.txt")):
                assert line.strip() in r.stderr
    # single-end reads with barcodes (MappingWithBarcode)
    out = str(tmp_path / "se_sc.bed")
    r = subprocess.run([cli, "--preset", "atac", "-x", idx, "-r", os.path.join(d, "ref.fa.gz"), "-1", os.path.join(d, "read1.fq.gz"),
                        "-b", os.path.join(d, "barcode.fq.gz"), "--barcode-whitelist", os.path.join(d, "whitelist.txt"), "-o", out], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(out, "rb").read() == gzip.open(os.path.join(d, "se_sc_whitelist.bed.gz")).read()


@pytest.mark.gpu
def test_cli_single_end(tmp_path, golden_dir):
    cli = _ensure_cli()
    d = os.path.join(golden_dir, "synth_small")
    idx = str(tmp_path / "ref.index")
    subprocess.check_call([cli, "-i", "-r", os.path.join(d, "ref.fa.gz"), "-o", idx], stderr=subprocess.DEVNULL)
    for case, extra in (("se_chip", ["--preset", "chip"]), ("se_q0dedup_tn5", ["-q", "0", "--remove-pcr-duplicates", "--Tn5-shift"]),
                        ("se_n3q0", ["-n", "3", "-q", "0"])):
        out = str(tmp_path / (case + ".bed"))
        r = subprocess.run([cli, "-x", idx, "-r", os.path.join(d, "ref.fa.gz"), "-1", os.path.join(d, "read1.fq.gz"), "-o", out] + extra,
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert open(out, "rb").read() == gzip.open(os.path.join(d, case + ".bed.gz")).read()


@pytest.mark.gpu
def test_cli_falls_back_to_the_host_reader_for_fasta_reads(tmp_path, golden_dir):
    """Reads given as FASTA (kseq accepts them) are not 4-line FASTQ: the device-side parser refuses them and the CLI
    switches to its host reader; --host-reader forces that path.  Same BED either way."""
    cli = _ensure_cli()
    d = os.path.join(golden_dir, "synth_small")
    idx = str(tmp_path / "ref.index")
    subprocess.check_call([cli, "-i", "-r", os.path.join(d, "ref.fa.gz"), "-o", idx], stderr=subprocess.DEVNULL)
    for which in ("read1", "read2"):
        lines = gzip.open(os.path.join(d, which + ".fq.gz")).read().split(b"\n")
        with open(str(tmp_path / (which + ".fa")), "wb") as f:
            for i in range(0, len(lines) - 3, 4):
                f.write(b">" + lines[i][1:] + b"\n" + lines[i + 1] + b"\n")
    want = gzip.open(os.path.join(d, "chip.bed.gz")).read()
    for reads, extra, note in (((str(tmp_path / "read1.fa"), str(tmp_path / "read2.fa")), [], "using the host reader"),
                               ((os.path.join(d, "read1.fq.gz"), os.path.join(d, "read2.fq.gz")), ["--host-reader"], None)):
        out = str(tmp_path / "out.bed")
        r = subprocess.run([cli, "--preset", "chip", "-x", idx, "-r", os.path.join(d, "ref.fa.gz"), "-1", reads[0], "-2", reads[1], "-o", out] + extra,
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert open(out, "rb").read() == want
        if note:
            assert note in r.stderr


@pytest.mark.gpu
def test_cli_tagalign(tmp_path, golden_dir):
    cli = _ensure_cli()
    d = os.path.join(golden_dir, "synth_small")
    idx = str(tmp_path / "ref.index")
    subprocess.check_call([cli, "-i", "-r", os.path.join(d, "ref.fa.gz"), "-o", idx], stderr=subprocess.DEVNULL)
    for reads, want in ((["-1", os.path.join(d, "read1.fq.gz"), "-2", os.path.join(d, "read2.fq.gz")], "chip.tagalign.gz"),
                        (["-1", os.path.join(d, "read1.fq.gz")], "se_chip.bed.gz")):  # single-end TagAlign text == BED text
        out = str(tmp_path / "out.txt")
        r = subprocess.run([cli, "--preset", "chip", "--TagAlign", "-x", idx, "-r", os.path.join(d, "ref.fa.gz"), "-o", out] + reads, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert open(out, "rb").read() == gzip.open(os.path.join(d, want)).read()


@pytest.mark.gpu
def test_cli_sam(tmp_path, golden_dir):
    cli = _ensure_cli()
    d = os.path.join(golden_dir, "synth_small")
    idx = str(tmp_path / "ref.index")
    subprocess.check_call([cli, "-i", "-r", os.path.join(d, "ref.fa.gz"), "-o", idx], stderr=subprocess.DEVNULL)
    for reads, extra, want in ((["-1", os.path.join(d, "read1.fq.gz"), "-2", os.path.join(d, "read2.fq.gz")], ["--preset", "chip"], "pe_chip.sam.gz"),
                               (["-1", os.path.join(d, "read1.fq.gz")], ["-n", "3", "-q", "0"], "se_n3.sam.gz")):
        out = str(tmp_path / "out.sam")
        r = subprocess.run([cli, "--SAM", "-x", idx, "-r", os.path.join(d, "ref.fa.gz"), "-o", out] + extra + reads, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert open(out, "rb").read() == gzip.open(os.path.join(d, want)).read()


@pytest.mark.gpu
@pytest.mark.parametrize("case,args,paired", [("pe_chip", ["--preset", "chip"], True), ("pe_q0d", ["-q", "0", "--remove-pcr-duplicates", "--Tn5-shift"], True),
                                              ("se_q0d", ["-q", "0", "--remove-pcr-duplicates", "--Tn5-shift"], False)])
def test_cli_paf_equals_reference_binary_output(case, args, paired, tmp_path, golden_dir):
    """--PAF through the GPU path end to end (records from the device, text by cmx_format_paf) == the reference binary's PAF."""
    cli = _ensure_cli()
    d = os.path.join(golden_dir, "synth_small")
    idx = str(tmp_path / "ref.index")
    subprocess.check_call([cli, "-i", "-r", os.path.join(d, "ref.fa.gz"), "-o", idx], stderr=subprocess.DEVNULL)
    out = str(tmp_path / "out.paf")
    reads = ["-1", os.path.join(d, "read1.fq.gz")] + (["-2", os.path.join(d, "read2.fq.gz")] if paired else [])
    subprocess.check_call([cli] + args + ["--PAF", "-x", idx, "-r", os.path.join(d, "ref.fa.gz")] + reads + ["-o", out], stderr=subprocess.DEVNULL)
    assert open(out, "rb").read() == gzip.open(os.path.join(d, case + ".paf.gz")).read()
