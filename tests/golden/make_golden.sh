#!/bin/bash
# Regenerates tests/golden/ from the UNMODIFIED reference binary (oracle/_ref/chromap, built by
# oracle/Makefile from /root/reference).  Run in the build container only.  Outputs are committed.
set -e
cd "$(dirname "$0")"
REPO=$(cd ../.. && pwd)
REF=$REPO/oracle/_ref/chromap
rm -rf synth_small && mkdir -p synth_small
python $REPO/tools/gen_synth.py --out synth_small --seed 11 --n-seq 3 --seq-len 300000 --n-pairs 6000 \
  --repeat-copies 20 --repeat-len 2000 --fam-copies 700 --short-frac 0.3 --lowercase-frac 0.05
cd synth_small
$REF -i -r ref.fa -o ref.index 2> /dev/null
run() { name=$1; shift; $REF "$@" -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o $name.bed -t 1 2> /dev/null; }
run chip --preset chip
run atac --preset atac
run default
run q0dedup --remove-pcr-duplicates -q 0
run e5 -e 5 -q 10 --Tn5-shift --remove-pcr-duplicates
run e12l300 -e 12 -l 300 -q 0
run n3q0 -n 3 -q 0
$REF --preset chip --TagAlign -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o chip.tagalign -t 1 2> /dev/null
# single-end (read 1 only)
runse() { name=$1; shift; $REF "$@" -x ref.index -r ref.fa -1 read1.fq -o $name.bed -t 1 2> /dev/null; }
runse se_default
runse se_chip --preset chip
runse se_q0dedup_tn5 -q 0 --remove-pcr-duplicates --Tn5-shift
runse se_n3q0 -n 3 -q 0
runse se_lowmem_q0 --low-mem -q 0 --remove-pcr-duplicates --Tn5-shift
# SAM (oracle groundwork for the round-2 CUDA path)
$REF --preset chip --SAM -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o pe_chip.sam -t 1 2> /dev/null
$REF -q 0 --remove-pcr-duplicates --SAM -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o pe_q0d.sam -t 1 2> /dev/null
$REF -n 3 -q 0 --SAM -x ref.index -r ref.fa -1 read1.fq -o se_n3.sam -t 1 2> /dev/null
# PAF (host writer over the BED-path records)
$REF --preset chip --PAF -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o pe_chip.paf -t 1 2> /dev/null
$REF -q 0 --remove-pcr-duplicates --Tn5-shift --PAF -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o pe_q0d.paf -t 1 2> /dev/null
$REF -q 0 --remove-pcr-duplicates --Tn5-shift --PAF -x ref.index -r ref.fa -1 read1.fq -o se_q0d.paf -t 1 2> /dev/null
md5sum *.bed > md5.txt
gzip -9 -n ref.fa read1.fq read2.fq *.bed chip.tagalign *.sam *.paf
rm -f ref.index
# the reference's own test data (README quick start): golden BEDs for SURVEY.md §4's md5s
cd .. && rm -rf ref_test && mkdir ref_test && cd ref_test
T=/root/reference/test
cp $T/ref.fa $T/read1.fq $T/read2.fq .
$REF -i -r ref.fa -o ref.index 2> /dev/null
$REF -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o default.bed -t 1 2> /dev/null
$REF --preset chip -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o chip.bed -t 1 2> /dev/null
$REF --preset atac -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o atac.bed -t 1 2> /dev/null
$REF --preset hic -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o hic.pairs -t 1 2> /dev/null
md5sum default.bed chip.bed atac.bed hic.pairs ref.index > md5.txt
gzip -9 -n ref.fa
# Hi-C (--preset hic: split alignment, pairs output): 2x150 bp with chimeric reads
cd .. && rm -rf synth_hic && mkdir -p synth_hic
python $REPO/tools/gen_synth.py --out synth_hic --seed 12 --n-seq 3 --seq-len 250000 --n-pairs 3000 --read-len 150 \
  --chimeric-frac 0.3 --repeat-copies 15 --repeat-len 2000 --fam-copies 500
cd synth_hic
$REF -i -r ref.fa -o ref.index 2> /dev/null
$REF --preset hic -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o hic.pairs -t 1 2> /dev/null
$REF --preset hic -q 0 -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o hic_q0.pairs -t 1 2> /dev/null
$REF --preset hic -q 0 -e 6 --remove-pcr-duplicates -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -o hic_e6dedup.pairs -t 1 2> /dev/null
md5sum *.pairs > md5.txt
gzip -9 -n ref.fa read1.fq read2.fq *.pairs
rm -f ref.index
# scATAC (--preset atac with -b / --barcode-whitelist): barcodes with substitutions, Ns and near-neighbour whitelist entries
cd .. && rm -rf synth_sc && mkdir -p synth_sc
python $REPO/tools/gen_synth.py --out synth_sc --seed 13 --n-seq 3 --seq-len 250000 --n-pairs 5000 --short-frac 0.3 --barcodes \
  --repeat-copies 15 --repeat-len 2000 --fam-copies 500
python $REPO/tools/perturb_barcodes.py synth_sc
cd synth_sc
$REF -i -r ref.fa -o ref.index 2> /dev/null
$REF --preset atac -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -b barcode.fq --barcode-whitelist whitelist.txt -o sc_whitelist.bed -t 1 2> sc.log
$REF --preset atac -x ref.index -r ref.fa -1 read1.fq -2 read2.fq -b barcode.fq -o sc_nowhitelist.bed -t 1 2> /dev/null
grep -E "Number of (barcodes|corrected)" sc.log > sc_stats.txt; rm sc.log
# single-end reads with barcodes (MappingWithBarcode)
$REF --preset atac -x ref.index -r ref.fa -1 read1.fq -b barcode.fq --barcode-whitelist whitelist.txt -o se_sc_whitelist.bed -t 1 2> /dev/null
$REF --preset atac -x ref.index -r ref.fa -1 read1.fq -b barcode.fq -o se_sc_nowhitelist.bed -t 1 2> /dev/null
$REF -q 0 --remove-pcr-duplicates --Tn5-shift -x ref.index -r ref.fa -1 read1.fq -b barcode.fq --barcode-whitelist whitelist.txt -o se_sc_inmem.bed -t 1 2> /dev/null
md5sum *.bed > md5.txt
gzip -9 -n ref.fa read1.fq read2.fq barcode.fq *.bed
rm -f ref.index
# what `chromap -i` writes, as digests (the index files themselves are too large to store)
python $REPO/tests/golden/make_index_digests.py
