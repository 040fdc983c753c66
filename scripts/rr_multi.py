"""rr for several units in one pass over the read file: `python rr_multi.py [--gpus N] reads.{fasta,fastq}[.gz]|reads.bam
unit1.fasta output1.fasta threshold1 [unit2.fasta output2.fasta threshold2 ...]` writes, for every triple, the file that
`rr unit.fasta reads output.fasta threshold` writes, reading and scanning the read file once.  The reads may be FASTA or
FASTQ, plain, gzip or bgzip, or unaligned BAM (BGZF files are inflated on the GPU).  With --gpus N the
records of every chunk are dealt out over cuda:0 .. N-1; the outputs are the same bytes."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from centroflye_b200.read_recruitment import main_units  # noqa: E402

if __name__ == "__main__":
    sys.exit(main_units())
