"""Drop-in for the reference's scripts/read_recruitment/rr binary: `python rr.py unit.fasta reads.fasta[.gz] output.fasta
edit_distance_threshold` (run_read_recruitment.sh calls `$SCRIPT_DIR/rr` with exactly these four arguments).  Besides
the reference's FASTA / FASTQ, plain or gzip, the reads may be bgzip-compressed or unaligned BAM (BGZF files are
inflated on the GPU).  The usage text on stdout is rr.cpp's; a note on the accepted read files goes to stderr."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from centroflye_b200.read_recruitment import main  # noqa: E402

if __name__ == "__main__":
    sys.exit(main())
