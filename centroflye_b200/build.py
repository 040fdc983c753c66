"""Build centroflye_b200/libcfk.so for sm_100a:  python -m centroflye_b200.build [--force]"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "cfk.cu")
INGEST_SRC = os.path.join(HERE, "csrc", "ncrf_ingest.cpp")  # host-side NCRF ingestion, same library
WRITER_SRC = os.path.join(HERE, "csrc", "result_writer.cpp")  # host-side edge file writer, same library
STREAM_SRC = os.path.join(HERE, "csrc", "docfreq_stream.cu")  # stage A, two-phase form (emit + apply)
PLACER_SRC = os.path.join(HERE, "csrc", "placer.cu")  # read_placer scoring on the cloud CSR (row f rank 2)
RR_SRC = os.path.join(HERE, "csrc", "rr_filter.cu")  # read recruitment pre-filter (row f rank 4)
SCAN_SRC = os.path.join(HERE, "csrc", "seq_scan.cpp")  # host-side FASTA / FASTQ record scanner of the streaming filter
BGZF_SRC = os.path.join(HERE, "csrc", "bgzf.cu")  # BGZF blocks inflated on the device (compressed read files)
BAM_SCAN_SRC = os.path.join(HERE, "csrc", "bam_scan.cpp")  # host-side BGZF block finder and BAM record scanner
COMMON_HDR = os.path.join(HERE, "csrc", "cfk_common.cuh")
SOURCES = [SRC, STREAM_SRC, PLACER_SRC, RR_SRC, BGZF_SRC, INGEST_SRC, WRITER_SRC, SCAN_SRC, BAM_SCAN_SRC]
HDR = os.path.join(os.path.dirname(HERE), "include", "cfk.h")
OUT = os.path.join(HERE, "libcfk.so")

NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-shared", "-Xcompiler", "-fPIC,-pthread"]


def nvcc_path():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built")


def up_to_date():
    return os.path.exists(OUT) and os.path.getmtime(OUT) >= max(os.path.getmtime(HDR), os.path.getmtime(COMMON_HDR), *(os.path.getmtime(p) for p in SOURCES))


def build(force=False, verbose=False):
    if not force and up_to_date():
        return OUT
    cmd = [nvcc_path()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", OUT] + SOURCES
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return OUT


def build_variant(tag, defines):
    """Tuning experiments: gpurun_tmp_libcfk_<tag>.so at the repo root with extra -D flags (loaded via CFK_LIBRARY)."""
    out = os.path.join(os.path.dirname(HERE), f"gpurun_tmp_libcfk_{tag}.so")
    cmd = [nvcc_path()] + NVCC_FLAGS + [f"-D{d}" for d in defines] + ["-o", out] + SOURCES
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
