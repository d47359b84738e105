"""Builds the in-tree CUDA library `nanosnp_b200/libnanosnp_b200.so` for sm_100a with nvcc.

The library is a plain C-ABI shared object (include/nanosnp_b200.h); it is loaded with ctypes and never
falls back to a CPU path.  nvcc cross-compiles without a GPU, so this runs in the build container.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent
CSRC = ROOT / "csrc"
LIB = ROOT / "libnanosnp_b200.so"
SOURCES = ["api.cu", "synth.cu", "pileup.cu", "select.cu", "model.cu", "model_tc.cu", "vcf.cu", "vcf_dev.cu", "bam.cu", "bam_stream.cu", "record.cu", "haplotype.cu", "haplotype_tc.cu", "hap_groups.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17", "--expt-relaxed-constexpr", "--extended-lambda",
    "-Xcompiler", "-fPIC,-O3,-Wall,-Wno-unused-function",
    "-Xptxas", "-v",
]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built (there is no CPU fallback)")


def needs_build() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = list(CSRC.glob("*")) + [ROOT.parent / "include" / "nanosnp_b200.h", Path(__file__)]
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return LIB
    nvcc = nvcc_path()
    objdir = ROOT / "build"
    objdir.mkdir(exist_ok=True)
    srcs = [s for s in SOURCES if (CSRC / s).exists()]
    procs = []
    for s in srcs:
        obj = objdir / (Path(s).stem + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(CSRC / s), "-o", str(obj)]
        procs.append((s, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    log = []
    for s, obj, p in procs:
        out, _ = p.communicate()
        log.append(f"== {s}\n{out}")
        if p.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {s}")
        objs.append(str(obj))
    (objdir / "ptxas.log").write_text("\n".join(log))
    if verbose:
        print("\n".join(log))
    cmd = [nvcc, "-shared", "-o", str(LIB), *objs, "-lcudart", "-lcuda", "-lpthread", "-lz"]
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
