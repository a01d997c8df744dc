"""Tuning sweeps: builds variant libraries (different -D geometry) under build/variants/.
Dev tooling only; the product library is always libdeflate_b200/libdeflate_b200.so."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from libdeflate_b200 import build as b  # noqa: E402

GEO_A = ["-DINF_LB=8", "-DINF_LSUB_SM=64", "-DINF_OB=6", "-DINF_OSUB_SM=64"]      # 896 B/lane, 7 warps/SM (default)
GEO_G = ["-DINF_LB=7", "-DINF_LSUB_SM=96", "-DINF_OB=6", "-DINF_OSUB_SM=64"]      # 704 B, 9 warps
GEO_C = ["-DINF_LB=7", "-DINF_LSUB_SM=64", "-DINF_OB=5", "-DINF_OSUB_SM=32"]      # 512 B, 13 warps
GEO_D = ["-DINF_LB=7", "-DINF_LSUB_SM=32", "-DINF_OB=5", "-DINF_OSUB_SM=32"]      # 448 B, 15 warps
VARIANTS = {
    # decode table geometries at 448 B per lane (offline count of global overflow lookups per lane-step on the bench corpus:
    # default 0.35 %, g6 0.20 %, o5s48l16 0.22 %): g6 = -DINF_LSUB_SM=16 -DINF_OB=6 -DINF_OSUB_SM=16 16.73 ms,
    # o5s48l16 = -DINF_LSUB_SM=16 -DINF_OB=5 -DINF_OSUB_SM=48 16.68 ms vs 16.54 ms default -- dropped
    "timing": ["-DLZ_TIMING"],
    # decode step, follow-on literals (INF_LIT2) at 65536 x 64 KiB: 0 / 1 / 2 / 3 / 4 -> 16.5 / 14.3 / 13.1 / 12.6 / 12.5 ms;
    # with the two-slot asynchronous lookahead (-DINF_WQ2=1) 2 / 3 -> 13.8 / 13.0 ms (slower again)
    "nofuse": ["-DINF_FUSE_OFF=0"],     # offset decoded in its own step (as before call V)
    "fuse_lit3": ["-DINF_LIT2=2"],
    # call W, on top of the fused step (default 10.14 ms): lit6 10.28, g6 10.20, g6lit6 10.27 -- no difference
    "lit6": ["-DINF_LIT2=6"],           # up to six follow-on literals (default four)
    "g6": ["-DINF_LSUB_SM=16", "-DINF_OB=6", "-DINF_OSUB_SM=16"],      # 6-bit main offset table: more matches take the fused path
    "g6lit6": ["-DINF_LSUB_SM=16", "-DINF_OB=6", "-DINF_OSUB_SM=16", "-DINF_LIT2=6"],
    # deflate schedule (scripts/gpu_pipeline_ab.sh): serial, and the pipeline with N search warps (default 22)
    "ser": ["-DLZ_PIPELINE=0"],
    "sert": ["-DLZ_PIPELINE=0", "-DLZ_TIMING"],
    "a18": ["-DLZ_A_WARPS=18"],
    "a20": ["-DLZ_A_WARPS=20"],
    "a22": [],
    "a22t": ["-DLZ_TIMING"],
}
# cache-streaming hints for the token stream off / 24 resolve warps per SM: no change / 10.5 ms (default 9.0)
# decode kernel with more warps per SM (code lengths in global memory, smaller tables, register cap): 18 / 21 / 24 warps
# 20.8 / 18.6 / 17.1 ms vs 16.7 ms at 15 warps -- dropped
# deflate kernel at 16384 chunks (base 79.2 ms, ratio 0.3022): 512 threads per CTA 97.5 ms; runs of 8 positions 84.0 ms / 0.3038;
# runs of 8 + depth 32: 90.0 / 0.3028; depth 16: 73.8 / 0.3035 -- nothing that is faster at the same ratio
# decode kernel, offset table geometry: 6-bit main + 16 shared subtable entries at 14 warps per SM 17.5 ms (= default);
# 13-warp geometries 27-28 ms (65536 chunks no longer fit one wave of lanes)
# decode steps between service phases, -DINF_QUANTUM=128/384/1024: 17.4 / 17.5 / 17.6 ms
# resolve kernel, warps (= chunks) per SM, -DRES_PER_SM=8/16/24/32: 25.9 / 14.2 / 10.6 / 9.0 ms per 65536 x 64 KiB
# measured and dropped: resumable chain walk of the deflate search (-DLZ_QUANTUM=6/8/12): 86.9 / 86.4 / 84.3 ms vs 79.2 ms
# per 16384 chunks (profiles/r02_deflate_quantum_ab.md)


def main():
    outdir = os.path.join(ROOT, "build", "variants")
    os.makedirs(outdir, exist_ok=True)
    nvcc = "/usr/local/cuda/bin/nvcc"
    for name, defs in VARIANTS.items():
        objs = []
        for src in b.SOURCES:
            obj = os.path.join(outdir, "%s_%s.o" % (name, src.replace(".cu", "")))
            subprocess.check_call([nvcc] + [f for f in b.NVCC_FLAGS if f not in ("-Xptxas", "-v")] + defs + ["-c", os.path.join(b.CSRC, src), "-o", obj])
            objs.append(obj)
        so = os.path.join(outdir, "libdeflate_b200_%s.so" % name)
        subprocess.check_call([nvcc, "-shared", "-o", so] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static"])
        print(so)


if __name__ == "__main__":
    main()
