"""Round trip of bench.py's workload against a variant library under build/variants/ (tuning and A/B runs only).
    python scripts/variant_roundtrip.py NAME [--level L] [--chunks N] [--chunk-size B] [--data-class C] [--steps K]
                                             [--dump-outputs DIR]
Prints bench.py's JSON line, then the deflate kernel's phase clocks if the variant was built with -DLZ_TIMING."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import libdeflate_b200 as ldb  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("name")
ap.add_argument("--level", type=int, default=6)
ap.add_argument("--chunks", type=int, default=65536)
ap.add_argument("--chunk-size", type=int, default=65536)
ap.add_argument("--data-class", type=int, default=0)
ap.add_argument("--steps", type=int, default=3)
ap.add_argument("--dump-outputs", default=None)
o = ap.parse_args()
ldb._lib = ldb.load_library(os.path.join(ROOT, "build", "variants", "libdeflate_b200_%s.so" % o.name))
import bench  # noqa: E402
bench.LEVEL = o.level
a = argparse.Namespace(gpus=1, steps=o.steps, warmup=2, impl="b200", workload="roundtrip", chunks=o.chunks, chunk_size=o.chunk_size,
                       level=o.level, no_e2e=True, no_cpu=True, no_extra=True, no_l12=True, no_origin=True, overlap=False,
                       data_class=o.data_class, dump_outputs=o.dump_outputs)
bench.run_b200(a)
try:
    ldb._lib.ldb_lz_timing_dump()
except AttributeError:
    pass
