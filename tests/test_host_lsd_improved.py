"""-m "not gpu": host side of the frame-range centre-window description built from a device weight map
(bsub_set_frame_weight_map_dev): the symbol is exported, declared and bound, and its kernel builds without spills."""
import os
import re
import subprocess

from background_subtraction_b200 import _cabi as C
from background_subtraction_b200 import build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAME = "bsub_set_frame_weight_map_dev"


def test_symbol_is_exported_declared_and_bound():
    lib = C.load()
    assert hasattr(lib, NAME) and NAME in C.SIGNATURES
    hdr = open(os.path.join(ROOT, "include", "bsub_b200.h")).read()
    assert re.search(r"int\s+%s\(bsub_solver\* s, int32_t rows, int32_t cols, int32_t f0, int32_t nf, const float\* weight, int64_t ld,"
                     r"\s*void\* stream\);" % NAME, hdr)


def test_weight_map_kernel_does_not_spill(tmp_path):
    src = os.path.join(build.CSRC, "mask.cu")
    cmd = [build.NVCC] + build.ARCH_FLAGS + [f for f in build.COMMON if not f.startswith("--use_fast_math")] + \
        ["-Xptxas", "-v", "-c", src, "-o", str(tmp_path / "mask.o")]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, check=True).stdout
    props = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", out)
    mine = [p for p in props if "weight_map_describe_kernel" in p[0]]
    assert mine, out
    for name, stack, st, ld in mine:
        assert (int(stack), int(st), int(ld)) == (0, 0, 0), (name, stack, st, ld)
