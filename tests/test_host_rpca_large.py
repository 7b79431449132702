"""-m "not gpu": host side of the stage-2 saliency batch's global-memory kernel (csrc/rpca_batch.cu): it builds without spills, and
a slice beyond its 4096 x 4096 limit is rejected by the C entry point before anything is launched."""
import ctypes
import os
import re
import subprocess

import pytest

from background_subtraction_b200 import _cabi as C
from background_subtraction_b200 import build


def test_rpca_batch_kernels_do_not_spill(tmp_path):
    """Both saliency RPCA kernels keep their state in registers, shared and global memory (no local-memory stack or spills)."""
    src = os.path.join(build.CSRC, "rpca_batch.cu")
    cmd = [build.NVCC] + build.ARCH_FLAGS + [f for f in build.COMMON if not f.startswith("--use_fast_math")] + \
        ["-Xptxas", "-v", "-c", src, "-o", str(tmp_path / "rpca_batch.o")]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, check=True).stdout
    props = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", out)
    names = [p[0] for p in props]
    assert any("rpca_rank1_large_kernel" in n for n in names) and any("rpca_rank1_batch_kernel" in n for n in names), out
    for name, stack, st, ld in props:
        assert (int(stack), int(st), int(ld)) == (0, 0, 0), (name, stack, st, ld)


@pytest.mark.parametrize("rows,cols", [(4097, 700), (100, 4097), (5000, 5000)])
def test_rpca_batch_rejects_slices_over_the_limit(rows, cols):
    """Dummy non-NULL pointers: the shape check fails first, so nothing is dereferenced or launched."""
    lib = C.load()
    p = ctypes.c_void_p(256)
    rc = lib.bsub_rpca_rank1_batch_dev(p, 3, rows, cols, 1.0, 1.2, 1e-7, 0.0, 10, p, p, p, p, p, None)
    assert rc != 0
    assert "larger than 4096 x 4096" in lib.bsub_last_error().decode()
