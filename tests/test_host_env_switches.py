"""-m "not gpu": the library's environment switches and the kernels the shrink and prox sources compile to.

Every environment variable the library reads is a fallback switch the tests compare against, a resource cap, or a name
bench.py reads (DESIGN.md section 4.8); a kernel variant that only a variable could select is not compiled in."""
import glob
import os
import re
import subprocess

from background_subtraction_b200 import build

KEPT_SWITCHES = {
    "BSUB_NO_FLAT", "BSUB_NO_PROJ", "BSUB_NO_I8", "BSUB_NO_STREAM",    # fast paths against their fallbacks (GPU tests)
    "BSUB_NO_EIG_FAST",                                                # full eigensolver as the parity reference
    "BSUB_GRAPH_XI_MB",                                                # dual workspace cap of the graph prox kernels
    "BSUB_NO_GRAM_CLUSTER",                                            # read by bench.py to name the Gram kernel
}

ENTRIES = {
    "shrink_flat.cu": ["bsub::rebuild_S_done_kernel", "bsub::rebuild_S_kernel", "bsub::shrink_flat_kernel<0>", "bsub::shrink_flat_kernel<2>"],
    "shrink_stream.cu": ["bsub::shrink_stream_kernel<0, 0>", "bsub::shrink_stream_kernel<48, 28>"],
    "shrink_tma.cu": ["bsub::shrink_tma_kernel"],
    "prox.cu": ["bsub::block_l2_apply_kernel", "bsub::block_l2_sums_kernel", "bsub::prox_copy_through_kernel", "bsub::prox_flat3_kernel",
                "bsub::prox_graph3_tile_kernel", "bsub::prox_groups_csr_kernel", "bsub::prox_l1_kernel"],
}


def test_library_reads_only_the_kept_switches():
    names = set()
    for path in glob.glob(os.path.join(build.CSRC, "*.cu")) + glob.glob(os.path.join(build.CSRC, "*.cuh")) + \
            glob.glob(os.path.join(build.CSRC, "*.h")):
        with open(path) as f:
            names |= set(re.findall(r'getenv\(\s*"([^"]+)"\s*\)', f.read()))
    assert names == KEPT_SWITCHES


def _ptxas(tmp_path, src):
    cmd = [build.NVCC] + build.ARCH_FLAGS + [f for f in build.COMMON if not f.startswith("--use_fast_math")] + \
        ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, src), "-o", str(tmp_path / (src + ".o"))]
    return subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)


def _demangle(names):
    filt = os.path.join(os.path.dirname(build.NVCC), "cu++filt")
    out = subprocess.run([filt], input="\n".join(names) + "\n", stdout=subprocess.PIPE, text=True, check=True).stdout.split("\n")
    return {n: re.sub(r"^void ", "", d.replace("(int)", "").split("(")[0]) for n, d in zip(names, out)}


def test_shrink_and_prox_kernels_are_the_ones_launched_and_shrink_kernels_do_not_spill(tmp_path):
    procs = {src: _ptxas(tmp_path, src) for src in ENTRIES}
    for src, p in procs.items():
        out, _ = p.communicate()
        assert p.returncode == 0, out
        entries = re.findall(r"Compiling entry function '(\S+)'", out)
        props = dict((m[0], m[1:]) for m in re.findall(
            r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", out))
        names = _demangle(entries)
        assert sorted(names.values()) == ENTRIES[src], out
        for mangled, name in names.items():
            if name.startswith("bsub::shrink_"):
                assert tuple(int(v) for v in props[mangled]) == (0, 0, 0), (name, props[mangled])
