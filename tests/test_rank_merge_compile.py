"""The kernels that evaluate sharded document sets (global candidate ids, the merge of rankings, the curve points;
gcgcn_b200/csrc/rank.cu) compile for sm_100a without local memory.  No GPU needed."""
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_KERNELS = ("rank_candidates_at_kernel", "merge_partition_kernel", "merge_tile_kernel", "curve_points_kernel")


def test_new_rank_kernels_compile_without_local_memory():
    """-Xptxas -v: no stack frame and no spills in the new kernels."""
    src = os.path.join(ROOT, "gcgcn_b200", "csrc", "rank.cu")
    out = subprocess.run([os.environ.get("NVCC", "nvcc"), "-gencode", "arch=compute_100a,code=sm_100a", "-O3",
                          "-std=c++17", "-I", os.path.join(ROOT, "include"), "-Xptxas", "-v", "-c", "-o", os.devnull,
                          src], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    frames = {}
    name = None
    for line in out.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            name = m.group(1)
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name is not None:
            frames[name] = m.groups()
    for kernel in NEW_KERNELS:
        hits = [v for k, v in frames.items() if kernel in k]
        assert len(hits) == 1, (kernel, sorted(frames))
        assert hits[0] == ("0", "0", "0"), (kernel, hits[0])
