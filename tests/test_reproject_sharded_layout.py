"""cg_reproject_sharded_stats as the C compiler lays it out equals the ctypes struct (no GPU)."""
import ctypes as C
import os
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reproject_sharded_stats_layout():
    from coxgraph_b200 import capi
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "coxgraph_b200.h"\n'
           'int main(void){printf("%zu %zu %zu\\n", sizeof(cg_reproject_sharded_stats),'
           'offsetof(cg_reproject_sharded_stats, blocks_dirty),'
           'offsetof(cg_reproject_sharded_stats, full_rebuild));return 0;}')
    with tempfile.TemporaryDirectory() as d:
        with open(os.path.join(d, "s.c"), "w") as f:
            f.write(src)
        subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"),
                               os.path.join(d, "s.c"), "-o", os.path.join(d, "s")])
        size, off_dirty, off_full = (int(x) for x in
                                     subprocess.check_output([os.path.join(d, "s")]).split())
    S = capi.ReprojectShardedStats
    assert size == C.sizeof(S) == 56
    assert off_dirty == S.blocks_dirty.offset and off_full == S.full_rebuild.offset
