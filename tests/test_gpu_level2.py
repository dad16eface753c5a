"""GPU: INTEGRATION.md "Level 2" end to end -- oracle/_ref/megagta_level2 (the reference's own option parser, loader and
SdbgWriter around the C ABI, integration/level2_build_graph.cpp) builds the golden cases and its files are compared with the
goldens of the unmodified reference.  The program is compiled from the reference's sources (oracle/Makefile), so the test
skips where they are absent; its CPU half is tests/test_level2_integration_cpu.py."""
import os
import subprocess

import pytest

from megagta_b200 import sdbg_io
from oracle import oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEVEL2 = os.path.join(ROOT, "oracle", "_ref", "megagta_level2")


@pytest.mark.parametrize("variant", ["", "_raw"])      # SdbgWriter::write per record / append_raw per delivery (patched tree)
@pytest.mark.parametrize("case", ["smoke_k31_m2", "adversarial_k27_m3"])
def test_level2_writes_the_reference_files(case, variant, golden, read_lib, tmp_path):
    if not os.path.exists(LEVEL2 + variant):
        pytest.skip("oracle/_ref/megagta_level2%s not built" % variant)
    g = golden["cases"][case]
    prefix, _ = read_lib(g["dataset"])
    out = str(tmp_path / "g")
    r = subprocess.run([LEVEL2 + variant, "buildgraph", "-k", str(g["k"]), "-m", str(g["m"]), "--host_mem", "4e9", "--num_cpu_threads", "4",
                        "--num_output_threads", "1", "--read_lib_file", prefix, "--output_prefix", out], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    hdr, stream, meta = sdbg_io.canonical(out)
    assert hdr["total_size"] == g["total_size"] and hdr["num_tips"] == g["num_tips"] and hdr["large_multi"] == g["large_multi"]
    assert O.stream_hash(stream) == g["stream_hash"] and O.meta_hash(meta) == g["meta_hash"]
