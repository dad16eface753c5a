"""GPU: the CUDA path on the 52 seeded random read sets of tests/test_oracle_fuzz.py (ragged lengths, repeats, palindromes,
k = 9 ... 127 around every word boundary, m = 1 ... 3, mercy) against the oracle, which that file pins on the reference
binary run live.  Its CPU counterpart (the product's __host__ __device__ logic on the same inputs) is
tests/test_logic_cpu.py::test_product_logic_on_random_inputs."""
import numpy as np
import pytest

from megagta_b200 import cabi
from oracle import oracle as O

pytestmark = pytest.mark.gpu


def test_gpu_equals_the_oracle_on_random_inputs(tmp_path):
    import test_oracle_fuzz as F
    bad, ran = [], 0
    for seed in range(52):
        prefix, k, m, mercy, fa = F.make_case(seed, str(tmp_path))
        rd = O.load_read_lib(prefix)
        exp = O.build_graph(rd, k, m, mercy)
        if int(exp["meta"][:, 0].sum()) == 0:
            continue                      # no solid edge: the reference itself aborts on this input, there is no parity target
        ran += 1
        with cabi.Context(k, m, need_mercy=mercy) as ctx:
            ctx.set_reads(rd["seq"], rd["start"], max_len=rd["max_len"])
            ok = True
            if m > 1:
                n = O.solid_bytes(rd, k)
                ok = np.array_equal(ctx.stage1(), exp["counting"]) and np.array_equal(ctx.get_is_solid()[:n], exp["is_solid"][:n])
            stream, meta, totals = ctx.stage2()
        if not (ok and np.array_equal(meta, exp["meta"]) and np.array_equal(totals, exp["totals"]) and stream == exp["stream"]):
            bad.append((seed, k, m, mercy))
    assert ran >= 40 and not bad, bad
