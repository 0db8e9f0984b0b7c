"""The FLOP numerators of bench.py's tensor-core roofline are constants taken from SURVEY App. D.  This test checks them
against the numbers measured on the REFERENCE's own modules (forward hooks on every nn.Conv2d, one image, CPU; stored in
tests/golden/bench_flops_reference.npz by make_golden_reference_state.py) and checks the expressions bench.py evaluates:
dense-conv FLOPs = 2 x MACs of the forward pass; per step what is actually executed (bench.py comments)."""
import os
import re

import numpy as np

from conftest import GOLDEN, ROOT


def test_bench_flop_constants_match_the_reference_modules():
    src = open(os.path.join(ROOT, "bench.py")).read()
    r = {k: float(v) for k, v in np.load(os.path.join(GOLDEN, "bench_flops_reference.npz")).items()}
    g256, d256, f256 = r["g256"], r["d256"], r["d_first256"]
    g512, d512, f512 = r["g512"], r["d512"], r["d_first512"]
    rec, rec_first = r["recon"], r["recon_first"]
    # cfg3: G step 3G + 2D, two D steps G + 6D each, minus the unexecuted first-layer input gradients of the 2B batch
    m = re.search(r"gf_img = (\(3 \* 17\.09 .*\))\n", src)
    assert m, "cfg3 FLOP expression not found in bench.py"
    want = (3 * g256 + 2 * d256) + 2 * (g256 + 6 * d256 - 2 * f256)
    assert abs(eval(m.group(1)) - want) < 2e-3 * want, (eval(m.group(1)), want)
    # cfg5 / cfg4 on one line: recon 3 x fwd - first-layer dgrad; 512^2 GAN as above
    m = re.search(r"gf_img = (3 \* 12\.21 - 0\.21) if cfg\[\"kind\"\] == \"recon\" else (\(3 \* 66\.56 .*\))\n", src)
    assert m, "cfg4 / cfg5 FLOP expression not found in bench.py"
    want4 = 3 * rec - rec_first
    assert abs(eval(m.group(1)) - want4) < 3e-3 * want4, (eval(m.group(1)), want4)
    want5 = (3 * g512 + 2 * d512) + 2 * (g512 + 6 * d512 - 2 * f512)
    assert abs(eval(m.group(2)) - want5) < 2e-3 * want5, (eval(m.group(2)), want5)
