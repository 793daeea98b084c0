"""IMAD-pipe budget of the Bandersnatch verify kernels (tools/sass_imad_budget.py), read from the built library's SASS.

The two kernels are bound by the integer-multiply pipe.  The reduction rows of the BLS12-381 Fr product and square issue as
fused IMAD.WIDE.U32.X with immediate moduli, and their low limb pair comes from borrow chains on the ALU (arith.cuh RedRows);
a change that splits the rows back into IMAD.X + IMAD.HI.U32.X pairs, or puts more moves and carry additions on the pipe,
fails here before any GPU time is spent.  Limits: the figures of the build that introduced this test plus 3 %."""
import json
import os
import shutil
import subprocess
import sys
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "ark_ec_vrfs_b200", "libvrfs_b200.so")
TOOL = os.path.join(ROOT, "tools", "sass_imad_budget.py")

# per item: (multiplying, non-multiplying) IMAD-pipe instructions
LIMITS = {"<2,0>": (264462, 99382), "<1,1>": (189050, 88437)}
MARGIN = 1.03


def _cuobjdump():
    return next((c for c in (os.environ.get("CUOBJDUMP"), "/usr/local/cuda/bin/cuobjdump", shutil.which("cuobjdump")) if c and os.path.exists(c)), None)


@pytest.mark.skipif(_cuobjdump() is None, reason="cuobjdump not available")
def test_verify_kernels_imad_budget():
    if not os.path.exists(LIB):
        pytest.skip("library not built")
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "budget.json")
        subprocess.run([sys.executable, TOOL, LIB, "--json", out], check=True, stdout=subprocess.DEVNULL)
        got = json.load(open(out))["kernels"]
    for label, (mult, nonmult) in LIMITS.items():
        p = got[label]["per_item"]
        assert p["imad_mult"] <= mult * MARGIN, (label, p)
        assert p["imad_nonmult"] <= nonmult * MARGIN, (label, p)
        # the reduction rows stay fused: no IMAD.HI.U32.X left in the product and the square
        for fn in ("mont_mul_call<BlsFr>", "mont_sqr_call<BlsFr>"):
            assert "IMAD.HI.U32.X" not in got[label]["functions"][fn]["forms"], (label, fn)
