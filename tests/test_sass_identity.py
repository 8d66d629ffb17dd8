"""The colour-only kernels that gained a depth / alpha template parameter (blend_fwd2_kernel<false>,
blend_bwd2_kernel<512,false>, blend_bwd2_kernel<256,false>, preprocess_bwd_kernel<false>) compile to the same
instructions as before they had it.  The reference listing (tests/golden/colour_kernels_sass.txt.gz, written by
tests/golden/make_blend_sass_reference.py from the commit before the change) records the nvcc that produced it; with
another nvcc the comparison says nothing, so the test skips."""
import gzip
import os

import pytest

from splatco_b200 import _lib
from splatco_b200.build import _nvcc
from tests import sass_listing as S

REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "colour_kernels_sass.txt.gz")


def test_colour_kernels_are_instruction_identical_to_the_reference_listing():
    if not S.tools_available():
        pytest.skip("cuobjdump / c++filt not on PATH")
    text = gzip.open(REF, "rt").read()
    ref_nvcc = "\n".join(ln[2:] for ln in text.splitlines() if ln.startswith("# "))
    here = S.nvcc_version(_nvcc())
    if here != ref_nvcc:
        pytest.skip(f"the library was built with another nvcc ({here!r}) than the reference listing ({ref_nvcc!r})")
    want = S.parse(text)
    got = S.listings(_lib.LIB_PATH)
    assert set(want) == set(S.KERNELS) and set(got) == set(S.KERNELS), (sorted(want), sorted(got))
    for k in sorted(S.KERNELS):
        a, b = got[k], want[k]
        if a != b:
            i = next((i for i, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
            pytest.fail(f"{k}: {len(a)} instructions, reference {len(b)}; first difference at {i}: "
                        f"{a[i] if i < len(a) else '<end>'!r} vs {b[i] if i < len(b) else '<end>'!r}")
