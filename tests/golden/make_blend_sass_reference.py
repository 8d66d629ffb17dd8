"""Writes tests/golden/colour_kernels_sass.txt.gz: the normalised SASS of the colour-only blend and
preprocess-backward kernels, which tests/test_sass_identity.py holds the current build to.

    python tests/golden/make_blend_sass_reference.py OBJ_OR_LIB [OBJ_OR_LIB ...]

The inputs are objects (or libsplatco_b200.so) built with splatco_b200/build.py's nvcc flags from the commit
whose kernels are the reference; the listing records that nvcc's version.  It was generated from the commit
before the depth / alpha kernels were added, so the test shows that adding them left the colour path's
machine code unchanged."""
import gzip
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from tests.sass_listing import KERNELS, dump, listings, nvcc_version  # noqa: E402

OUT = os.path.join(HERE, "colour_kernels_sass.txt.gz")


def main(paths):
    lst = {}
    for p in paths:
        lst.update(listings(p))
    missing = set(KERNELS) - set(lst)
    assert not missing, f"kernels not found: {sorted(missing)}"
    text = "".join(f"# {ln}\n" for ln in nvcc_version().splitlines()) + dump(lst)
    with gzip.GzipFile(OUT, "wb", mtime=0) as f:
        f.write(text.encode())
    print(OUT, {k: len(v) for k, v in sorted(lst.items())})


if __name__ == "__main__":
    main(sys.argv[1:])
