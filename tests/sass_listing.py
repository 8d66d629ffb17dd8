"""Normalised SASS listings of the colour-only blend / preprocess-backward kernels (used by
tests/test_sass_identity.py and tests/golden/make_blend_sass_reference.py).

A kernel's listing is its instruction text from `cuobjdump -sass`, one instruction per line, with the
addresses and the encoding comments stripped; the kernel's name is replaced by a stable key, so a kernel that
became a template (blend_fwd2_kernel -> blend_fwd2_kernel<false>) is compared with its former self."""
from __future__ import annotations

import re
import shutil
import subprocess

# key -> demangled-name pattern matching both the pre-template and the template spelling
KERNELS = {
    "blend_fwd2_kernel<false>": re.compile(r"splatco::blend_fwd2_kernel(<false>)?\("),
    "blend_bwd2_kernel<512,false>": re.compile(r"splatco::blend_bwd2_kernel<512(, false)?>\("),
    "blend_bwd2_kernel<256,false>": re.compile(r"splatco::blend_bwd2_kernel<256(, false)?>\("),
    "preprocess_bwd_kernel<false>": re.compile(r"splatco::preprocess_bwd_kernel(<false>)?\("),
}

_FUNC = re.compile(r"\s*Function : (\S+)")
_INSN = re.compile(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;?\s*(/\*.*\*/)?\s*$")


def tools_available() -> bool:
    return shutil.which("cuobjdump") is not None and shutil.which("c++filt") is not None


def nvcc_version(nvcc: str = "nvcc") -> str:
    """The `Cuda compilation tools, release ...` and `Build ...` lines of `nvcc --version`."""
    out = subprocess.run([nvcc, "--version"], capture_output=True, text=True, check=True).stdout
    return "\n".join(ln.strip() for ln in out.splitlines() if ln.startswith(("Cuda compilation tools", "Build ")))


def listings(path: str) -> dict:
    """{key: [instruction, ...]} of the KERNELS found in a cubin-carrying object or library."""
    sass = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    raw, cur = {}, None
    for ln in sass.splitlines():
        m = _FUNC.match(ln)
        if m:
            cur = raw.setdefault(m.group(1), [])
            continue
        m = _INSN.match(ln)
        if m and cur is not None:
            cur.append(m.group(1).rstrip(" ;"))
    names = list(raw)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.splitlines()
    out = {}
    for mangled, d in zip(names, dem):
        for key, pat in KERNELS.items():
            if pat.search(d):
                assert key not in out, f"two kernels match {key}"
                out[key] = raw[mangled]
    return out


def dump(lst: dict) -> str:
    return "".join(f"== {k}\n" + "".join(i + "\n" for i in v) for k, v in sorted(lst.items()))


def parse(text: str) -> dict:
    out, cur = {}, None
    for ln in text.splitlines():
        if ln.startswith("== "):
            cur = out.setdefault(ln[3:], [])
        elif cur is not None and ln:
            cur.append(ln)
    return out
