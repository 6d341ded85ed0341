#!/usr/bin/env python
"""A/B builds of the CUDA library: tools/build_variant.py <tag> [nvcc flags ...] -> build/variants/libidocp_b200_<tag>.so
(the flags are appended to __graft_entry__.NVCC_FLAGS; select the library with IDOCP_B200_LIBRARY=<path> python bench.py ...)."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as g  # noqa: E402


def main():
    tag, flags = sys.argv[1], sys.argv[2:]
    out_dir = os.path.join(ROOT, "build", "variants")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, "libidocp_b200_%s.so" % tag)
    cmd = [os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")] + g.NVCC_FLAGS + flags + ["-o", out, os.path.join(g.CSRC, "capi.cu")]
    res = subprocess.run(cmd, cwd=g.CSRC, capture_output=True, text=True)
    with open(out[:-3] + ".ptxas.log", "w") as f:
        f.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
    if res.returncode != 0:
        print(res.stdout + res.stderr)
        raise SystemExit("nvcc failed")
    print(out)


if __name__ == "__main__":
    main()
