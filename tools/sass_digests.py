"""Fingerprints of the solver kernels' machine code: sha256 of the SASS of every solve-kernel instantiation, the team
kernel and the whole-grid kernel in a built library, instruction text only (addresses and encodings stripped), with
the nvcc release that compiled them.  tests/test_problem_info.py compares the in-tree build with
tests/golden/sass_solver_kernels.json: a change that should leave those kernels alone leaves them alone.

    python tools/sass_digests.py [LIB] [--write]      # LIB defaults to piplib_b200/lib/libpiplib_dp.so

--write stores the fingerprints as the golden file; do that only for a change that is meant to alter the solver
kernels, or when the project moves to another nvcc release.
"""
import hashlib
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "sass_solver_kernels.json")
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")


def tool(name):
    return os.path.join(CUDA, "bin", name)


def nvcc_release():
    """e.g. "12.9, V12.9.86" """
    out = subprocess.run([tool("nvcc"), "--version"], capture_output=True, text=True, check=True).stdout
    return re.search(r"release (.*)", out).group(1).strip()


def digests(lib):
    text = subprocess.run([tool("cuobjdump"), "-sass", lib], capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for line in text.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1) if re.match(r"_Z\d+pip_(solve|team|large)_kernel", m.group(1)) else None
            if cur:
                out[cur] = hashlib.sha256()
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;", line)
        if cur and m:
            out[cur].update((m.group(1) + "\n").encode())
    return {k: h.hexdigest() for k, h in sorted(out.items())}


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    lib = args[0] if args else os.path.join(ROOT, "piplib_b200", "lib", "libpiplib_dp.so")
    res = dict(nvcc=nvcc_release(), kernels=digests(lib))
    if "--write" in sys.argv:
        with open(GOLDEN, "w") as f:
            json.dump(res, f, indent=1)
            f.write("\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
