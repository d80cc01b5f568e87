"""CPU-only checks of the drop-in boundary: the library builds, loads, exports every symbol the
headers declare, and its structs have the reference's LP64 layout (SURVEY.md section 8b)."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def libpath():
    from piplib_b200 import build
    return build.build()


def _declared_functions():
    names = set()
    for hdr in ("include/piplib/piplib.h", "include/piplib_b200.h"):
        text = open(os.path.join(ROOT, hdr)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        text = "\n".join(ln for ln in text.split("\n") if not ln.strip().startswith("#"))
        for m in re.finditer(r"\b((?:pip|sol)_[a-z0-9_]+)\s*\(", text):
            names.add(m.group(1))
    return sorted(names)


def test_exports_every_declared_symbol(libpath):
    lib = C.CDLL(libpath)
    names = _declared_functions()
    assert "pip_solve_dp" in names and "pip_solve_batch_dp" in names and len(names) >= 25
    assert "sol_quast_edit_dp" in names
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


# sizeof / offsetof of the six public structs on LP64 with the int64 Entier, derived from the
# reference's include/piplib/piplib.h:194-207 (PipMatrix), 218-222 (PipVector), 234-239 (PipNewparm),
# 249-252 (PipList), 265-272 (PipQuast), 283-327 (PipOptions)
LAYOUT = {
    "PipMatrix": (32, {"NbRows": 0, "NbColumns": 4, "p": 8, "p_Init": 16, "p_Init_size": 24}),
    "PipVector": (24, {"nb_elements": 0, "the_vector": 8, "the_deno": 16}),
    "PipNewparm": (32, {"rank": 0, "vector": 8, "deno": 16, "next": 24}),
    "PipList": (16, {"vector": 0, "next": 8}),
    "PipQuast": (48, {"newparm": 0, "list": 8, "condition": 16, "next_then": 24, "next_else": 32, "father": 40}),
    "PipOptions": (32, {"Nq": 0, "Verbose": 4, "Simplify": 8, "Deepest_cut": 12, "Maximize": 16,
                        "Urs_parms": 20, "Urs_unknowns": 24, "Compute_dual": 28}),
}


def _probe_layout(include_dir, tmp_path, tag, extra=()):
    """compile a probe against a header tree and return {struct: (size, {field: offset})}"""
    import json
    import subprocess
    src = ["#include <stdio.h>", "#include <stddef.h>", "#include <piplib/piplib64.h>", "int main(void){", 'printf("{");']
    first = True
    for name, (_, fields) in LAYOUT.items():
        src.append('printf("%s\\"%s\\": [%%zu, {", sizeof(%s));' % ("" if first else ", ", name, name))
        first = False
        for k, f in enumerate(fields):
            src.append('printf("%s\\"%s\\": %%zu", offsetof(%s, %s));' % ("" if k == 0 else ", ", f, name, f))
        src.append('printf("}]");')
    src += ['printf("}\\n");', "return 0;}"]
    c = tmp_path / ("probe_%s.c" % tag)
    c.write_text("\n".join(src))
    exe = tmp_path / ("probe_%s" % tag)
    subprocess.check_call(["gcc", "-w", "-I", include_dir, *extra, str(c), "-o", str(exe)])
    out = json.loads(subprocess.check_output([str(exe)]).decode())
    return {k: (v[0], v[1]) for k, v in out.items()}


def test_struct_layouts_match_reference(tmp_path):
    """all six structs: size and every field offset, our header against the values derived from the
    reference header"""
    ours = _probe_layout(os.path.join(ROOT, "include"), tmp_path, "ours")
    assert ours == {k: (v[0], v[1]) for k, v in LAYOUT.items()}
    from piplib_b200 import api
    assert C.sizeof(api.PipMatrix) == 32 and C.sizeof(api.PipOptions) == 32


def build_example(libpath, out_dir):
    """the reference's example program (tests/fixtures/example.c: test infrastructure, never product)
    compiled against include/ and linked with -lpiplib_dp"""
    import subprocess
    exe = os.path.join(str(out_dir), "example_dp")
    subprocess.check_call(["gcc", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "fixtures", "example.c"), "-o", exe,
                           "-L", os.path.dirname(libpath), "-lpiplib_dp", "-Wl,-rpath," + os.path.dirname(libpath)])
    return exe


def test_reference_example_compiles_against_our_headers(libpath, tmp_path):
    """the reference's only in-tree caller (example/example.c) builds against include/ and links with
    -lpiplib_dp"""
    assert os.path.exists(build_example(libpath, tmp_path))


def test_host_side_objects_without_gpu(libpath):
    """matrix / options allocation and the option defaults never touch the device."""
    from piplib_b200 import api
    L = api.lib()
    m = L.pip_matrix_alloc_dp(3, 4)
    assert m.contents.NbRows == 3 and m.contents.NbColumns == 4 and m.contents.p_Init_size == 12
    assert m.contents.p[2][3] == 0
    L.pip_matrix_free_dp(m)
    o = L.pip_options_init_dp()
    assert (o.contents.Nq, o.contents.Verbose, o.contents.Simplify, o.contents.Maximize) == (1, 0, 0, 0)
    L.pip_options_free_dp(o)
    assert b"sm_100a" in L.pip_b200_version()


def test_no_cpu_solver_in_product():
    """the product tree must not reference the oracle (parity claims depend on it)."""
    bad = []
    for dp, _, files in os.walk(os.path.join(ROOT, "piplib_b200")):
        for f in files:
            if f.endswith((".py", ".h", ".cpp", ".cu")):
                t = open(os.path.join(dp, f), errors="ignore").read()
                if re.search(r"oracle/|piporacle|pipref|libpipemu", t) and f != "pip_host.cpp":
                    bad.append(f)
    assert not bad, bad


def test_process_exits_after_the_host_pool_started(libpath):
    """the dense entry point starts the persistent host thread pool before it touches the device; a process
    that used it must still exit (a destroyed condition variable with parked workers blocks in glibc).
    Without a GPU the call itself fails loudly (-1): there is no CPU path."""
    import subprocess
    import sys
    code = ("import numpy as np\n"
            "from piplib_b200 import api\n"
            "dom = np.zeros((4, 3, 5), dtype=np.int64)\n"
            "try:\n    api.solve_dense(dom, None, -1)\nexcept RuntimeError as e:\n    print('refused:', e)\n"
            "print('bye')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "bye" in r.stdout
