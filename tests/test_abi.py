"""CPU-side checks of the boundary: the C-ABI library loads, exports every symbol the header
declares, and the product path fails loudly without a GPU (no CPU fallback)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "easyhybrid_cuda.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(eh_[a-z_0-9]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(eh):
    from easyhybrid_b200 import _abi, _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = _header_symbols()
    assert len(names) >= 24
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/easyhybrid_cuda.h but not exported"
    # and the ctypes mirror declares a signature for each of them
    assert sorted(_abi.SIGNATURES) == names


def test_struct_layout_matches_header(eh):
    """sizeof(eh_model_desc) as seen by a C compiler == the ctypes mirror"""
    import subprocess
    import tempfile
    from easyhybrid_b200 import _abi
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write('#include <stdio.h>\n#include "easyhybrid_cuda.h"\nint main(){printf("%zu %zu %zu %zu",'
                           'sizeof(eh_model_desc),sizeof(eh_chain_desc),sizeof(eh_pm_instr),sizeof(eh_pm_arg));return 0;}')
        exe = os.path.join(d, "s")
        subprocess.check_call(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        sizes = [int(x) for x in subprocess.check_output([exe]).split()]
    assert sizes == [ctypes.sizeof(_abi.eh_model_desc), ctypes.sizeof(_abi.eh_chain_desc),
                     ctypes.sizeof(_abi.eh_pm_instr), ctypes.sizeof(_abi.eh_pm_arg)]


def test_no_cpu_fallback(eh):
    """without a CUDA device eh_create must fail with EH_ECUDA (and say so).  The session is created in a child process
    that sees no device (CUDA_VISIBLE_DEVICES empty), so the check also runs on a machine that has a GPU."""
    import subprocess
    import sys
    from easyhybrid_b200 import _abi
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "import easyhybrid_b200 as eh\n"
            "from conftest import rbq10_model\n"
            "try:\n"
            "    eh.FusedSession(rbq10_model(eh)).close()\n"
            "except eh.EasyHybridCudaError as e:\n"
            "    print(e.status)\n"
            "    print(e)\n") % (ROOT, os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr[-4000:]
    out = r.stdout.split("\n", 1)
    assert len(out) == 2, "eh_create succeeded without a visible CUDA device"
    assert int(out[0]) == _abi.EH_ECUDA
    assert "no CPU fallback" in out[1] or "sm_100a" in out[1]


def test_product_does_not_import_oracle():
    """the oracle is test infrastructure: nothing under the package may reference it"""
    pkg = os.path.join(ROOT, "easyhybrid.jl_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dp, f), errors="ignore").read()
                assert "oracle" not in txt.lower().replace("test infrastructure", ""), os.path.join(dp, f)
