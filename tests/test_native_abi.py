"""CPU-side checks of the C-ABI library: it loads, exports every symbol the header
declares, and its argument validation / layout helpers work without a GPU."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

from dmdqn_b200 import _native as N
from dmdqn_b200 import build as B

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


@pytest.fixture(scope="module")
def lib():
    B.build()
    return N.lib()


def test_every_declared_symbol_is_exported_and_bound(lib):
    header = open(os.path.join(ROOT, "include", "dmdqn_b200.h")).read()
    declared = set(re.findall(r"^(?:const char\*|int)\s+(dmdqn_\w+)\(", header, re.M))
    assert declared == set(N.SIGNATURES), declared ^ set(N.SIGNATURES)
    for name in declared:
        assert getattr(lib, name) is not None


def test_layout_and_workspace_helpers(lib):
    d = N.Dims(256, 256, 89, 96, 256, 4, 256, 30000)
    lay = N.Layout()
    N.check(lib.dmdqn_param_layout(C.byref(d), C.byref(lay)))
    assert (lay.w1, lay.b1, lay.w2, lay.b2, lay.w3, lay.b3) == (0, 96 * 256, 96 * 256 + 256, 96 * 256 + 256 + 65536,
                                                                  96 * 256 + 512 + 65536, 96 * 256 + 512 + 65536 + 1024)
    assert lay.stride % 32 == 0 and lay.stride >= lay.b3 + 4
    nbytes = C.c_size_t()
    N.check(lib.dmdqn_workspace_bytes(C.byref(d), C.byref(nbytes)))
    assert nbytes.value > 3 * 256 * 256 * 256 * 4


@pytest.mark.parametrize("field,value", [("hidden", 100), ("obs_stride", 90), ("n_actions", 5), ("n_nets", 3),
                                         ("batch", 0), ("capacity", 0)])
def test_bad_dims_are_rejected_with_a_message(lib, field, value):
    d = N.Dims(4, 4, 89, 96, 64, 4, 32, 100)
    setattr(d, field, value)
    assert lib.dmdqn_param_layout(C.byref(d), C.byref(N.Layout())) == N.ERR_ARG
    assert field.split("_")[0] in lib.dmdqn_last_error().decode()
    with pytest.raises(N.NativeError):
        N.check(N.ERR_ARG)


def test_no_cpu_fallback():
    """Without a CUDA device AgentGroup refuses to start.  A child process with every device hidden makes the check
    the same on a machine with a GPU."""
    code = ("from dmdqn_b200 import _native as N\nfrom dmdqn_b200.group import AgentGroup\n"
            "try:\n    AgentGroup(2, {'nn_layers': [64, 64]})\nexcept N.NativeError as exc:\n    print(exc)\n")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=600,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stderr[-500:]
    assert "no CPU fallback" in out.stdout, out.stdout
