"""Device-memory I/O on the CPU: the tensor -> hb_setup_device argument mapping (shape, strides, dtype) and the rule
that numpy callers never import torch."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _mapped(Z, n):
    """The [n, d] matrix the library reads through hb_setup_device's (cell stride, PC stride) from Z's storage."""
    import torch
    from harmony_b200.harmony import tensor_abi_args
    code, cs, ps, d = tensor_abi_args(Z, n)
    return code, (cs, ps, d), torch.as_strided(Z, (n, d), (cs, ps), Z.storage_offset())


@pytest.mark.parametrize("dtype, code", [("float32", 0), ("float64", 1)])
def test_tensor_abi_args_layouts(dtype, code):
    import torch
    dt = getattr(torch, dtype)
    n, d = 37, 11
    base = torch.arange(n * d, dtype=dt).reshape(n, d)
    wide = torch.arange(n * 20, dtype=dt).reshape(n, 20)
    pcs_by_cells = base.T.contiguous()                            # [d, n]
    cases = {
        "contiguous [n, d]": (base, base, (d, 1, d)),
        "[d, n] tensor": (pcs_by_cells, base, (1, n, d)),
        "[d, n].T view": (pcs_by_cells.T, base, (1, n, d)),
        "column slice": (wide[:, 3:14], wide[:, 3:14], (20, 1, 11)),
    }
    for name, (Z, want, strides) in cases.items():
        c, st, got = _mapped(Z, n)
        assert c == code, name
        assert st == strides, name
        assert torch.equal(got, want), name


def test_tensor_abi_args_rejects():
    import torch
    from harmony_b200.harmony import tensor_abi_args
    with pytest.raises(TypeError, match="float32 or float64"):
        tensor_abi_args(torch.zeros(10, 4, dtype=torch.float16), 10)
    with pytest.raises(TypeError):
        tensor_abi_args(torch.zeros(10, 4, dtype=torch.int32), 10)
    with pytest.raises(ValueError, match="2-D"):
        tensor_abi_args(torch.zeros(10), 10)
    with pytest.raises(ValueError, match="2-D"):
        tensor_abi_args(torch.zeros(10, 4, 2), 10)
    with pytest.raises(ValueError, match="number of cells"):
        tensor_abi_args(torch.zeros(10, 4), 9)


def test_numpy_callers_do_not_import_torch():
    """prepare_inputs and harmony.setup with numpy input (the C library replaced by a recorder) leave torch unloaded."""
    code = r"""
import sys
import numpy as np
from harmony_b200 import prepare_inputs
from harmony_b200.harmony import harmony
Z = np.random.default_rng(0).standard_normal((300, 8))
a = prepare_inputs(Z, {"b": np.arange(300) % 3}, "b", nclust=5)
class Rec:
    def __init__(self): self.calls = []
    def __getattr__(self, name):
        return lambda *args: (self.calls.append(name), 0)[1]
g = object.__new__(harmony)
object.__setattr__(g, "_L", Rec())
object.__setattr__(g, "_h", None)
g.setup(a["Z"], a["phi_i"], a["sigma"], a["theta"], a["lambda_"], a["alpha"], a["max_iter_kmeans"],
        a["epsilon_kmeans"], a["epsilon_harmony"], a["K"], a["block_size"], a["B_vec"], a["batch_proportion_cutoff"])
assert "hb_setup" in g._L.calls and "hb_setup_device" not in g._L.calls, g._L.calls
print("torch" in sys.modules)
"""
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-s", "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip() == "False"
