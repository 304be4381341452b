"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol include/rlppo.h
declares, refuses to compute without a B200, and its host-side permutation is NumPy's, bit for bit."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "rlppo.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rlppo_[a-z0-9_]+)\s*\(", src)))


def _exported(path):
    """The rlppo_* functions the shared library defines (its dynamic symbol table)."""
    out = subprocess.run(["nm", "-D", "--defined-only", path], check=True, capture_output=True, text=True).stdout
    return sorted({f[2] for f in (line.split() for line in out.splitlines()) if len(f) == 3 and f[2].startswith("rlppo_")})


def test_header_symbols_exported_and_bound():
    from rlgym_ppo_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/rlppo.h but not exported"
        assert n in _lib.EXPORTED, f"{n} not bound in rlgym_ppo_b200/_lib.py"
    assert sorted(_lib.EXPORTED) == names
    # and nothing beyond the header: an entry point whose declaration is gone must not linger in a .cu file
    undeclared = sorted(set(_exported(_lib.LIB_PATH)) - set(names))
    assert not undeclared, f"exported by the library but not declared in include/rlppo.h: {undeclared}"
    assert _lib.version() >= 100


def test_no_cpu_fallback():
    import torch
    from rlgym_ppo_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_lib.RlppoError):
        _lib.require_device()
    # a compute entry point called without a device must fail, not compute on the host
    x = np.zeros(8, np.float32)
    rc = _lib._lib.rlppo_rows_to_bf16(x.ctypes.data, 8, 1, 8, None, None, 5.0, x.ctypes.data, 8, None, 0, None)
    assert rc == -3 and "no CPU fallback" in _lib.last_error()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "rlgym_ppo_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.replace("no oracle", ""), f"{f} references the oracle"


@pytest.mark.parametrize("seed,n", [(7, 1000), (123, 150000), (0, 1), (5, 2), (9, 65537)])
def test_host_permutation_is_numpy_legacy(seed, n):
    from rlgym_ppo_b200 import _lib
    a, b = np.random.RandomState(seed), np.random.RandomState(seed)
    for _ in range(3):
        assert np.array_equal(_lib.host_permutation(a, n), b.permutation(n))
    assert np.array_equal(a.permutation(17), b.permutation(17))  # generator state handed back intact


def test_host_permutation_golden(golden):
    from rlgym_ppo_b200 import _lib
    g = golden("buffer")
    r = np.random.RandomState(123)
    assert np.array_equal(_lib.host_permutation(r, 150000)[:64], g["perm150000.head"])
    assert np.array_equal(_lib.host_permutation(r, 150000)[:64], g["perm150000.second_head"])
