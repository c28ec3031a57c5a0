"""TEST INFRASTRUCTURE ONLY.  Stored values that pin the CPU tests which compare the oracle and the product's host logic with
the original project's own classes (tests/test_host_logic_cpu.py, test_oracle_cpu.py, test_oracle_flow_cpu.py), so that
those tests check something on every machine, not only where the original source tree is present.

Each such test module has a dict PINS: group -> function returning [(key, tensor, tol)], the oracle / product values of
seeded CPU inputs.  The test compares them with tests/golden/pins_<module>.npz: bit for bit when tol == 0 (where the
live comparison with the original is bit for bit), else max|a-b| / max|b| < tol.  Where the original tree is present
(oracle/ref_shim.py) the tests still run their live comparison with it as well.

    python -m oracle.golden_pins        # rewrite tests/golden/pins_*.npz from the tests' PINS functions
"""
from __future__ import annotations

import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
MODULES = ("test_host_logic_cpu", "test_oracle_cpu", "test_oracle_flow_cpu")
_cache = {}


def _path(module):
    return os.path.join(GOLD, f"pins_{module.replace('test_', '', 1)}.npz")


def check(module, group, pairs):
    """Compare [(key, tensor, tol)] with the stored values of `module` / `group`."""
    if module not in _cache:
        _cache[module] = dict(np.load(_path(module)))
    stored = _cache[module]
    for key, t, tol in pairs:
        want = torch.from_numpy(stored[f"{group}/{key}"])
        got = t.detach().cpu()
        assert got.shape == want.shape and got.dtype == want.dtype, (group, key, got.shape, want.shape, got.dtype, want.dtype)
        if tol == 0:
            assert torch.equal(got, want), f"{group}/{key} differs from the stored value"
        else:
            err = float((got.double() - want.double()).abs().max() / want.double().abs().max().clamp_min(1e-30))
            assert err < tol, (f"{group}/{key}", err, tol)


def main():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    sys.path.insert(0, ROOT)
    for module in MODULES:
        mod = importlib.import_module(module)
        data = {}
        for group, fn in mod.PINS.items():
            for key, t, _ in fn():
                name, a = f"{group}/{key}", t.detach().cpu().numpy()
                if name in data:           # several implementations checked against one value: they must agree
                    assert np.array_equal(data[name], a), name
                data[name] = a
        np.savez_compressed(_path(module), **data)
        print(_path(module), f"{os.path.getsize(_path(module)) / 1e6:.2f} MB", len(data), "arrays")


if __name__ == "__main__":
    main()
