"""The drop-in boundary (SURVEY.md 8(b)): every public method of the reference's hot-path classes exists here with the same
parameter names, order and defaults (extra trailing optional parameters are allowed: device=, process_group=, ...).
The fixture was recorded from the unmodified reference (tests/golden/make_api_surface.py).  CPU only: nothing is launched."""
import importlib
import inspect
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SURFACE = json.load(open(os.path.join(ROOT, "tests", "golden", "api_surface.json")))


def _resolve(path):
    parts = path.split(".")
    for cut in range(len(parts) - 1, 0, -1):
        try:
            obj = importlib.import_module("rlgym_ppo_b200." + ".".join(parts[:cut]))
        except ImportError:
            continue
        for name in parts[cut:]:
            obj = getattr(obj, name)
        return obj
    raise ImportError(path)


@pytest.mark.parametrize("path", sorted(SURFACE))
def test_surface_matches_reference(path):
    ours = _resolve(path)
    for name, want in SURFACE[path].items():
        member = ours if name == "__call__" else inspect.getattr_static(ours, name, None)
        assert member is not None, f"{path}.{name} is missing"
        if want == "property":
            assert isinstance(member, property), f"{path}.{name} must be a property"
            continue
        fn = member.__func__ if isinstance(member, (staticmethod, classmethod)) else member
        got = [[p.name, None if p.default is inspect.Parameter.empty else repr(p.default)]
               for p in inspect.signature(fn).parameters.values()]
        assert got[:len(want)] == want, f"{path}.{name}: {got[:len(want)]} != {want}"
        for extra in got[len(want):]:
            assert extra[1] is not None, f"{path}.{name}: extra parameter {extra[0]} must be optional"


@pytest.mark.parametrize("output_shape", [0, 66, 128])
def test_continuous_policy_rejects_unsupported_widths(output_shape):
    """ContinuousPolicy serves 1 to 32 actions (2 to 64 outputs): anything else is refused at construction, before any
    device work, rather than by the kernel at the first call."""
    from rlgym_ppo_b200.ppo import ContinuousPolicy
    with pytest.raises(ValueError, match="1 to 32 actions"):
        ContinuousPolicy(8, output_shape, (64,), "cuda:0")
