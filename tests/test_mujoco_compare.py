"""tools/compare_with_mujoco.py: the direct oracle-vs-MuJoCo check.  The real comparison needs the `mujoco` package and robosuite's
mesh files and skips itself where they are absent; the script's seeded state, torque script and MJCF rewrite are checked without them."""
import importlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _tool():
    from tools import compare_with_mujoco

    return compare_with_mujoco


def test_helpers_are_deterministic_and_shaped():
    from tests.util import load

    t = _tool()
    m = load("Lift_Panda")
    q1, q2 = t.seeded_state(m, 3), t.seeded_state(m, 3)
    assert np.array_equal(q1, q2) and q1.shape == (m.nq,)
    assert not np.array_equal(q1, np.asarray(m.qpos0))
    assert np.array_equal(q1[9:], np.asarray(m.qpos0)[9:])  # only the robot joints are perturbed
    s = t.torque_script(m.nu, 7, 400, 0)
    assert s.shape == (400, m.nu) and np.abs(s[:, :7]).max() <= 4.0
    assert set(np.unique(s[:, 7:])) == {-1.0, 1.0}
    xml = t.load_mjcf("Lift_Panda", "/somewhere/assets")
    assert "/root/reference" not in xml and "<texture" not in xml and "/somewhere/assets/robots/panda/meshes/link0.stl" in xml


def _real_mujoco():
    """the real package, not oracle/mujoco_shim (which other tests put on sys.path)"""
    saved = sys.modules.pop("mujoco", None)
    path = [p for p in sys.path if "mujoco_shim" not in p]
    old, sys.path = sys.path, path
    try:
        mod = importlib.import_module("mujoco")
        return None if "b2s" in getattr(mod, "__version__", "") else mod
    except ImportError:
        return None
    finally:
        sys.path = old
        if saved is not None:
            sys.modules["mujoco"] = saved
        else:
            sys.modules.pop("mujoco", None)


def test_against_real_mujoco(capsys):
    if _real_mujoco() is None:
        pytest.skip("mujoco is not installed here (no network in the build container / on the GPU box)")
    assets = os.environ.get("B2S_ROBOSUITE_ASSETS")
    if assets is None:
        try:
            import robosuite

            assets = os.path.join(os.path.dirname(robosuite.__file__), "models", "assets")
        except ImportError:
            pytest.skip("set B2S_ROBOSUITE_ASSETS to robosuite/models/assets")
    sys.modules.pop("mujoco", None)
    rc = _tool().main(["--assets", assets, "--steps", "250"])
    assert rc == 0, capsys.readouterr().out
