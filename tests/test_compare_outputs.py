"""tools/compare_outputs.py: the verdict per array and the exit status over two dump directories."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from compare_outputs import compare  # noqa: E402


def test_identical_arrays_are_bit_identical():
    a = np.array([1.0, -0.0, np.nan, np.inf])
    assert compare(a, a.copy()) == "bit-identical"


def test_signed_zero_is_equal_in_value_but_not_bit_identical():
    assert compare(np.array([1.0, -0.0]), np.array([1.0, 0.0])).startswith("equal in value")


def test_nan_payload_only_does_not_raise():
    a = np.array([np.nan, np.nan])
    b = np.frombuffer(np.array([0x7FF8000000000001, 0x7FF8000000000002], dtype=np.uint64).tobytes(), dtype=np.float64)
    assert compare(a, b).startswith("equal in value")


def test_matching_infinities_do_not_turn_the_difference_into_nan():
    res = compare(np.array([np.inf, 1.0]), np.array([np.inf, 1.0 + 2.0 ** -52]))
    assert res.startswith("max rel 2.2") and "nan" not in res


def test_mismatches_are_named():
    assert compare(np.array([np.inf]), np.array([-np.inf])).startswith("infinities differ")
    assert compare(np.array([np.nan, 1.0]), np.array([1.0, 1.0])).startswith("NaN in different places")
    assert compare(np.zeros(2), np.zeros(3)).startswith("shape")


@pytest.mark.parametrize("same", [True, False])
def test_exit_status_gates_bit_identity(tmp_path, same):
    a, b = tmp_path / "a", tmp_path / "b"
    a.mkdir(); b.mkdir()
    np.save(a / "qpos.npy", np.arange(4.0))
    np.save(b / "qpos.npy", np.arange(4.0) if same else np.arange(4.0) * (1 + 1e-15))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "compare_outputs.py"), str(a), str(b)], capture_output=True, text=True)
    assert r.returncode == (0 if same else 1), r.stdout
