"""Batch.solve_load_cases checks the shape and dtype of the loads before it calls the library."""
from types import SimpleNamespace

import numpy as np
import pytest

from fea_diffusion_b200.solver import Batch


def stand_in(n_vertices):
    """A batch whose library calls would fail: only validation may run."""
    return SimpleNamespace(packed=SimpleNamespace(n_vertices=n_vertices), ctx=None, h=None)


@pytest.mark.parametrize("loads, error", [
    (np.zeros((2, 5, 2), np.float32), TypeError),
    (np.zeros((2, 5, 2), np.int64), TypeError),
    ([[[0.0, 0.0]] * 5], TypeError),
    (np.zeros((5, 2)), ValueError),
    (np.zeros((2, 4, 2)), ValueError),
    (np.zeros((2, 5, 3)), ValueError),
    (np.zeros((2, 5, 2, 1)), ValueError),
])
def test_loads_are_validated_before_the_library_call(loads, error):
    with pytest.raises(error):
        Batch.solve_load_cases(stand_in(5), loads)
