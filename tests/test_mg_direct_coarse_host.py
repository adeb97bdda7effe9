"""Batch.set_coarse_solver and Batch.coarse_solve check the solver name and the vector's dtype before they call the
library."""
from types import SimpleNamespace

import numpy as np
import pytest

from fea_diffusion_b200.solver import Batch


def stand_in():
    """A batch whose library calls would fail: only validation may run."""
    return SimpleNamespace(COARSE_SOLVERS=Batch.COARSE_SOLVERS, ctx=None, h=None)


@pytest.mark.parametrize("name", ["", "CG", "Direct", "lu", "dense", None, 0, 1, b"cg"])
def test_solver_names_are_validated_before_the_library_call(name):
    with pytest.raises(ValueError):
        Batch.set_coarse_solver(stand_in(), name)


@pytest.mark.parametrize("r", [np.zeros(6, np.float32), np.zeros(6, np.int64), [0.0] * 6, np.zeros(6, np.complex128)])
def test_coarse_solve_takes_float64_only(r):
    with pytest.raises(TypeError):
        Batch.coarse_solve(stand_in(), r)


def test_the_names_are_those_of_the_header():
    assert Batch.COARSE_SOLVERS == {"cg": 0, "direct": 1}
