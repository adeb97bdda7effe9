"""The load-case output methods of Batch check their arguments before they call the library."""
from types import SimpleNamespace

import numpy as np
import pytest

from fea_diffusion_b200.solver import Batch


def stand_in():
    """A batch whose library calls would fail: only validation may run."""
    b = Batch.__new__(Batch)
    b.packed, b.ctx, b.h = SimpleNamespace(n_vertices=5, n_cells=3), None, None
    return b


@pytest.mark.parametrize("size", [0, -1, 8193, 2.5, "64", True, None])
def test_image_size_is_validated(size):
    with pytest.raises(ValueError):
        stand_in().load_case_images(size, np.zeros(4))


@pytest.mark.parametrize("affine", [np.zeros(3), np.zeros((2, 4)), []])
def test_the_camera_has_four_values(affine):
    with pytest.raises(ValueError):
        stand_in().load_case_images(64, affine)


@pytest.mark.parametrize("names", [[], ["stress_x"] * 5, ["stress_z"], "stress_x", ["stress_x", "Stress_y"]])
def test_component_names_are_validated(names):
    with pytest.raises(ValueError):
        stand_in().load_case_cell_components(0, names)
