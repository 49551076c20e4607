"""CPU: the feature-transform oracle (oracle/ft_oracle.c) equals SciPy's distance_transform_edt(..., return_indices=True)
bit for bit, and distance_transform_edt's argument handling raises SciPy's errors before it touches the GPU."""
import itertools
import os

import numpy as np
import pytest

from oracle.ft_oracle import distances_from_ft, ft_oracle

ndi = pytest.importorskip("scipy.ndimage")

SAMPLINGS = [None, (0.1, 0.3, 0.7), (1.3, 0.5, 2.0), 0.7, (0.5, 2.0, 1.3)]
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "edt_ft")


def assert_scipy(mask, sampling):
    dt, ft = ndi.distance_transform_edt(mask, sampling=sampling, return_indices=True)
    mine = ft_oracle(mask, sampling)
    assert np.array_equal(mine, ft), (mask.shape, sampling)
    assert np.array_equal(distances_from_ft(mine, sampling), dt), (mask.shape, sampling)


@pytest.mark.parametrize("sampling", SAMPLINGS)
def test_every_2x2x2_mask(sampling):
    for bits in itertools.product((0, 1), repeat=8):
        if all(bits):
            continue  # no zero voxel: the transform is undefined
        assert_scipy(np.array(bits, np.uint8).reshape(2, 2, 2), sampling)


@pytest.mark.parametrize("sampling", SAMPLINGS)
def test_random_and_lattice_masks(sampling):
    rng = np.random.default_rng(7)
    for it in range(60):
        shape = tuple(int(v) for v in rng.integers(1, 11, size=3))
        if it % 2:
            m = rng.random(shape) < rng.uniform(0.3, 0.97)
        else:  # zeros on a lattice: ties everywhere
            m = np.ones(shape, bool)
            step = rng.integers(1, 5, size=3)
            off = [int(rng.integers(0, s)) for s in step]
            m[off[0]::step[0], off[1]::step[1], off[2]::step[2]] = False
        if m.all():
            m.flat[int(rng.integers(m.size))] = False
        assert_scipy(m, sampling)


@pytest.mark.parametrize("name", sorted(f[:-4] for f in os.listdir(GOLDEN) if f.endswith(".npz")))
def test_oracle_reproduces_fixture(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    for tag, s in (("unit", None), ("sampled", tuple(g["sampling"]))):
        ft = ft_oracle(g["mask"], s)
        assert np.array_equal(ft, g["ft_" + tag])
        assert np.array_equal(distances_from_ft(ft, s), g["dt_" + tag])


@pytest.fixture
def no_gpu(monkeypatch):
    """Any attempt to reach the library fails the test: the errors below must come from the host-side checks."""
    from arterynetwork_b200 import _native

    def refuse(*a, **k):
        raise AssertionError("the library was called")
    monkeypatch.setattr(_native, "load", refuse)


M = np.ones((3, 4, 5), np.uint8)
M[1, 2, 3] = 0


@pytest.mark.parametrize("kwargs, exc, text", [
    (dict(return_distances=False), RuntimeError, "at least one of return_distances/return_indices"),
    (dict(return_distances=False, distances=np.empty((3, 4, 5))), RuntimeError, "return_distances must be True"),
    (dict(indices=np.empty((3, 3, 4, 5), np.int32)), RuntimeError, "return_indices must be True"),
    (dict(return_indices=True, indices=np.empty((3, 4, 5), np.int32)), RuntimeError, "indices array has wrong shape"),
    (dict(return_indices=True, indices=np.empty((3, 3, 4, 5), np.int64)), RuntimeError, "indices array must be int32"),
    (dict(distances=np.empty((3, 4, 6))), RuntimeError, "distances array has wrong shape"),
    (dict(distances=np.empty((3, 4, 5), np.float32)), RuntimeError, "distances array must be float64"),
    (dict(sampling=(1.0, 2.0)), RuntimeError, "sequence argument must have length equal to input rank"),
    (dict(sampling=0.0), ValueError, "positive and finite"),
    (dict(sampling=(1.0, -1.0, 1.0)), ValueError, "positive and finite"),
    (dict(sampling=(1.0, 1.0, np.nan)), ValueError, "positive and finite"),
    (dict(sampling=np.inf), ValueError, "positive and finite"),
])
def test_argument_errors_before_the_gpu(no_gpu, kwargs, exc, text):
    from arterynetwork_b200.generateVesselVolume import distance_transform_edt
    with pytest.raises(exc, match=text):
        distance_transform_edt(M, **kwargs)
    if exc is RuntimeError and "sampling" not in kwargs:  # the same call is an error for SciPy too, of the same type
        with pytest.raises(exc):
            ndi.distance_transform_edt(M, **kwargs)


def test_two_dimensional_input_refused_before_the_gpu(no_gpu):
    from arterynetwork_b200.generateVesselVolume import distance_transform_edt
    with pytest.raises(ValueError, match="3-D"):
        distance_transform_edt(np.ones((4, 5)), return_indices=True)
