"""B200: distance_transform_edt with SciPy's signature -- sampling, return_indices, in-place outputs -- through
vrg_edt_ft / vrg_edt_ft_device, against SciPy's fixtures, SciPy at run time, the CPU oracle and the default EDT."""
import os

import numpy as np
import pytest

from oracle.ft_oracle import distances_from_ft, ft_oracle

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "edt_ft")
FIXTURES = sorted(f[:-4] for f in os.listdir(GOLDEN) if f.endswith(".npz"))


def edt(*a, **k):
    from arterynetwork_b200.generateVesselVolume import distance_transform_edt
    return distance_transform_edt(*a, **k)


def blobs(shape, seed, keep=0.6):
    from scipy import ndimage as ndi  # only for smoothing the noise
    rng = np.random.default_rng(seed)
    b = ndi.gaussian_filter(rng.random(shape), 1.5)
    return (b > np.quantile(b, 1.0 - keep)).astype(np.uint8)


def expect(mask, sampling):
    ft = ft_oracle(mask, sampling)
    return distances_from_ft(ft, sampling), ft


@pytest.mark.parametrize("name", FIXTURES)
def test_fixture_bit_for_bit(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    for tag, s in (("unit", None), ("sampled", tuple(g["sampling"]))):
        dt, ft = edt(g["mask"], sampling=s, return_indices=True)
        assert ft.dtype == np.int32 and ft.shape == (3,) + g["mask"].shape and ft.flags.c_contiguous
        assert dt.dtype == np.float64 and dt.shape == g["mask"].shape
        assert np.array_equal(ft, g["ft_" + tag]), tag
        assert np.array_equal(dt, g["dt_" + tag]), tag


@pytest.mark.parametrize("sampling", [None, (0.1, 0.3, 0.7), (1.3, 0.5, 2.0), 0.7])
@pytest.mark.parametrize("shape", [(33, 40, 47), (16, 64, 96), (7, 9, 130)])
def test_random_blobs_equal_scipy(shape, sampling):
    ndi = pytest.importorskip("scipy.ndimage")
    for seed, keep in ((1, 0.6), (2, 0.93)):
        m = blobs(shape, seed, keep)
        dt, ft = edt(m, sampling=sampling, return_indices=True)
        rdt, rft = ndi.distance_transform_edt(m, sampling=sampling, return_indices=True)
        assert np.array_equal(ft, rft), (seed, keep)
        assert np.array_equal(dt, rdt), (seed, keep)


def test_c2_vessel_mask_anisotropic_equals_scipy():
    ndi = pytest.importorskip("scipy.ndimage")
    import torch
    import bench
    shape = (170, 512, 512)
    d_data, _ = bench.device_phantom(shape, 0, 0, shape[0], 0)
    vessel = (d_data > 0.5).to(torch.uint8)
    s = (0.8, 0.4, 0.4)
    dt, ft = edt(vessel, sampling=s, return_indices=True)
    rdt, rft = ndi.distance_transform_edt(vessel.cpu().numpy(), sampling=s, return_indices=True)
    assert np.array_equal(ft.cpu().numpy(), rft)
    assert np.array_equal(dt.cpu().numpy(), rdt)


@pytest.mark.parametrize("shape", [(1, 40, 50), (40, 1, 50), (40, 50, 1), (1, 1, 200), (1, 200, 1), (200, 1, 1)])
@pytest.mark.parametrize("sampling", [None, (1.3, 0.5, 0.7)])
def test_thin_volumes(shape, sampling):
    m = blobs(shape, 3, 0.8)
    if m.all():
        m.flat[0] = 0
    dt, ft = edt(m, sampling=sampling, return_indices=True)
    rdt, rft = expect(m, sampling)
    assert np.array_equal(ft, rft) and np.array_equal(dt, rdt)


def test_f_ordered_input_on_the_callers_axes():
    ndi = pytest.importorskip("scipy.ndimage")
    m = np.asfortranarray(blobs((20, 26, 31), 4, 0.85))
    s = (0.5, 1.3, 0.7)
    dt, ft = edt(m, sampling=s, return_indices=True)
    rdt, rft = ndi.distance_transform_edt(m, sampling=s, return_indices=True)
    assert dt.flags.c_contiguous and ft.flags.c_contiguous
    assert np.array_equal(ft, rft) and np.array_equal(dt, rdt)


def test_default_call_keeps_its_path_and_unit_distances_match_it():
    for m in (blobs((40, 48, 57), 5, 0.9), np.asfortranarray(blobs((30, 20, 50), 6, 0.7))):
        default = edt(m)
        dt = edt(m, return_indices=True)[0]
        assert np.array_equal(dt, default)
        assert np.array_equal(edt(m, sampling=1.0), default)
        # the default call still hands an F-ordered volume back as the transposed view of today's path
        assert default.flags.f_contiguous == (m.flags.f_contiguous and not m.flags.c_contiguous)


def test_return_distances_false_and_in_place_numpy():
    m = blobs((24, 30, 35), 7, 0.8)
    s = (0.3, 0.7, 1.1)
    rdt, rft = expect(m, s)
    ft = edt(m, sampling=s, return_distances=False, return_indices=True)
    assert isinstance(ft, np.ndarray) and np.array_equal(ft, rft)
    dist = np.full(m.shape, -1.0)
    ind = np.zeros((3,) + m.shape, np.int32)
    assert edt(m, sampling=s, return_indices=True, distances=dist, indices=ind) is None
    assert np.array_equal(dist, rdt) and np.array_equal(ind, rft)
    ind_f = np.asfortranarray(np.zeros((3,) + m.shape, np.int32))  # not C order: filled through a copy
    out = edt(m, sampling=s, return_indices=True, indices=ind_f)
    assert np.array_equal(out, rdt) and np.array_equal(ind_f, rft)
    dist2 = np.zeros(m.shape)
    ft2 = edt(m, sampling=s, return_indices=True, distances=dist2)
    assert np.array_equal(dist2, rdt) and np.array_equal(ft2, rft)


def test_cuda_tensors_in_place_and_side_stream():
    import torch
    m = blobs((30, 44, 53), 8, 0.85)
    s = (0.8, 0.4, 0.4)
    rdt, rft = expect(m, s)
    t = torch.from_numpy(m).cuda()
    dt, ft = edt(t, sampling=s, return_indices=True)
    assert dt.is_cuda and ft.is_cuda and ft.dtype == torch.int32 and ft.shape == (3,) + m.shape
    assert np.array_equal(dt.cpu().numpy(), rdt) and np.array_equal(ft.cpu().numpy(), rft)
    ft_only = edt(t, sampling=s, return_distances=False, return_indices=True)
    assert np.array_equal(ft_only.cpu().numpy(), rft)
    dist = torch.full(m.shape, -1.0, dtype=torch.float64, device="cuda")
    ind = torch.zeros((3,) + m.shape, dtype=torch.int32, device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())  # the outputs were filled on the default stream
    with torch.cuda.stream(side):
        tb = (t != 0)  # a bool input
        assert edt(tb, sampling=s, return_indices=True, distances=dist, indices=ind) is None
        got_d, got_i = dist.cpu().numpy(), ind.cpu().numpy()
    assert np.array_equal(got_d, rdt) and np.array_equal(got_i, rft)
    ind_t = torch.zeros((m.shape[2], m.shape[1], m.shape[0], 3), dtype=torch.int32, device="cuda").permute(3, 2, 1, 0)
    d_only = edt(t.permute(2, 1, 0).contiguous().permute(2, 1, 0), sampling=s, return_indices=True, indices=ind_t)
    assert np.array_equal(d_only.cpu().numpy(), rdt) and np.array_equal(ind_t.cpu().numpy(), rft)


def test_errors():
    import torch
    with pytest.raises(ValueError, match="no zero voxel"):
        edt(np.ones((4, 5, 6), np.uint8), return_indices=True)
    with pytest.raises(ValueError, match="no zero voxel"):
        edt(torch.ones((4, 5, 6), dtype=torch.uint8, device="cuda"), sampling=2.0)
    with pytest.raises(ValueError, match="3-D"):
        edt(torch.zeros((4, 5), dtype=torch.uint8, device="cuda"), return_indices=True)
    t = torch.zeros((4, 5, 6), dtype=torch.uint8, device="cuda")
    with pytest.raises(RuntimeError, match="indices array must be int32"):
        edt(t, return_indices=True, indices=torch.zeros((3, 4, 5, 6), dtype=torch.int64, device="cuda"))
    with pytest.raises(RuntimeError, match="distances array has wrong shape"):
        edt(t, distances=torch.zeros((4, 5, 7), dtype=torch.float64, device="cuda"))
    with pytest.raises(RuntimeError, match="at least one"):
        edt(t, return_distances=False)
