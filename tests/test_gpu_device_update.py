"""``update()`` (VRG:124-261) on CUDA tensors (B200 only): state, flips, band rows and Parzen sums on the device.

The bar is the host ``update()`` on the same inputs, bit for bit -- labels, segmentedMap, the three row lists and both sum
volumes -- and the recordings of the unmodified reference function in tests/golden/update."""
import glob
import os

import numpy as np
import pytest

from golden_util import load_golden

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

UPDATE_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "update")
NAMES = sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(UPDATE_DIR, "*.npz")))
DTYPES = ["uint8", "int8", "int16", "int32", "int64", "float32", "float64"]
RTOL = 1e-12


def mod():
    from arterynetwork_b200 import variationalRegionGrowing as m
    return m


def cuda(a, dtype=None):
    t = torch.from_numpy(np.asarray(a)).cuda()  # keeps the array's strides (an F-ordered array stays F-ordered)
    return t if dtype is None else t.to(dtype)


def host(t):
    return t.cpu().numpy()


def rows_sorted(a):
    a = np.asarray(a, dtype=np.int64).reshape(-1, 3)
    return a[np.lexsort(a.T[::-1])]


def bits(a):
    """The bytes of an array, dtype and shape included: equal bits, not just equal values (-0.0 != 0.0, NaN == NaN)."""
    a = np.ascontiguousarray(a)
    return a.dtype.str, a.shape, a.tobytes()


def assert_same_as_host(tout, hout, init_branch=False):
    """The 7-tuple of the tensor call against the host call's, bit for bit."""
    for i, (t, h) in enumerate(zip(tout, hout)):
        if i == 0 and init_branch:
            assert t is h  # the caller's object on the init branch
            continue
        assert isinstance(t, torch.Tensor) and t.is_cuda, i
        if i in (0, 3, 4):
            assert t.dtype == torch.int64 and t.is_contiguous(), i
        if i in (5, 6):
            assert t.dtype == torch.float64, i
        assert bits(host(t)) == bits(h), i


def first_flips(out):
    """The flips of the reference driver's next decision (VRG:79-88) from an update() result, on host arrays."""
    _, seg_map, vm, ib, ob, ip, op = out
    allb = np.concatenate((ib, ob))
    n_in = np.count_nonzero(vm <= 1)
    n_out = np.count_nonzero((vm == 2) | (vm == 3))
    mask = np.logical_xor(seg_map[tuple(allb.T)], ip[tuple(allb.T)] / n_in >= op[tuple(allb.T)] / n_out)
    return allb[mask]


def state_after_init(data, vm0, H):
    """(segmented, segmentedMap, valueMap, innerBnd, outerBnd, innerProb, outerProb) of the host init branch."""
    vm = np.array(vm0, dtype=np.int64)
    segmented = np.argwhere(vm == 0)
    seg_map = np.zeros(vm.shape, dtype=np.int64)
    seg_map[tuple(segmented.T)] = 1
    return mod().update(data, segmented, seg_map, vm, H)


def init_and_flips(data, vm0, H):
    """One init call and one flips call (the first decision's flips) through tensors and through host arrays; returns both
    flips calls' results after checking the init calls'.  The tensors keep the arrays' dtypes and layouts."""
    m = mod()
    vm_h = np.array(vm0)
    segmented = np.argwhere(vm_h == 0)
    seg_h = np.zeros_like(vm_h)
    seg_h[tuple(segmented.T)] = 1
    seg_t, vm_t = cuda(seg_h), cuda(vm_h)
    d_t = cuda(data)
    h0 = m.update(data, segmented, seg_h, vm_h, H)
    t0 = m.update(d_t, segmented, seg_t, vm_t, H)
    assert_same_as_host(t0, h0, init_branch=True)
    flips = first_flips(h0)
    assert len(flips)
    h1 = m.update(data, h0[0], seg_h, vm_h, H, flips, h0[3], h0[4], h0[5], h0[6])
    t1 = m.update(d_t, t0[0], seg_t, vm_t, H, cuda(flips), t0[3], t0[4], t0[5], t0[6])
    assert t1[1] is seg_t and t1[2] is vm_t and t1[5] is t0[5] and t1[6] is t0[6]
    return t1, h1


# ---- 1. the recordings, call by call -----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", NAMES)
def test_update_recordings_through_tensors(name):
    m = mod()
    f = np.load(os.path.join(UPDATE_DIR, name + ".npz"))
    k = f["k"].astype(np.int64)
    data = k if bool(f["data_is_int"]) else k.astype(np.float64) / int(f["quantum"])
    H = float(f["H"])
    shape = k.shape
    d_t = cuda(data)
    for c in range(int(f["n_calls"])):
        seg_in = np.unpackbits(f["c%d_seg_in" % c])[: k.size].reshape(shape).astype(np.int64)
        vm_in = f["c%d_vm_in" % c].astype(np.int64)
        segmented_in = np.argwhere(seg_in == 1)
        flips = f["c%d_flips" % c]
        seg_t, vm_t = cuda(seg_in), cuda(vm_in)
        if c == 0:
            hout = m.update(data, segmented_in, seg_in.copy(), vm_in.copy(), H)
            tout = m.update(d_t, segmented_in, seg_t, vm_t, H)
        else:
            prev_in, prev_out = f["c%d_inner" % (c - 1)], f["c%d_outer" % (c - 1)]
            ip, op = (torch.full(shape, -3.5, dtype=torch.float64, device="cuda") for _ in range(2))  # overwritten everywhere
            hout = m.update(data, segmented_in, seg_in.copy(), vm_in.copy(), H, flips, prev_in, prev_out,
                            np.zeros(shape), np.zeros(shape))
            tout = m.update(d_t, segmented_in, seg_t, vm_t, H, cuda(flips), prev_in, prev_out, ip, op)
            assert tout[5] is ip and tout[6] is op  # the caller's tensors, as in the reference
        assert tout[1] is seg_t and tout[2] is vm_t  # updated in place, same objects
        assert_same_as_host(tout, hout, init_branch=c == 0)
        # the assertions of the host test against the recording
        segmented, seg_map, vm, inner, outer, iprob, oprob = (host(x) if isinstance(x, torch.Tensor) else x for x in tout)
        assert np.array_equal(vm, f["c%d_vm_out" % c])
        assert np.array_equal(seg_map == 1, np.unpackbits(f["c%d_seg_out" % c])[: k.size].reshape(shape).astype(bool))
        assert np.array_equal(rows_sorted(segmented), f["c%d_segmented" % c])
        assert np.array_equal(rows_sorted(inner), f["c%d_inner" % c]) and np.array_equal(rows_sorted(outer), f["c%d_outer" % c])
        band = np.concatenate([f["c%d_inner" % c], f["c%d_outer" % c]])
        np.testing.assert_allclose(iprob[tuple(band.T)], f["c%d_pin" % c], rtol=RTOL, atol=0)
        np.testing.assert_allclose(oprob[tuple(band.T)], f["c%d_pout" % c], rtol=RTOL, atol=0)
        assert [np.count_nonzero(iprob), np.count_nonzero(oprob)] == f["c%d_prob_nonzero" % c].tolist()


# ---- 2. map dtypes -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["valueMap", "segmentedMap"])
@pytest.mark.parametrize("dtype", DTYPES)
def test_map_dtypes(dtype, which):
    m = mod()
    f = np.load(os.path.join(UPDATE_DIR, "excl32.npz"))  # labels 0, 3 and 4
    k = f["k"].astype(np.int64)
    data = k if bool(f["data_is_int"]) else k.astype(np.float64) / int(f["quantum"])
    H, shape, c = float(f["H"]), k.shape, 1
    seg_in = np.unpackbits(f["c%d_seg_in" % c])[: k.size].reshape(shape).astype(np.int64)
    vm_in = f["c%d_vm_in" % c].astype(np.int64)
    if which == "valueMap":
        vm_in = vm_in.astype(getattr(np, dtype))
    else:
        seg_in = seg_in.astype(getattr(np, dtype))
    segmented_in = np.argwhere(seg_in == 1)
    args = (f["c%d_flips" % c], f["c%d_inner" % (c - 1)], f["c%d_outer" % (c - 1)])
    hout = m.update(data, segmented_in, seg_in.copy(), vm_in.copy(), H, *args, np.zeros(shape), np.zeros(shape))
    seg_t, vm_t = cuda(seg_in), cuda(vm_in)
    tout = m.update(cuda(data), segmented_in, seg_t, vm_t, H, cuda(args[0]), args[1], args[2],
                    torch.zeros(shape, dtype=torch.float64, device="cuda"), torch.zeros(shape, dtype=torch.float64, device="cuda"))
    assert (seg_t if which == "segmentedMap" else vm_t).dtype == getattr(torch, dtype)
    assert_same_as_host(tout, hout)
    assert np.array_equal(host(vm_t), f["c%d_vm_out" % c])


# ---- 3. the reference's driver loop in torch ---------------------------------------------------------------------------
def test_reference_loop_in_torch_reproduces_the_whole_run():
    """VRG:47-117 written in torch around the tensor update(): the iteration count and labels of the whole-run fixture."""
    m = mod()
    g = load_golden("tube_clean")
    data, vm = cuda(g["data"]), cuda(g["value_map_in"])
    segmented = torch.nonzero(vm == 0)
    seg_map = torch.zeros_like(vm)
    seg_map[tuple(segmented.T)] = 1
    segmented, seg_map, vm, ib, ob, ip, op = m.update(data, segmented, seg_map, vm, g["H"])
    it = 1
    while it <= 200:
        allb = torch.cat((ib, ob))
        idx = tuple(allb.T)
        n_in = int(((vm == 0) | (vm == 1)).sum())
        n_out = int(((vm == 2) | (vm == 3)).sum())
        mask = torch.logical_xor(seg_map[idx] != 0, ip[idx] / n_in >= op[idx] / n_out)
        flips = allb[mask]
        if len(flips) == 0:
            break
        segmented, seg_map, vm, ib, ob, ip, op = m.update(data, segmented, seg_map, vm, g["H"], flips, ib, ob, ip, op)
        it += 1
    assert it == g["iterations"]
    assert np.array_equal(host(vm), g["labels"]) and np.array_equal(host(seg_map) == 1, g["seg_bool"])
    assert np.array_equal(host(segmented), np.argwhere(g["seg_bool"]))


# ---- 4. flips ----------------------------------------------------------------------------------------------------------
def _state(g):
    """Host state after the init call, and fresh tensor copies of it."""
    h = state_after_init(g["data"], g["value_map_in"], g["H"])
    return h, tuple(cuda(x) for x in h[1:3]) + tuple(cuda(x) for x in h[5:7])


def test_flips_in_every_form():
    m = mod()
    g = load_golden("tube_clean")
    h0, _ = _state(g)
    flips = first_flips(h0)
    d_t = cuda(g["data"])
    forms = {"cuda_int64": (cuda(flips), flips), "cuda_int32": (cuda(flips, torch.int32), flips), "host": (flips, flips),
             "host_list": (flips.tolist(), flips),
             "empty": (torch.zeros((0, 3), dtype=torch.int64, device="cuda"), np.zeros((0, 3), dtype=np.int64))}
    for name, (ft, fh) in forms.items():
        h, (seg_t, vm_t, ip_t, op_t) = _state(g)
        hout = m.update(g["data"], h[0], h[1], h[2], g["H"], fh, h[3], h[4], h[5], h[6])
        tout = m.update(d_t, cuda(h[0]), seg_t, vm_t, g["H"], ft, None, None, ip_t, op_t)
        assert_same_as_host(tout, hout)
        if name == "empty":  # nothing flips: the state and the bands are those of the init call
            assert np.array_equal(host(vm_t), h0[2]) and bits(host(tout[3])) == bits(h0[3])


def test_points_outside_the_bands_are_ignored_and_outside_the_volume_rejected():
    m = mod()
    g = load_golden("tube_clean")
    h, (seg_t, vm_t, ip_t, op_t) = _state(g)
    d_t = cuda(g["data"])
    far = np.array([[0, 0, 0], [1, 2, 3]])  # label 3, far from every seed
    hout = m.update(g["data"], h[0], h[1].copy(), h[2].copy(), g["H"], far, h[3], h[4], h[5].copy(), h[6].copy())
    tout = m.update(d_t, cuda(h[0]), seg_t, vm_t, g["H"], cuda(far), None, None, ip_t, op_t)
    assert_same_as_host(tout, hout)
    assert np.array_equal(host(vm_t), h[2]) and bits(host(tout[3])) == bits(h[3])
    before = [bits(host(t)) for t in (seg_t, vm_t, ip_t, op_t)]
    good = first_flips(h)
    for bad in (np.array([[0, 0, 99]]), np.concatenate([good, [[0, -1, 0]], good]), np.array([[g["data"].shape[0], 0, 0]])):
        with pytest.raises(ValueError, match="outside the volume"):
            m.update(d_t, cuda(h[0]), seg_t, vm_t, g["H"], cuda(bad), None, None, ip_t, op_t)
        assert [bits(host(t)) for t in (seg_t, vm_t, ip_t, op_t)] == before  # bit-unchanged


# ---- 5. layouts --------------------------------------------------------------------------------------------------------
def test_f_ordered_tensors():
    g = load_golden("forest_two_trees")  # (40, 56, 72): the three axes differ
    data_f, vm_f = np.asfortranarray(g["data"]), np.asfortranarray(g["value_map_in"])
    t1, h1 = init_and_flips(data_f, vm_f, g["H"])
    assert not t1[1].is_contiguous() and t1[1].permute(2, 1, 0).is_contiguous()
    assert_same_as_host(t1, h1)
    # F-ordered data, C-ordered maps: the maps are worked on as copies and written back
    t1c, h1c = init_and_flips(data_f, np.ascontiguousarray(vm_f), g["H"])
    assert_same_as_host(t1c, h1c)
    assert bits(host(t1c[2])) == bits(host(t1[2]))


def test_strided_views_are_written_back():
    m = mod()
    g = load_golden("forest40")
    Z, Y, X = g["data"].shape
    h, _ = _state(g)
    flips = first_flips(h)

    def strided(a, dtype, fill):
        big = torch.full((Z, Y, 2 * X), fill, dtype=dtype, device="cuda")
        v = big[:, :, ::2]
        v.copy_(cuda(a).to(dtype))
        assert not v.is_contiguous()
        return big, v
    bd, d = strided(g["data"], torch.float64, -7.0)
    bs, seg_t = strided(h[1], torch.int32, 9)
    bv, vm_t = strided(h[2], torch.int16, 9)
    bi, ip_t = strided(h[5], torch.float64, -1.0)
    bo, op_t = strided(h[6], torch.float64, -1.0)
    hout = m.update(g["data"], h[0], h[1].astype(np.int32), h[2].astype(np.int16), g["H"], flips, h[3], h[4], h[5], h[6])
    tout = m.update(d, cuda(h[0]), seg_t, vm_t, g["H"], cuda(flips), None, None, ip_t, op_t)
    assert tout[1] is seg_t and tout[2] is vm_t and tout[5] is ip_t and tout[6] is op_t
    assert_same_as_host(tout, hout)
    for big, fill in ((bd, -7.0), (bs, 9), (bv, 9), (bi, -1.0), (bo, -1.0)):
        assert bool((big[:, :, 1::2] == fill).all())  # the gaps are untouched


def _image():
    rng = np.random.default_rng(3)
    img = np.zeros((40, 48)); img[10:30, 20:26] = 1.0
    img = np.round((img + rng.normal(0, 0.1, img.shape)) * 64) / 64
    vm = np.full(img.shape, 3); vm[18:20, 22:24] = 0
    return img, vm


def test_two_dimensional_inputs():
    img, vm = _image()
    t1, h1 = init_and_flips(img, vm, 2.25)
    assert tuple(t1[3].shape)[1:] == (2,)
    assert_same_as_host(t1, h1)
    t1, h1 = init_and_flips(np.asfortranarray(img), np.asfortranarray(vm), 2.25)
    assert_same_as_host(t1, h1)


def test_one_dimensional_inputs():
    rng = np.random.default_rng(5)
    line = np.zeros(300); line[100:180] = 1.0
    line = np.round((line + rng.normal(0, 0.1, line.shape)) * 64) / 64
    vm = np.full(line.shape, 3); vm[140:142] = 0
    t1, h1 = init_and_flips(line, vm, 2.25)
    assert tuple(t1[3].shape)[1:] == (1,)
    assert_same_as_host(t1, h1)


def test_intensity_dtypes():
    g = load_golden("straight_line")  # int64 intensities
    for dt in (torch.int32, torch.int16, torch.uint8, torch.float32):
        t1, h1 = init_and_flips(g["data"].astype(getattr(np, str(dt).split(".")[1])), g["value_map_in"], g["H"])
        assert_same_as_host(t1, h1)


# ---- 6. errors and streams ---------------------------------------------------------------------------------------------
def test_errors():
    m = mod()
    g = load_golden("tube_clean")
    h, (seg_t, vm_t, ip_t, op_t) = _state(g)
    d_t = cuda(g["data"])
    flips = cuda(first_flips(h))
    before = [bits(host(t)) for t in (seg_t, vm_t, ip_t, op_t)]
    H = g["H"]
    with pytest.raises(TypeError):
        m.update(g["data"], h[0], seg_t, vm_t, H, flips, None, None, ip_t, op_t)  # host data
    with pytest.raises(TypeError):
        m.update(d_t, h[0], h[1], vm_t, H, flips, None, None, ip_t, op_t)  # host segmentedMap
    with pytest.raises(TypeError):
        m.update(d_t, h[0], seg_t, vm_t, H, flips, None, None, h[5], op_t)  # host innerProb
    with pytest.raises(TypeError):
        m.update(g["data"], h[0], h[1], h[2], H, first_flips(h), None, None, ip_t, h[6])  # host maps, tensor innerProb
    with pytest.raises(TypeError):
        m.update(d_t, h[0], seg_t, vm_t, H, flips, None, None, ip_t.to(torch.float32), op_t)  # wrong dtype
    with pytest.raises(TypeError):
        m.update(d_t, h[0], seg_t, vm_t, H, flips.to(torch.float64), None, None, ip_t, op_t)  # fractional coordinates
    with pytest.raises(ValueError):
        m.update(d_t, h[0], seg_t[:, :, :20], vm_t, H, flips, None, None, ip_t, op_t)  # shapes differ
    with pytest.raises(ValueError):
        m.update(d_t, h[0], seg_t, vm_t, H, flips, None, None, ip_t[:, :, :20], op_t)
    nan = d_t.clone(); nan[0, 0, 0] = float("nan")
    with pytest.raises(ValueError):
        m.update(nan, h[0], seg_t, vm_t, H, flips, None, None, ip_t, op_t)
    assert [bits(host(t)) for t in (seg_t, vm_t, ip_t, op_t)] == before  # bit-unchanged after every error
    from arterynetwork_b200 import _native as nat
    big = np.random.default_rng(2).normal(0, 1, (48, 48, 48))  # continuous data: 110592 distinct intensities
    vm_big = np.full(big.shape, 3); vm_big[20:22, 20:22, 20:22] = 0
    seg_big = (vm_big == 0).astype(np.int64)
    vb, sb = cuda(vm_big), cuda(seg_big)
    with pytest.raises(nat.LevelsError):
        m.update(big, np.argwhere(seg_big), seg_big.copy(), vm_big.copy(), H)  # the host path's error
    with pytest.raises(nat.LevelsError):
        m.update(cuda(big), np.argwhere(seg_big), sb, vb, H)
    assert np.array_equal(host(vb), vm_big) and np.array_equal(host(sb), seg_big)


def test_inputs_from_a_busy_side_stream():
    """Inputs produced on a non-default stream behind a slow kernel, the calls made inside that stream's context: they run
    on torch's current stream, so they see the finished inputs without any synchronisation by the caller."""
    m = mod()
    g = load_golden("forest40")
    h, _ = _state(g)
    flips = first_flips(h)
    hout = m.update(g["data"], h[0], h[1].copy(), h[2].copy(), g["H"], flips, h[3], h[4], h[5].copy(), h[6].copy())
    srcs = [cuda(g["data"]), cuda(h[1]), cuda(h[2]), cuda(flips)]
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)  # about 0.1 s of device clock ahead of the inputs
        d, seg_t, vm_t, fl = (s.clone() for s in srcs)
        tout = m.update(d, cuda(h[0]), seg_t, vm_t, g["H"], fl)
        res = [host(x) for x in tout]
    for i in (1, 2, 3, 4, 5, 6):
        assert bits(res[i]) == bits(hout[i]), i


# ---- 7. full size ------------------------------------------------------------------------------------------------------
def test_c2_init_then_first_decision_flips():
    """One C2-sized pair of calls (init, then the flips of the first decision): tensors against host arrays, bit for bit."""
    import bench
    shape = bench.WORKLOADS["c2"]
    d, v = bench.device_phantom(shape, 0, 0, shape[0], 0)
    torch.cuda.synchronize()
    t1, h1 = init_and_flips(host(d), host(v), 2.25)
    assert_same_as_host(t1, h1)
    assert len(h1[3]) > 0 and len(h1[4]) > len(h1[3])  # both bands present after the flips
