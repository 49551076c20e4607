"""The drop-in functions on CUDA tensors (B200 only): ``variationalRegionGrowing`` with device-resident inputs, the typed label
ingest / egress and the device compaction of the segmented rows behind it, and the mask-side drop-ins on tensors.

The bar is the host path: the same labels, segmentedMap, segmented rows, stdout and LAST_RUN counters as the NumPy call on
the same input, and the committed fixtures' results."""
import contextlib
import io
import warnings

import numpy as np
import pytest

from golden_util import golden_names, load_golden
from mask_golden_util import load_mask_case, mask_names, rule_names

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

TABLE_NAMES = [n for n in golden_names() if not n.endswith("_cont")]
MODES = ["f64_dense", "f64_band", "index"]
LABEL_DTYPES = ["uint8", "int8", "int16", "int32", "int64", "float32", "float64"]


def mod():
    from arterynetwork_b200 import variationalRegionGrowing as m
    return m


def call(data, vm, **kw):
    """One drop-in call: (segmented, segmentedMap, valueMap), stdout, LAST_RUN counters, order-dependence warnings."""
    m = mod()
    buf = io.StringIO()
    with warnings.catch_warnings(record=True) as w, contextlib.redirect_stdout(buf):
        warnings.simplefilter("always")
        out = m.variationalRegionGrowing(data, vm, **kw)
    # kernel_launches depends on whether the batches ran as CUDA graphs (not on the legacy default stream), not on the result
    counters = {k: v for k, v in m.LAST_RUN.items() if k not in ("host_seconds", "kernel_launches")}
    return out, buf.getvalue(), counters, [str(x.message) for x in w if issubclass(x.category, m.VRGOrderDependenceWarning)]


def cuda(a, dtype=None):
    t = torch.from_numpy(np.asarray(a)).cuda()  # keeps the array's strides (an F-ordered array stays F-ordered)
    return t if dtype is None else t.to(dtype)


def host(t):
    return t.cpu().numpy()


def assert_same_as_host(tout, nout, vm_t):
    """Tensor results against the host call's on the same input."""
    (seg_t, map_t, vm_out), out_t, run_t, warn_t = tout
    (seg_n, map_n, vm_n), out_n, run_n, warn_n = nout
    assert vm_out is vm_t
    assert np.array_equal(host(vm_t), vm_n)
    assert map_t.is_cuda and map_t.dtype == torch.int64 and map_t.is_contiguous() and map_t.device == vm_t.device
    assert tuple(map_t.shape) == map_n.shape and np.array_equal(host(map_t), map_n)
    assert seg_t.is_cuda and seg_t.dtype == torch.int64 and tuple(seg_t.shape) == seg_n.shape
    assert np.array_equal(host(seg_t), seg_n)
    assert out_t == out_n
    assert run_t == run_n
    assert warn_t == warn_n


# ---- 1. golden fixtures ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", TABLE_NAMES)
def test_golden_fixtures_through_tensors(name):
    g = load_golden(name)
    kw = dict(H=g["H"], maxSegmentSize=g["max_segment_size"])
    nout = call(g["data"], g["value_map_in"].copy(), **kw)
    vm_t = cuda(g["value_map_in"])  # int64, the reference's dtype
    tout = call(cuda(g["data"]), vm_t, **kw)
    assert_same_as_host(tout, nout, vm_t)
    (seg_t, map_t, _), out_t, run_t, _ = tout
    assert vm_t.dtype == torch.int64 and np.array_equal(host(vm_t), g["labels"])
    assert np.array_equal(host(map_t) == 1, g["seg_bool"])
    assert np.array_equal(host(seg_t), np.argwhere(g["seg_bool"]))
    assert out_t == str(g["stdout"])
    assert run_t["iterations"] == g["iterations"]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", ["tube_clean", "excl32", "forest40", "maxseg"])
def test_golden_fixtures_in_every_intensity_mode(name, mode, monkeypatch):
    monkeypatch.setattr(mod(), "INTENSITY", mode)
    g = load_golden(name)
    kw = dict(H=g["H"], maxSegmentSize=g["max_segment_size"])
    nout = call(g["data"], g["value_map_in"].astype(np.uint8), **kw)
    vm_t = cuda(g["value_map_in"], torch.uint8)
    tout = call(cuda(g["data"]), vm_t, **kw)
    assert_same_as_host(tout, nout, vm_t)
    assert np.array_equal(host(vm_t), g["labels"]) and tout[1] == str(g["stdout"])


# ---- 2. label dtypes ---------------------------------------------------------------------------------------------------
def _bad_values(dtype):
    if dtype == "uint8":
        return [5, 255]
    if dtype.startswith("int"):
        return [5, -1]
    return [5.0, -1.0, 2.5, float("nan"), 4.000001]


@pytest.mark.parametrize("dtype", LABEL_DTYPES)
def test_label_dtypes(dtype):
    g = load_golden("excl32")  # labels 0, 3 and 4
    tdt = getattr(torch, dtype)
    kw = dict(H=g["H"], maxSegmentSize=g["max_segment_size"])
    nout = call(g["data"], g["value_map_in"].astype(getattr(np, dtype)), **kw)
    vm_t = cuda(g["value_map_in"], tdt)
    tout = call(cuda(g["data"]), vm_t, **kw)
    assert vm_t.dtype == tdt
    assert_same_as_host(tout, nout, vm_t)
    assert np.array_equal(host(vm_t), g["labels"])
    data_t = cuda(g["data"])
    for bad in _bad_values(dtype):
        v = cuda(g["value_map_in"], tdt)
        v.view(-1)[v.numel() // 2 + 7] = bad
        bits = v.view(torch.uint8).clone()
        with pytest.raises(ValueError):
            call(data_t, v, **kw)
        assert torch.equal(v.view(torch.uint8), bits), bad  # bit-unchanged (NaN included)


# ---- 3. data dtypes and layouts ----------------------------------------------------------------------------------------
def test_int_and_float32_data():
    g = load_golden("straight_line")  # int64 intensities
    nout = call(g["data"], g["value_map_in"].copy())
    vm_t = cuda(g["value_map_in"])
    assert_same_as_host(call(cuda(g["data"]), vm_t), nout, vm_t)
    for dt in (torch.int32, torch.int16, torch.uint8):
        vm_t = cuda(g["value_map_in"])
        assert_same_as_host(call(cuda(g["data"], dt), vm_t), nout, vm_t)
    g = load_golden("tube_clean")
    d32 = g["data"].astype(np.float32)
    nout = call(d32, g["value_map_in"].copy())
    vm_t = cuda(g["value_map_in"])
    assert_same_as_host(call(cuda(d32), vm_t), nout, vm_t)


def test_f_ordered_tensors():
    g = load_golden("forest_two_trees")  # (40, 56, 72): the three axes differ
    kw = dict(H=g["H"], maxSegmentSize=g["max_segment_size"])  # the fixture's arguments (its run ends by convergence)
    data_f, vm_f = np.asfortranarray(g["data"]), np.asfortranarray(g["value_map_in"])
    nout = call(data_f, vm_f.copy(order="F"), **kw)
    d, v = cuda(data_f), cuda(vm_f)
    assert not d.is_contiguous() and d.permute(2, 1, 0).is_contiguous()
    tout = call(d, v, **kw)
    assert_same_as_host(tout, nout, v)
    assert not v.is_contiguous() and np.array_equal(host(v), g["labels"])
    assert np.array_equal(host(tout[0][0]), np.argwhere(g["seg_bool"])) and tout[1] == str(g["stdout"])
    # F-ordered data with a C-ordered valueMap (and the other way round): the map is worked on as a copy and written back
    v2 = cuda(g["value_map_in"])
    assert_same_as_host(call(d, v2, **kw), nout, v2)
    v3 = cuda(vm_f, torch.uint8)
    nout8 = call(g["data"], g["value_map_in"].astype(np.uint8), **kw)
    assert_same_as_host(call(cuda(g["data"]), v3, **kw), nout8, v3)
    assert np.array_equal(host(v3), g["labels"])


def test_one_and_two_dimensional_inputs():
    rng = np.random.default_rng(3)
    img = np.zeros((40, 48)); img[10:30, 20:26] = 1.0
    img = np.round((img + rng.normal(0, 0.1, img.shape)) * 64) / 64
    vm = np.full(img.shape, 3); vm[18:20, 22:24] = 0
    nout = call(img, vm.copy(), maxSegmentSize=10 ** 9)
    v = cuda(vm)
    assert_same_as_host(call(cuda(img), v, maxSegmentSize=10 ** 9), nout, v)
    # 2-D, F-ordered
    img_f, vm_f = np.asfortranarray(img), np.asfortranarray(vm)
    nout = call(img_f, vm_f.copy(order="F"), maxSegmentSize=10 ** 9)
    v = cuda(vm_f)
    assert_same_as_host(call(cuda(img_f), v, maxSegmentSize=10 ** 9), nout, v)
    # 1-D: a bright run in a noisy line
    line = np.zeros(300); line[100:180] = 1.0
    line = np.round((line + rng.normal(0, 0.1, line.shape)) * 64) / 64
    vm1 = np.full(line.shape, 3); vm1[140:142] = 0
    nout = call(line, vm1.copy(), maxSegmentSize=10 ** 9)
    v = cuda(vm1)
    tout = call(cuda(line), v, maxSegmentSize=10 ** 9)
    assert_same_as_host(tout, nout, v)
    assert tuple(tout[0][0].shape) == (nout[0][0].shape[0], 1)


def test_strided_views_are_written_back():
    g = load_golden("forest40")
    Z, Y, X = g["data"].shape
    big_vm = torch.full((Z, Y, 2 * X), 9, dtype=torch.int32, device="cuda")
    big_d = torch.full((Z, 2 * Y, X), -7.0, dtype=torch.float64, device="cuda")
    v = big_vm[:, :, ::2]
    d = big_d[:, ::2, :]
    v.copy_(cuda(g["value_map_in"]))
    d.copy_(cuda(g["data"]))
    assert not v.is_contiguous() and not d.is_contiguous()
    kw = dict(H=g["H"], maxSegmentSize=g["max_segment_size"])
    nout = call(g["data"], g["value_map_in"].astype(np.int32), **kw)
    tout = call(d, v, **kw)
    assert_same_as_host(tout, nout, v)
    assert np.array_equal(host(v), g["labels"])
    assert bool((big_vm[:, :, 1::2] == 9).all()) and bool((big_d[:, 1::2, :] == -7.0).all())  # the gaps are untouched


@pytest.mark.parametrize("dtype", ["uint8", "int16", "float32"])
def test_odd_storage_offsets(dtype):
    g = load_golden("excl32")
    n = g["data"].size
    tdt = getattr(torch, dtype)
    raw_v = torch.zeros(n + 3, dtype=tdt, device="cuda")
    raw_d = torch.zeros(n + 1, dtype=torch.float64, device="cuda")
    v = raw_v[3:].view(g["data"].shape)
    d = raw_d[1:].view(g["data"].shape)
    assert v.storage_offset() == 3 and d.storage_offset() == 1 and d.data_ptr() % 16 == 8
    v.copy_(cuda(g["value_map_in"]))
    d.copy_(cuda(g["data"]))
    kw = dict(H=g["H"], maxSegmentSize=g["max_segment_size"])
    nout = call(g["data"], g["value_map_in"].astype(getattr(np, dtype)), **kw)
    tout = call(d, v, **kw)
    assert_same_as_host(tout, nout, v)
    assert np.array_equal(host(v), g["labels"])
    assert bool((raw_v[:3] == 0).all()) and float(raw_d[0]) == 0.0


# ---- 4. other paths ----------------------------------------------------------------------------------------------------
def test_resume_from_a_returned_tensor_map():
    g = load_golden("maxseg")  # stops at maxSegmentSize = 50 with band labels 1 / 2 in the map
    vm_n = g["value_map_in"].copy()
    call(g["data"], vm_n, maxSegmentSize=50)
    vm_t = cuda(g["value_map_in"])
    d = cuda(g["data"])
    first = call(d, vm_t, maxSegmentSize=50)
    assert "(Max segment size reached)" in first[1]
    assert set(np.unique(host(vm_t)).tolist()) >= {1, 2}
    nout = call(g["data"], vm_n, maxSegmentSize=10 ** 9)
    assert_same_as_host(call(d, vm_t, maxSegmentSize=10 ** 9), nout, vm_t)


def test_continuous_fallback_with_tensors():
    """More than 65536 distinct intensities: the brute-force Parzen path on attached tensors, as on host arrays."""
    rng = np.random.default_rng(7)
    data = np.zeros((40, 41, 41)); data[17:23, 17:23, 8:34] = 1.0
    data = data + rng.normal(0, 0.1, data.shape)
    vm = np.full(data.shape, 3); vm[19:21, 19:21, 20:22] = 0
    nout = call(data, vm.copy(), maxSegmentSize=10 ** 9)
    v = cuda(vm)
    assert_same_as_host(call(cuda(data), v, maxSegmentSize=10 ** 9), nout, v)


def test_errors(monkeypatch):
    m = mod()
    data = torch.zeros((6, 6, 40), dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError):
        m.variationalRegionGrowing(data, torch.full(data.shape, 3, device="cuda"))  # empty seed
    with pytest.raises(ValueError):
        m.variationalRegionGrowing(data, torch.zeros(data.shape, dtype=torch.int64, device="cuda"))  # no boundary
    vm = torch.full(data.shape, 3, device="cuda"); vm[2, 2, 2] = 0
    bad = data.clone(); bad[0, 0, 0] = float("nan")
    before = vm.clone()
    with pytest.raises(ValueError):
        m.variationalRegionGrowing(bad, vm)
    assert torch.equal(vm, before)
    with pytest.raises(ValueError):
        m.variationalRegionGrowing(data[:, :, :20], vm)  # shapes differ
    with pytest.raises(TypeError):
        m.variationalRegionGrowing(host(data), vm)  # mixed: host data, tensor map
    with pytest.raises(TypeError):
        m.variationalRegionGrowing(data, host(vm))  # mixed: tensor data, host map
    with pytest.raises(TypeError):
        m.variationalRegionGrowing(data, vm.to(torch.bool))
    monkeypatch.setattr(m, "DEVICES", [0])
    with pytest.raises(NotImplementedError, match="DEVICES"):
        m.variationalRegionGrowing(data, vm)
    monkeypatch.setattr(m, "DEVICES", None)
    monkeypatch.setattr(m, "LIST_ORDER", True)
    with pytest.raises(NotImplementedError, match="LIST_ORDER"):
        m.variationalRegionGrowing(data, vm)
    assert torch.equal(vm, before)


# ---- 5. stream ordering ------------------------------------------------------------------------------------------------
def test_inputs_from_a_busy_side_stream():
    """Inputs produced on a non-default stream behind a slow kernel, the call made inside that stream's context: the call
    runs on torch's current stream, so it sees the finished inputs without any synchronisation by the caller."""
    g = load_golden("forest40")
    d0, v0 = cuda(g["data"]), cuda(g["value_map_in"])
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)  # about 0.1 s of device clock ahead of the inputs
        d = d0 * 1.0
        v = v0.clone()
        tout = call(d, v, H=g["H"], maxSegmentSize=g["max_segment_size"])
        labels = host(v)
        segmap = host(tout[0][1])
    assert np.array_equal(labels, g["labels"]) and np.array_equal(segmap == 1, g["seg_bool"])
    assert tout[1] == str(g["stdout"])


# ---- 6. engine level ---------------------------------------------------------------------------------------------------
def _engine_agreement(eng, shape):
    from arterynetwork_b200 import _native as nat
    codes = dict(zip(LABEL_DTYPES, range(7)))
    lab = eng.labels()
    seg_i64 = eng.segmented_map_i64()
    rows = eng.segmented()
    for name, code in codes.items():
        out = torch.full(shape, 7, dtype=getattr(torch, name), device="cuda")
        eng.labels_device_typed(out.data_ptr(), code)
        torch.cuda.synchronize()
        assert np.array_equal(host(out), lab.astype(getattr(np, name))), name
        eng.labels_device_typed(out.data_ptr(), code, segmented_only=True)
        torch.cuda.synchronize()
        assert np.array_equal(host(out), seg_i64.astype(getattr(np, name))), name
    assert codes["int64"] == nat.DTYPE_I64
    r = torch.empty((len(rows), 3), dtype=torch.int64, device="cuda")
    assert eng.segmented_device(r.data_ptr(), len(rows)) == len(rows)
    assert np.array_equal(host(r), rows)
    assert eng.segmented_device(None, 0) == len(rows)
    few = torch.full((5, 3), -1, dtype=torch.int64, device="cuda")
    assert eng.segmented_device(few.data_ptr(), 5) == len(rows)
    assert np.array_equal(host(few), rows[:5])


def test_engine_entry_points_on_a_fixture():
    from arterynetwork_b200.engine import VRGEngine
    g = load_golden("excl32")
    with VRGEngine(g["data"].shape, H=g["H"], max_segment_size=g["max_segment_size"], intensity="index") as eng:
        eng.upload(g["data"], g["value_map_in"].astype(np.uint8))
        eng.init()
        eng.run()
        assert np.array_equal(eng.labels(), g["labels"])
        _engine_agreement(eng, g["data"].shape)


def test_engine_entry_points_on_c2():
    import bench
    from arterynetwork_b200 import _native as nat
    from arterynetwork_b200.engine import VRGEngine
    shape = bench.WORKLOADS["c2"]
    d, v = bench.device_phantom(shape, 0, 0, shape[0], 0)
    v64 = v.to(torch.int64)
    torch.cuda.synchronize()
    with VRGEngine(shape, max_segment_size=10 ** 15, intensity="index") as eng:
        eng.attach_device(d.data_ptr(), v.data_ptr())
        eng.init()
        res = eng.run()
        ref = eng.labels()
        _engine_agreement(eng, shape)
        # the same run from the int64 map, read by vrg_init in its own dtype
        eng.attach_device_typed(d.data_ptr(), v64.data_ptr(), nat.DTYPE_I64)
        eng.init()
        res64 = eng.run()
        assert (res64["iterations"], res64["n_in"], res64["n_out"]) == (res["iterations"], res["n_in"], res["n_out"])
        assert np.array_equal(eng.labels(), ref)


# ---- 7. mask drop-ins --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", mask_names())
def test_mask_dropins_on_tensors(name):
    from arterynetwork_b200.generateVesselVolume import distance_transform_edt, labelVolume, maskVolume
    g = load_mask_case(name)
    m = g["mask"].astype(np.uint8)
    for arr in (m, np.asfortranarray(m)):
        e_n = distance_transform_edt(arr)
        e_t = distance_transform_edt(cuda(arr))
        assert e_t.is_cuda and e_t.dtype == torch.float64 and np.array_equal(host(e_t), e_n)
        assert np.array_equal(e_n, g["edt"])
        lab_n, res_n = labelVolume(arr)
        lab_t, res_t = labelVolume(cuda(arr))
        assert lab_t.is_cuda and lab_t.dtype == torch.int32 and np.array_equal(host(lab_t), lab_n)
        assert res_t == res_n and isinstance(res_t, list)
    vol = np.arange(m.size, dtype=np.float64).reshape(m.shape)
    mv = maskVolume(cuda(vol), cuda(m))
    assert mv.is_cuda and np.array_equal(host(mv), maskVolume(vol, m))


@pytest.mark.parametrize("name", rule_names())
def test_vessel_mask_on_tensors(name):
    from arterynetwork_b200.generateVesselVolume import vesselnessToVesselMask
    g = load_mask_case(name)
    for vess, brain in ((g["vesselness"], g["brain"]), (np.asfortranarray(g["vesselness"]), np.asfortranarray(g["brain"]))):
        kw = dict(minComponentSize=g["min_size"], return_info=True)
        with contextlib.redirect_stdout(io.StringIO()) as b_n:
            out_n, info_n = vesselnessToVesselMask(vess, brain, **kw)
        with contextlib.redirect_stdout(io.StringIO()) as b_t:
            out_t, info_t = vesselnessToVesselMask(cuda(vess), cuda(brain), **kw)
        assert out_t.is_cuda and out_t.dtype == torch.uint8 and np.array_equal(host(out_t), out_n)
        assert np.array_equal(out_n, g["vessel_mask"])
        assert info_t == info_n and b_t.getvalue() == b_n.getvalue()
    with pytest.raises(TypeError):
        vesselnessToVesselMask(cuda(g["vesselness"]), g["brain"])


# ---- 8. resident pipeline ----------------------------------------------------------------------------------------------
def test_resident_pipeline_equals_host_pipeline():
    """vesselness -> vessel mask -> seeds -> VRG -> distance transform, all on CUDA tensors, against the same steps on host
    arrays."""
    from arterynetwork_b200.generateVesselVolume import distance_transform_edt, labelVolume, vesselnessToVesselMask
    from arterynetwork_b200.phantom import make_phantom
    shape = (48, 64, 96)
    vess, _, _ = make_phantom(shape, seed=1, cell=shape, margin=4, depth=3, root_r2=9, min_len=10, max_len=20)
    brain = np.zeros(shape, dtype=np.uint8); brain[2:-2, 2:-2, 2:-2] = 1
    kw = dict(edgeDistance=3, fraction=0.6, minComponentSize=20)

    def pipeline(v, b, xp_where):
        with contextlib.redirect_stdout(io.StringIO()) as buf:
            mask = vesselnessToVesselMask(v, b, **kw)
            labeled, comps = labelVolume(mask)
            seeds = labeled == 1  # the first component seeds the growth
            vm = xp_where(seeds)
            segmented, segmap, vm = mod().variationalRegionGrowing(v, vm, maxSegmentSize=10 ** 9)
            radii = distance_transform_edt(segmap)
        return mask, comps, vm, segmented, segmap, radii, buf.getvalue()

    h = pipeline(vess, brain, lambda s: np.where(s, 0, 3))
    t = pipeline(cuda(vess), cuda(brain), lambda s: torch.where(s, 0, 3))
    assert int(h[0].sum()) > 0 and len(h[1]) > 1
    for a, b in zip(h[:-1], t[:-1]):
        if isinstance(a, list):
            assert a == b
        else:
            assert b.is_cuda and np.array_equal(host(b), a)
    assert t[-1] == h[-1]
