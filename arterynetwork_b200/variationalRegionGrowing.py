"""Drop-in for the reference module ``Code/variationalRegionGrowing.py``.

Same entry points, same arguments, same return values, same stdout lines
(VRG:10, VRG:94-96, VRG:124, VRG:263, VRG:284-314) -- the iteration runs on
B200s through ``libvrg_b200.so``.

    from arterynetwork_b200.variationalRegionGrowing import variationalRegionGrowing
    segmented, segmentedMap, valueMap = variationalRegionGrowing(dataArray, valueMap)

CUDA tensors: when ``valueMap`` is a CUDA tensor (and ``dataArray`` a CUDA tensor on the same device) the call runs on
that device and torch's current stream and returns tensors -- ``valueMap`` is the same tensor, updated in place and kept
in its own dtype (uint8, int8, int16, int32, int64, float32 or float64; the kernels read and write the labels in that dtype),
``segmentedMap`` a new C-contiguous int64 CUDA tensor, ``segmented`` an int64 CUDA tensor (K, ndim) in C order of the
caller's axes; stdout, ``LAST_RUN`` and the warning as below.  Nothing of volume size crosses PCIe.  C-contiguous tensors
are used as they are, F-contiguous ones (``torch.from_numpy(nibabel_volume).cuda()``) through their reversed-axes view,
other strides through a contiguous copy whose labels are copied back; intensities other than float64 are converted once.
On any error the caller's ``valueMap`` is left bit-unchanged.  ``DEVICES`` and ``LIST_ORDER = True`` take host arrays only.
``update`` takes CUDA tensors the same way (see its docstring): state, flips, band rows and Parzen sums stay on the device,
and the results are bit-identical to the call on host arrays.

Module switches (the reference has none; defaults reproduce it):

``DEVICES``   ``None`` = one GPU (``DEVICE``); a list of CUDA ordinals or ``"all"`` =
              the volume is cut into z-slabs, one per GPU, inside this one process
              (one host thread per GPU, halo planes and the statistics all-reduce
              move over NVLink peer memory) -- the call itself does not change.
``INTENSITY`` how the sweep reads intensities (``index`` | ``f64_band`` | ``f64_dense``).
``MAX_SECONDS`` the reference's 120 s wall-clock exit (VRG:97); ``None`` disables it.
``LIST_ORDER`` ``False`` = the order-free result (below); ``True`` = the strict engine (``csrc/vrg_strict.cu``): the
              reference WITH the effects of its list processing order -- flipped points walked in ``allBnd`` order,
              stale band labels kept in ``valueMap``, drifting running Parzen sums, ``segmented`` rows in the
              reference's own order (VRG:156-259).  One GPU, level-table data, fresh maps (labels 0 / 3 / 4).

Differences from the reference, all deliberate (DESIGN.md "Boundary"):

* the caller's ``valueMap`` is still mutated in place and returned as the same
  object (VRG:137-228).  A map that already holds band labels (1, 2: the output
  of an earlier call) is read as the state those labels describe and the run
  resumes from it; the reference re-seeds such a map from label 0 only
  (VRG:44) and then dies with a ValueError at VRG:111 once its outer band list
  runs empty;
* an empty seed set or a seed without boundary raises ``ValueError`` (the
  reference dies with ``IndexError`` at VRG:88);
* ``segmented`` rows come back in C order (the reference's row order is the
  history of its list appends); as a set it is ``argwhere(segmentedMap == 1)``;
* the 120 s wall-clock exit (VRG:97) is kept (``MAX_SECONDS``) but is checked
  between batches of iterations; set ``MAX_SECONDS = None`` for parity runs;
* intensities are processed as float64 whatever the input dtype (the reference
  silently drops to float32 sums for float32 input under NumPy 2);
* results are those of the order-free restatement of the band state machine:
  bit-identical to the reference wherever the reference's own result does not
  depend on its list order (SURVEY.md section 8(a), quirks Q2-Q4).  Every call
  leaves its counters in ``LAST_RUN``; when the run touched a flip pattern on
  which the reference is order-dependent a ``VRGOrderDependenceWarning`` says so.
"""
from __future__ import annotations

import itertools
import sys
import time
import warnings
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from . import _native as nat
from .engine import VRGEngine

A = (2 * np.pi) ** (-0.5)  # VRG:7
MAX_SECONDS = 120.0  # VRG:97
ITER_MAX = 200  # VRG:56
DEVICE = 0
DEVICES = None  # None: DEVICE only; "all" or a list of CUDA ordinals: z-slabs over those GPUs, in this process
INTENSITY = "index"  # how the sweep reads intensities: f64_dense | f64_band | index | continuous
CONTINUOUS_MAX_VOXELS = 1 << 24  # fall back to the brute-force Parzen mode (continuous data) up to this volume size
HOST_THREADS = max(1, min(16, (__import__("os").cpu_count() or 8)))  # host-side conversions (label dtype, int64 segmentedMap) run in z-chunks on this many threads
LIST_ORDER = False  # True: bug-compatible list-order semantics (SURVEY.md section 8(f) N4), see the module docstring
LAST_RUN = {}  # result of the most recent call: iterations, exit_reason, n_in, ..., q_* order-dependence counters

_EXIT_SUFFIX = {nat.EXIT_CONVERGED: "", nat.EXIT_MAX_TIME: " (Max time reached)",
                nat.EXIT_MAX_SEGMENT: " (Max segment size reached)"}


class VRGOrderDependenceWarning(UserWarning):
    """The run applied flips on which the reference's sequential list processing is order-dependent (SURVEY.md
    section 8(a) Q2-Q4): the result returned is the order-free one; the reference's own may differ by its list order."""


def _as_zyx(a):
    """View ``a`` as a C-contiguous (Z, Y, X) array; returns (view3d, transposed?)."""
    a = np.asarray(a)
    if a.ndim > 3 or a.ndim == 0:
        raise NotImplementedError("variationalRegionGrowing: 1-D to 3-D volumes only, got ndim=%d" % a.ndim)
    transposed = a.ndim > 1 and a.flags.f_contiguous and not a.flags.c_contiguous
    if transposed:
        a = a.T  # nibabel-style F-ordered volume: the slowest axis becomes z (SURVEY.md section 8(e))
    return a.reshape((1,) * (3 - a.ndim) + a.shape), transposed


def _chunks(nz, parts):
    parts = max(1, min(parts, nz))
    b = [nz * i // parts for i in range(parts + 1)]
    return [(b[i], b[i + 1]) for i in range(parts) if b[i + 1] > b[i]]


def _pool_map(fn, items):
    items = list(items)
    if len(items) <= 1:
        return [fn(x) for x in items]
    with ThreadPoolExecutor(len(items)) as ex:
        return list(ex.map(fn, items))  # re-raises the first exception


def _labels_u8(vm3):
    """uint8 copy of the caller's valueMap (any numeric dtype), validated: integral labels 0..4 only."""
    if vm3.dtype == np.uint8:
        out = vm3 if vm3.flags.c_contiguous else np.ascontiguousarray(vm3)
        if out.size and int(out.max()) > 4:
            raise ValueError("valueMap may only hold the labels 0..4")
        return out
    out = np.empty(vm3.shape, dtype=np.uint8)

    def conv(zz):
        c = vm3[zz[0]:zz[1]]
        with np.errstate(invalid="ignore"):
            u = c.astype(np.uint8)
        out[zz[0]:zz[1]] = u
        return bool((u == c).all()) and (u.size == 0 or int(u.max()) <= 4)
    if not all(_pool_map(conv, _chunks(vm3.shape[0], HOST_THREADS))):
        raise ValueError("valueMap may only hold the labels 0..4")
    return out


def _device_list():
    if DEVICES is None:
        return [DEVICE]
    if isinstance(DEVICES, str):
        if DEVICES != "all":
            raise ValueError("DEVICES must be None, 'all' or a list of CUDA ordinals")
        import torch
        return list(range(torch.cuda.device_count()))
    return [int(d) for d in DEVICES]


class _Run:
    """One run of the path on one GPU or on z-slabs over several (same calls either way)."""

    def __init__(self, shape, H, max_segment_size, mode, devices):
        from .distributed import slab_bounds
        Z = shape[0]
        devices = devices[: max(1, min(len(devices), Z // max(1, 2 * nat.HALO)))]  # slabs of at least 4 planes
        if mode == "continuous":
            devices = devices[:1]  # brute-force Parzen mode: single slab
        self.shape, self.world = shape, len(devices)
        b = slab_bounds(Z, self.world) if self.world > 1 else [0, Z]
        self.bounds = b
        self.engines = [VRGEngine(shape, H=H, max_segment_size=max_segment_size, iter_max=ITER_MAX, device=d, intensity=mode,
                                  z_begin=b[r], z_end=b[r + 1], max_seconds=MAX_SECONDS or 0.0)
                        for r, d in enumerate(devices)]

    def close(self):
        for e in self.engines:
            e.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _each(self, fn):
        return _pool_map(fn, self.engines)

    def upload(self, data3, vm8):
        def up(e):
            d = data3[e.ext_lo:e.ext_hi]
            e.upload(d if d.dtype == np.float64 and d.flags.c_contiguous else np.ascontiguousarray(d, dtype=np.float64),
                     vm8[e.ext_lo:e.ext_hi])
        self._each(up)

    def run(self):
        if self.world > 1:
            levels = np.unique(np.concatenate(self._each(lambda e: e.scan_levels())))
            for e in self.engines:
                e.set_levels(levels)
            hs = (nat.vp * self.world)(*[e._h.value for e in self.engines])
            nat.check(self.engines[0].lib.vrg_p2p_connect_local(hs, self.world))

        def go(e):  # the ranks wait for each other on the device, so every handle needs its own host thread
            e.init()
            return e.run()
        return self._each(go)[0]

    def labels_into(self, out3):
        self._each(lambda e: nat.check(e.lib.vrg_download_labels(e._h, out3[e.z_begin:e.z_end].ctypes.data)))

    def segmented_map_i64_into(self, out3):
        self._each(lambda e: e.segmented_map_i64(out3[e.z_begin:e.z_end]))

    def segmented(self, at_most=None):
        return np.concatenate(self._each(lambda e: e.segmented(at_most)))

    def count_nonzero(self):
        return sum(self._each(lambda e: e.count_nonzero()))


def _warn_order_dependence(res):
    n = res["q_add_to_inside"] + res["q_remove_to_outside"] + res["q_cancel_repromoted"]
    if n:
        warnings.warn("variationalRegionGrowing: %d applied flips met a pattern on which the reference's list processing is "
                      "order-dependent (added-to-inside %d, removed-to-outside %d, cancelled-then-repromoted %d); the result "
                      "is the order-free one (see LAST_RUN)" % (n, res["q_add_to_inside"], res["q_remove_to_outside"],
                                                                res["q_cancel_repromoted"]),
                      VRGOrderDependenceWarning, stacklevel=3)


def _finish_lines(res, segmented, data3, nz=None):
    if nz is None:
        nz = sum(_pool_map(lambda zz: int(np.count_nonzero(data3[zz[0]:zz[1]])), _chunks(data3.shape[0], HOST_THREADS)))
    if res["exit_reason"] == nat.EXIT_MAX_ITER:  # VRG:118-120
        print('Segmented points are: \n', segmented if isinstance(segmented, np.ndarray) else segmented.cpu().numpy())
        print('Max iteration reached! Finished at iteration {}'.format(res["iterations"]))
    else:  # VRG:94-104
        print('Finished at iteration {}{}'.format(res["iterations"], _EXIT_SUFFIX[res["exit_reason"]]))
    print('Total segmented voxels: ' + '{}/{}'.format(segmented.shape[0], nz))


def _list_order_run(dataArray, valueMap, H, maxSegmentSize):
    """``LIST_ORDER = True``: the strict engine.  The list order is the raster order of the USER's axes, so an F-ordered
    volume is copied to C order instead of being transposed."""
    global LAST_RUN
    from .strict import StrictEngine
    if dataArray.ndim > 3 or dataArray.ndim == 0:
        raise NotImplementedError("variationalRegionGrowing: 1-D to 3-D volumes only, got ndim=%d" % dataArray.ndim)
    shape3 = (1,) * (3 - dataArray.ndim) + dataArray.shape
    data3 = np.ascontiguousarray(dataArray, dtype=np.float64).reshape(shape3)
    vm8 = _labels_u8(np.ascontiguousarray(valueMap).reshape(shape3))
    if not np.isin(vm8, (0, 3, 4)).all():
        raise ValueError("variationalRegionGrowing (LIST_ORDER): the initial valueMap may only hold the labels 0, 3 and 4")
    with StrictEngine(shape3, H=H, max_segment_size=maxSegmentSize, iter_max=ITER_MAX, device=DEVICE,
                      max_seconds=MAX_SECONDS or 0.0) as eng:
        eng.init(data3, vm8)
        res = eng.run()
        labels = eng.value_map()
        segmented = eng.segmented()[:, 3 - dataArray.ndim:]
    LAST_RUN = dict(res)
    valueMap[...] = labels.reshape(dataArray.shape)
    segmentedMap = (labels <= 1).astype(np.int64).reshape(dataArray.shape)
    _finish_lines(res, segmented, data3)
    return segmented, segmentedMap, valueMap


def _label_dtype_code(torch, dtype):
    return {torch.uint8: nat.DTYPE_U8, torch.int8: nat.DTYPE_I8, torch.int16: nat.DTYPE_I16, torch.int32: nat.DTYPE_I32,
            torch.int64: nat.DTYPE_I64, torch.float32: nat.DTYPE_F32, torch.float64: nat.DTYPE_F64}.get(dtype)


def _tensor_layout(dataArray):
    """(reversed axes, transposed?) of a CUDA tensor volume: a nibabel-style F-ordered one is used through its reversed-axes
    view, as _as_zyx does for ndarrays.  The other tensors of the call are viewed the same way."""
    nd = dataArray.dim()
    rev = tuple(range(nd - 1, -1, -1))
    return rev, nd > 1 and not dataArray.is_contiguous() and dataArray.permute(rev).is_contiguous()


def _tensor_data3(torch, dataArray, rev, transposed):
    """The intensities as a C-contiguous float64 (Z, Y, X) tensor: the caller's own when it already is one, otherwise converted
    once (processed as float64 whatever the input dtype, like the host path)."""
    d = dataArray.permute(rev) if transposed else dataArray
    if d.dtype != torch.float64:
        d = d.to(torch.float64)
    return d.contiguous().reshape((1,) * (3 - d.dim()) + tuple(d.shape))


def _tensor_work(t, rev, transposed):
    """(``t`` in (Z, Y, X) axis order, a C-contiguous tensor of it for the kernels): that view itself, or for other strides a
    copy that the caller writes back on success."""
    v = t.permute(rev) if transposed else t
    return v, (v if v.is_contiguous() else v.contiguous())


def _tensor_user_rows(torch, rows, shape, transposed):
    """(n, 3) int64 device rows in C order of (Z, Y, X) -> (n, ndim) rows in C order of the caller's axes (``shape``)."""
    nd = len(shape)
    r = rows[:, 3 - nd:]
    if not transposed:
        return r.contiguous()
    r = r.flip(1)
    key = r[:, 0].clone()
    for ax in range(1, nd):
        key = key * shape[ax] + r[:, ax]
    return r[torch.argsort(key)]


def _check_tensor(torch, name, t, like):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError("valueMap is a CUDA tensor: %s must be a CUDA tensor on the same device, got %s" % (name, type(t).__name__))
    if t.device != like.device:
        raise ValueError("%s (%s) and valueMap (%s) are on different devices" % (name, t.device, like.device))


def _tensor_run(dataArray, valueMap, H, maxSegmentSize):
    """The call on CUDA tensors: inputs attached where they are (the valueMap in its own dtype), labels written back by the
    kernels in that dtype, segmentedMap and the segmented rows built on the device.  Nothing of volume size crosses PCIe."""
    global LAST_RUN
    import torch
    _check_tensor(torch, "dataArray", dataArray, valueMap)
    if tuple(dataArray.shape) != tuple(valueMap.shape):
        raise ValueError("dataArray and valueMap must have the same shape")
    if LIST_ORDER:
        raise NotImplementedError("variationalRegionGrowing: LIST_ORDER = True (the strict engine) takes host arrays, not "
                                  "CUDA tensors")
    if DEVICES is not None:
        raise NotImplementedError("variationalRegionGrowing: DEVICES (z-slabs over several GPUs) takes host arrays, not CUDA "
                                  "tensors; set DEVICES = None to run on the tensors' device")
    nd = dataArray.dim()
    if nd > 3 or nd == 0:
        raise NotImplementedError("variationalRegionGrowing: 1-D to 3-D volumes only, got ndim=%d" % nd)
    code = _label_dtype_code(torch, valueMap.dtype)
    if code is None:
        raise TypeError("valueMap dtype %s: uint8, int8, int16, int32, int64, float32 or float64 only" % valueMap.dtype)
    if dataArray.is_complex():
        raise TypeError("dataArray must hold real intensities, got %s" % dataArray.dtype)
    clock = [time.perf_counter()]
    host_seconds = {}

    def lap(name):  # wall time per stage; stages that end in a synchronisation include the device work queued before them
        now = time.perf_counter()
        host_seconds[name] = host_seconds.get(name, 0.0) + now - clock[0]
        clock[0] = now
    dev = valueMap.device
    rev, transposed = _tensor_layout(dataArray)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev)
        d3 = _tensor_data3(torch, dataArray, rev, transposed)  # (Z, Y, X), C order
        vm_zyx, work = _tensor_work(valueMap, rev, transposed)
        vm3 = work.reshape(d3.shape)
        lap("prepare_inputs")

        def run(mode):
            with VRGEngine(d3.shape, H=H, max_segment_size=maxSegmentSize, iter_max=ITER_MAX, device=dev.index,
                           intensity=mode, max_seconds=MAX_SECONDS or 0.0) as eng:
                eng.set_stream(stream.cuda_stream)
                eng.attach_device_typed(d3.data_ptr(), vm3.data_ptr(), code)
                lap("create_handle")
                eng.init()
                res = eng.run()
                lap("levels_init_iterations")
                cap = res["n_in"]
                rows = torch.empty((cap, 3), dtype=torch.int64, device=dev)
                n = eng.segmented_device(rows.data_ptr() if cap else None, cap)
                if n > cap:  # not expected on one GPU (n_in is the count); once more with the right size
                    rows = torch.empty((n, 3), dtype=torch.int64, device=dev)
                    eng.segmented_device(rows.data_ptr(), n)
                rows = rows[:n]
                lap("segmented_rows")
                nonzero = eng.count_nonzero()  # np.count_nonzero(dataArray) of VRG:95
                lap("count_nonzero_on_device")
                seg3 = torch.empty(d3.shape, dtype=torch.int64, device=dev)
                eng.labels_device_typed(seg3.data_ptr(), nat.DTYPE_I64, segmented_only=True)
                # the caller's map is written last, once everything else has succeeded (VRG:137-228: in place)
                eng.labels_device_typed(vm3.data_ptr(), code)
                lap("labels_out")
            lap("destroy_handle")
            return res, rows, nonzero, seg3

        try:
            res, rows, nonzero, seg3 = run(INTENSITY)
        except nat.LevelsError:
            if d3.numel() > CONTINUOUS_MAX_VOXELS:  # same fallback as the host path
                raise
            res, rows, nonzero, seg3 = run("continuous")
        if work is not vm_zyx:
            vm_zyx.copy_(work)
        segmented = _tensor_user_rows(torch, rows, tuple(dataArray.shape), transposed)
        if transposed:
            segmentedMap = seg3.reshape(d3.shape[3 - nd:]).permute(rev).contiguous()
        else:
            segmentedMap = seg3.reshape(dataArray.shape)
        lap("user_layout")
    LAST_RUN = dict(res)
    LAST_RUN["host_seconds"] = host_seconds
    _finish_lines(res, segmented, None, nonzero)
    lap("print")
    return segmented, segmentedMap, valueMap


def variationalRegionGrowing(dataArray, valueMap, H=2.25, maxSegmentSize=5000):
    """B200 implementation of VRG:10-121.  See the module docstring for the contract."""
    global LAST_RUN
    torch = sys.modules.get("torch")  # a tensor can only come from an imported torch
    if torch is not None and isinstance(valueMap, torch.Tensor) and valueMap.is_cuda:
        out = _tensor_run(dataArray, valueMap, H, maxSegmentSize)
        _warn_order_dependence(LAST_RUN)
        return out
    if torch is not None and isinstance(dataArray, torch.Tensor) and dataArray.is_cuda:
        raise TypeError("dataArray is a CUDA tensor: valueMap must be a CUDA tensor on the same device too")
    dataArray = np.asarray(dataArray)
    if not isinstance(valueMap, np.ndarray):
        raise TypeError("valueMap must be an ndarray (it is updated in place, as in the reference)")
    if dataArray.shape != valueMap.shape:
        raise ValueError("dataArray and valueMap must have the same shape")
    if LIST_ORDER:
        return _list_order_run(dataArray, valueMap, H, maxSegmentSize)
    clock = [time.perf_counter()]
    host_seconds = {}

    def lap(name):  # where the wall time of a call goes: LAST_RUN["host_seconds"]
        now = time.perf_counter()
        host_seconds[name] = host_seconds.get(name, 0.0) + now - clock[0]
        clock[0] = now
    data3, transposed = _as_zyx(dataArray)
    vm_view = valueMap.T if transposed else valueMap
    vm3 = vm_view.reshape(data3.shape)
    vm8 = _labels_u8(vm3)
    lap("labels_to_uint8")
    direct = not transposed  # user arrays are C-ordered views of (Z, Y, X): results are written straight into them
    devices = _device_list()
    # The labels come back into the uint8 copy of the caller's map (or into the caller's map itself when that is uint8: it is
    # updated in place anyway, VRG:137-228): pages that are already mapped, not 0.5 GB of fresh ones.
    lab3 = vm8
    nonzero = [None]

    def run(mode):
        lap("allocate_outputs")
        with _Run(data3.shape, H, maxSegmentSize, mode, devices) as r:
            lap("create_handles")
            r.upload(data3, vm8)
            lap("upload")
            res = r.run()
            lap("levels_init_iterations")
            r.labels_into(lab3)
            lap("download_labels")
            seg = r.segmented(res["n_in"])
            lap("download_segmented_rows")
            nonzero[0] = r.count_nonzero()  # np.count_nonzero(dataArray) of VRG:95, counted where the volume already is
            lap("count_nonzero_on_device")
        lap("destroy_handles")
        return res, seg

    try:
        res, seg_zyx = run(INTENSITY)
    except nat.LevelsError:
        # more than 65536 distinct intensities: no level table.  Small volumes take the brute-force path, which is the
        # reference's own arithmetic (VRG:151-155, 232-255); large ones are as infeasible here as in the reference.
        if data3.size > CONTINUOUS_MAX_VOXELS:
            raise
        res, seg_zyx = run("continuous")
    LAST_RUN = dict(res)
    LAST_RUN["host_seconds"] = host_seconds
    # in place, VRG:137-228 (z-chunks on host threads: a uint8 -> int64 pass over the whole volume otherwise)
    if lab3 is vm3:
        pass  # the caller's own uint8 map was the download target
    elif direct and valueMap.flags.c_contiguous:
        out3 = valueMap.reshape(data3.shape)
        _pool_map(lambda zz: out3.__setitem__(slice(zz[0], zz[1]), lab3[zz[0]:zz[1]]), _chunks(data3.shape[0], HOST_THREADS))
    else:
        lab_user = lab3.reshape(vm_view.shape)
        valueMap[...] = lab_user.T if transposed else lab_user
    lap("value_map_in_place")
    segmented = seg_zyx[:, 3 - dataArray.ndim:]
    if transposed:
        segmented = segmented[:, ::-1]
        segmented = np.ascontiguousarray(segmented[np.lexsort(segmented.T[::-1])])  # C order of the user's axes
    # VRG:45-46 as the reference does it: a zero-filled int64 map with ones at the segmented voxels -- downloading the map as
    # int64 was 4 GB and a second of single-threaded page faults at C3
    segmentedMap = np.empty(dataArray.shape, dtype=np.int64)
    flat_map = segmentedMap.reshape(-1)
    n_all = flat_map.size  # zero-filled in parallel: first-touch page faults are what a fresh 4 GB array costs
    _pool_map(lambda ab: flat_map[ab[0]:ab[1]].fill(0), [(n_all * i // HOST_THREADS, n_all * (i + 1) // HOST_THREADS) for i in range(HOST_THREADS)])
    if len(segmented):
        flat = segmented[:, 0].copy()
        for ax in range(1, dataArray.ndim):
            flat *= dataArray.shape[ax]
            flat += segmented[:, ax]
        flat_map[flat] = 1
    lap("segmented_map_int64")
    _finish_lines(res, segmented, data3, nonzero[0])
    lap("print")
    _warn_order_dependence(res)
    return segmented, segmentedMap, valueMap


def _tensor_update(dataArray, segmented, segmentedMap, valueMap, H, flipedPoints, innerProb, outerProb):
    """update() on CUDA tensors: the state read from the caller's maps where they are, the flips, the band rows and the Parzen
    sum volumes on the device, on torch's current stream.  Nothing of volume size crosses PCIe."""
    import torch
    _check_tensor(torch, "dataArray", dataArray, valueMap)
    _check_tensor(torch, "segmentedMap", segmentedMap, valueMap)
    shape = tuple(dataArray.shape)
    if shape != tuple(valueMap.shape) or shape != tuple(segmentedMap.shape):
        raise ValueError("dataArray, segmentedMap and valueMap must have the same shape")
    new_prob = innerProb is None or outerProb is None
    if not new_prob:
        for name, t in (("innerProb", innerProb), ("outerProb", outerProb)):
            _check_tensor(torch, name, t, valueMap)
            if t.dtype != torch.float64:
                raise TypeError("%s must be a float64 CUDA tensor, got %s" % (name, t.dtype))
            if tuple(t.shape) != shape:
                raise ValueError("%s must have the shape of dataArray" % name)
    nd = dataArray.dim()
    if nd > 3 or nd == 0:
        raise NotImplementedError("update: 1-D to 3-D volumes only, got ndim=%d" % nd)
    seg_code, vm_code = _label_dtype_code(torch, segmentedMap.dtype), _label_dtype_code(torch, valueMap.dtype)
    if seg_code is None or vm_code is None:
        raise TypeError("segmentedMap / valueMap dtype %s / %s: uint8, int8, int16, int32, int64, float32 or float64 only"
                        % (segmentedMap.dtype, valueMap.dtype))
    if dataArray.is_complex():
        raise TypeError("dataArray must hold real intensities, got %s" % dataArray.dtype)
    dev = valueMap.device
    rev, transposed = _tensor_layout(dataArray)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev)
        d3 = _tensor_data3(torch, dataArray, rev, transposed)
        shape3 = tuple(d3.shape)
        pairs = [_tensor_work(segmentedMap, rev, transposed), _tensor_work(valueMap, rev, transposed)]
        seg_w, vm_w = pairs[0][1], pairs[1][1]
        if flipedPoints is not None:
            if isinstance(flipedPoints, torch.Tensor) and flipedPoints.is_cuda:
                if flipedPoints.dtype.is_floating_point or flipedPoints.dtype.is_complex or flipedPoints.dtype == torch.bool:
                    raise TypeError("flipedPoints must hold integer coordinates, got %s" % flipedPoints.dtype)
                if flipedPoints.device != dev:
                    raise ValueError("flipedPoints (%s) and valueMap (%s) are on different devices" % (flipedPoints.device, dev))
                pts = flipedPoints.reshape(-1, nd).to(torch.int64)
            else:  # a host list of points is small: copied to the device once
                pts = torch.from_numpy(np.asarray(flipedPoints, dtype=np.int64).reshape(-1, nd)).to(dev)
            if transposed:
                pts = pts.flip(1)
            flips = torch.cat([pts.new_zeros((pts.shape[0], 3 - nd)), pts], dim=1).contiguous()  # (z, y, x) rows
        with VRGEngine(shape3, H=H, max_segment_size=2 ** 62, iter_max=ITER_MAX, device=dev.index, intensity="f64_band") as eng:
            eng.set_stream(stream.cuda_stream)
            eng.attach_state_typed(d3.data_ptr(), seg_w.data_ptr(), seg_code, vm_w.data_ptr(), vm_code)
            eng.init()
            if flipedPoints is None:
                eng.enqueue_table()
                res = eng.poll()
            else:  # rows outside the volume raise here, before anything of the caller's is written
                res = eng.apply_flips_device(flips.data_ptr() if len(flips) else None, len(flips))

            def rows(which, cap):
                out = torch.empty((cap, 3), dtype=torch.int64, device=dev)
                n = eng.band_rows_device(which, out.data_ptr() if cap else None, cap)
                if n > cap:
                    out = torch.empty((n, 3), dtype=torch.int64, device=dev)
                    eng.band_rows_device(which, out.data_ptr(), n)
                return _tensor_user_rows(torch, out[:n], shape, transposed)
            innerBnd = rows(1, res["n_in"])  # the inner band is part of the segmented set
            outerBnd = rows(2, 0)  # counted first
            segmentedOut = segmented if flipedPoints is None else rows(0, res["n_in"])
            if new_prob:  # VRG:132-133
                pin3 = torch.empty(shape3, dtype=torch.float64, device=dev)
                pout3 = torch.empty(shape3, dtype=torch.float64, device=dev)
            else:
                pairs += [_tensor_work(innerProb, rev, transposed), _tensor_work(outerProb, rev, transposed)]
                pin3, pout3 = pairs[2][1], pairs[3][1]
            eng.band_sums_device(pin3.data_ptr(), pout3.data_ptr())
            eng.labels_device_typed(seg_w.data_ptr(), seg_code, segmented_only=True)
            eng.labels_device_typed(vm_w.data_ptr(), vm_code)
        for view, work in pairs:
            if work is not view:
                view.copy_(work)
        if new_prob:
            zyx_shape = shape3[3 - nd:]
            innerProb, outerProb = ((t.reshape(zyx_shape).permute(rev).contiguous() if transposed else t.reshape(shape))
                                    for t in (pin3, pout3))
    return segmentedOut, segmentedMap, valueMap, innerBnd, outerBnd, innerProb, outerProb


def update(dataArray, segmented, segmentedMap, valueMap, H, flipedPoints=None, innerBnd=None, outerBnd=None,
           innerProb=None, outerProb=None):
    """One call of the reference's ``update`` (VRG:124-261) on the GPU: the init branch (``flipedPoints is None``,
    VRG:129-155) or one application of the band state machine to the caller's flip list (VRG:156-259).

    The state is ``segmentedMap`` (1 = segmented) and the excluded voxels of ``valueMap`` (label 4); the band lists and
    the Parzen sums are functions of that state, so ``innerBnd`` / ``outerBnd`` / ``innerProb`` / ``outerProb`` are
    accepted for signature compatibility and rebuilt: ``innerBnd = argwhere(valueMap == 1)``, ``outerBnd =
    argwhere(valueMap == 2)`` (C order; the reference's row order is its append history) and ``innerProb[p]`` /
    ``outerProb[p]`` = the unnormalised sums of VRG:154-155 at every band voxel, 0 elsewhere (within 1e-12 relative of the
    reference's where its incremental sums have not drifted).  ``valueMap`` and ``segmentedMap`` are updated in place
    and returned as the same objects, like the reference does; listed voxels that are in neither band are ignored.
    Level-table data only (at most 65536 distinct intensities), one GPU (``DEVICE``).

    CUDA tensors: when ``valueMap`` is a CUDA tensor the call runs on its device and torch's current stream, and nothing of
    volume size crosses PCIe.  ``dataArray`` and ``segmentedMap`` must be CUDA tensors on that device (mixing host arrays and
    tensors raises ``TypeError``); intensities of any real dtype are converted to float64 once, the two maps are read in
    their own dtypes (uint8, int8, int16, int32, int64, float32, float64): ``segmentedMap == 1`` is segmented, ``valueMap ==
    4`` excluded.  ``flipedPoints`` may be a CUDA integer tensor ``(F, ndim)`` or anything ``np.asarray`` takes (copied to the
    device once); a point outside the volume raises ``ValueError`` before anything is modified.  ``valueMap`` and
    ``segmentedMap`` are updated in place in their dtypes; ``innerBnd`` / ``outerBnd`` come back as int64 CUDA tensors
    ``(n, ndim)`` in C order of the caller's axes, ``segmented`` too (the caller's object on the init branch);
    ``innerProb`` / ``outerProb`` must then be float64 CUDA tensors (``TypeError`` otherwise) and are updated in place, or
    are returned as new C-contiguous ones when either is None.  Layouts as in ``variationalRegionGrowing``; on any error
    the four caller tensors are bit-unchanged.  Results are bit-identical to the call on host arrays.
    """
    torch = sys.modules.get("torch")  # a tensor can only come from an imported torch
    if torch is not None and isinstance(valueMap, torch.Tensor) and valueMap.is_cuda:
        return _tensor_update(dataArray, segmented, segmentedMap, valueMap, H, flipedPoints, innerProb, outerProb)
    if torch is not None and any(isinstance(a, torch.Tensor) and a.is_cuda for a in (dataArray, segmentedMap, innerProb, outerProb)):
        raise TypeError("update: valueMap is not a CUDA tensor, so dataArray, segmentedMap, innerProb and outerProb may not be")
    dataArray = np.asarray(dataArray)
    if not isinstance(valueMap, np.ndarray) or not isinstance(segmentedMap, np.ndarray):
        raise TypeError("valueMap and segmentedMap must be ndarrays (they are updated in place, as in the reference)")
    if dataArray.shape != valueMap.shape or dataArray.shape != segmentedMap.shape:
        raise ValueError("dataArray, segmentedMap and valueMap must have the same shape")
    data3, transposed = _as_zyx(dataArray)
    nd = dataArray.ndim

    def zyx(a):
        return (a.T if transposed else a).reshape(data3.shape)
    seg_in, vm_in = zyx(segmentedMap), zyx(valueMap)
    vm8 = np.full(data3.shape, 3, dtype=np.uint8)
    vm8[vm_in == 4] = 4
    vm8[seg_in == 1] = 0

    def to_zyx_rows(pts):
        pts = np.asarray(pts, dtype=np.int64).reshape(-1, nd)
        if transposed:
            pts = pts[:, ::-1]
        return np.concatenate([np.zeros((len(pts), 3 - nd), dtype=np.int64), pts], axis=1)

    def to_user_rows(rows):
        rows = rows[:, 3 - nd:]
        if transposed:
            rows = rows[:, ::-1]
            rows = rows[np.lexsort(rows.T[::-1])]  # C order of the user's axes
        return np.ascontiguousarray(rows)

    with VRGEngine(data3.shape, H=H, max_segment_size=2 ** 62, iter_max=ITER_MAX, device=DEVICE, intensity="f64_band") as eng:
        eng.upload(np.ascontiguousarray(data3, dtype=np.float64), vm8)
        eng.init()
        if flipedPoints is None:
            eng.enqueue_table()
            res = eng.poll()
        else:
            res = eng.apply_flips(to_zyx_rows(flipedPoints))
        labels = eng.labels()
        seg_rows = eng.segmented()
        lv, pin, pout = eng.table()
    zyx(valueMap)[...] = labels
    zyx(segmentedMap)[...] = labels <= 1
    inner = labels == 1
    outer = labels == 2
    new_prob = innerProb is None or outerProb is None
    if new_prob:
        innerProb = np.zeros(dataArray.shape)  # VRG:132-133
        outerProb = np.zeros(dataArray.shape)
    else:
        innerProb[...] = 0
        outerProb[...] = 0
    band = inner | outer
    idx = np.searchsorted(lv, np.asarray(data3, dtype=np.float64)[band])
    ip, op = zyx(innerProb), zyx(outerProb)
    ip[band] = pin[idx] * res["n_in"]    # the table holds the normalised sums (VRG:81-82)
    op[band] = pout[idx] * res["n_out"]
    innerBndOut = to_user_rows(np.argwhere(inner))
    outerBndOut = to_user_rows(np.argwhere(outer))
    segmentedOut = segmented if flipedPoints is None else to_user_rows(seg_rows)
    return segmentedOut, segmentedMap, valueMap, innerBndOut, outerBndOut, innerProb, outerProb


def get_neighbours(p, exclude_p=True, shape=None):
    """In-bounds 3^ndim neighbourhood of ``p`` in lexicographic order, last axis fastest (VRG:263-282)."""
    p = np.asarray(p)
    offsets = np.array(list(itertools.product((-1, 0, 1), repeat=len(p))), dtype=np.int64)
    if exclude_p:
        offsets = offsets[np.any(offsets != 0, axis=1)]
    neighbours = p + offsets
    if shape is not None:
        ok = np.all((neighbours >= 0) & (neighbours < np.asarray(shape)), axis=1)
        neighbours = neighbours[ok]
    return neighbours


def _verdict(name, volume, segmented):
    inside = bool(np.all(volume[tuple(segmented.T)]))
    complete = bool(np.count_nonzero(volume) == len(segmented))
    if inside and complete:
        print('{} test passed!'.format(name))
    elif inside:
        print('{} test partially failed: Segmented volume not complete!'.format(name))
    elif complete:
        print('{} test partially failed: Wrong segments included!'.format(name))
    else:
        print('{} test failed!'.format(name))
    return bool(inside and complete)


def test_StraightLine():
    """The reference's first self-test (VRG:284-298): a 2x2x20 bar in a 50x50x150 volume, seeded by 2x2x3 voxels of it."""
    volume = np.zeros((50, 50, 150), dtype=int)
    volume[20:22, 20:22, 20:40] = 1
    valueMap = np.full(volume.shape, 3)
    valueMap[20:22, 20:22, 22:25] = 0
    segmented, segmentedMap, valueMap = variationalRegionGrowing(volume, valueMap)
    return _verdict('Straight line', volume, segmented)


def test_Sphere():
    """The reference's second self-test (VRG:300-314): a ball of radius 10 in a 50^3 volume, seeded by its central 2^3."""
    x, y, z = np.mgrid[:50, :50, :50]
    volume = ((x - 25) ** 2 + (y - 25) ** 2 + (z - 25) ** 2 <= 100).astype(int)
    print(np.count_nonzero(volume))
    valueMap = np.full(volume.shape, 3)
    valueMap[25:27, 25:27, 25:27] = 0
    segmented, segmentMap, valueMap = variationalRegionGrowing(volume, valueMap)
    return _verdict('Sphere', volume, segmented)
