"""GPU drop-ins for the array operations of the reference's ``Code/generateVesselVolume.py`` (GVV:line) and for the
distance transform ``Code/manualCorrectionGUI.py:248`` runs on the VRG output -- SURVEY.md section 8(f), rows N2 / N3.

Same names, arguments and return conventions as the reference where it has a function (``labelVolume``,
``maskVolume``); the threshold / component-filter rule that the reference writes inline in ``main()`` (GVV:183-200) is
``vesselnessToVesselMask``; ``distance_transform_edt`` stands in for the SciPy call of the same name, with SciPy's
signature (``sampling``, ``return_indices``, in-place outputs) for 3-D volumes.  NIfTI I/O (``loadVolume`` / ``saveVolume``) is out of scope: nibabel is the reference's storage layer.

Everything runs through the C-ABI of ``include/vrg_b200.h`` on the GPU; there is no CPU fallback.  NumPy arrays are
copied to the device and back; CUDA tensors stay where they are (``*_device`` entry points, on the tensor's device and
torch's current stream) and the results come back as CUDA tensors on that device -- vesselness, mask, seeds,
``variationalRegionGrowing`` and the distance transform can run without the volume ever leaving the GPU.
"""
from __future__ import annotations

import ctypes
import sys

import numpy as np

from . import _native as nat

__all__ = ["distance_transform_edt", "labelVolume", "maskVolume", "vesselnessToVesselMask"]


def _shape3(a):
    if a.ndim != 3:
        raise ValueError("3-D volumes only, got shape %r" % (a.shape,))
    return (nat.i64 * 3)(*a.shape)


def _isotropic_view(a, dtype):
    """C-contiguous (Z, Y, X) array for an operation that does not care about axis order: an F-ordered volume (what
    nibabel hands out, GVV:35) is used through its transpose instead of being copied.  Returns (array, transposed)."""
    a = np.asarray(a)
    if a.ndim == 3 and a.flags.f_contiguous and not a.flags.c_contiguous:
        return np.ascontiguousarray(a.T, dtype=dtype), True
    return np.ascontiguousarray(a, dtype=dtype), False


def _cuda_torch(*arrays):
    """torch when the arguments are CUDA tensors (all of them, on one device), None when none is; a mix is an error."""
    torch = sys.modules.get("torch")  # a tensor can only come from an imported torch
    if torch is None:
        return None
    cuda = [isinstance(a, torch.Tensor) and a.is_cuda for a in arrays]
    if not any(cuda):
        return None
    if not all(cuda) or len({a.device for a in arrays}) != 1:
        raise TypeError("pass either host arrays or CUDA tensors on one device, not a mix")
    return torch


def _tensor_view(torch, t, dtype):
    """``_isotropic_view`` for a CUDA tensor: an F-ordered volume is used through its reversed-axes view."""
    if t.dim() != 3:
        raise ValueError("3-D volumes only, got shape %r" % (tuple(t.shape),))
    transposed = not t.is_contiguous() and t.permute(2, 1, 0).is_contiguous()
    if transposed:
        t = t.permute(2, 1, 0)
    return t.to(dtype).contiguous(), transposed


def _stream(torch, t):
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream or None)


def distance_transform_edt(input, sampling=None, return_distances=True, return_indices=False, distances=None, indices=None,
                           device: int = 0):
    """``scipy.ndimage.distance_transform_edt`` (GVV:183, manualCorrectionGUI.py:248) for 3-D volumes: float64 Euclidean
    distance of every non-zero voxel to the nearest zero voxel and, with ``return_indices``, the feature transform: int32
    ``(3, Z, Y, X)`` coordinates of that zero voxel.

    Arguments, return values (``dt``, ``ft``, a tuple of both, or ``None`` when every requested output was written in
    place into ``distances`` / ``indices``) and argument errors are SciPy's, and so is every output value, ties between
    equally near zero voxels and the rounding of anisotropic ``sampling`` (a scalar or one spacing per axis, positive and
    finite) included.  A CUDA tensor in gives CUDA tensors out (on its device and torch's current stream; ``device`` is
    then not used), and ``distances`` / ``indices`` may then be CUDA tensors on that device.  The call with default
    arguments runs the plain distance transform; any other runs SciPy's feature transform on the caller's axes."""
    if sampling is not None or not return_distances or return_indices or distances is not None or indices is not None:
        return _edt_ft(input, sampling, return_distances, return_indices, distances, indices, device)
    torch = _cuda_torch(input)
    if torch is not None:
        m, transposed = _tensor_view(torch, input != 0, torch.uint8)
        out = torch.empty(m.shape, dtype=torch.float64, device=m.device)
        shp = (nat.i64 * 3)(*m.shape)
        with torch.cuda.device(m.device):
            nat.check(nat.load().vrg_edt_device(m.device.index, m.data_ptr(), ctypes.addressof(shp), out.data_ptr(),
                                                _stream(torch, m)))
        return out.permute(2, 1, 0) if transposed else out
    m, transposed = _isotropic_view(np.asarray(input) != 0, np.uint8)
    out = np.empty(m.shape, dtype=np.float64)
    shp = _shape3(m)  # kept alive across the call
    nat.check(nat.load().vrg_edt(device, m.ctypes.data, ctypes.addressof(shp), out.ctypes.data))
    return out.T if transposed else out


def _sampling3(sampling):
    """SciPy's normalisation of ``sampling`` (a scalar for every axis, or one value per axis) as 3 C doubles, or None."""
    if sampling is None:
        return None
    if not isinstance(sampling, str) and np.iterable(sampling):
        s = list(sampling)
        if len(s) != 3:
            raise RuntimeError("sequence argument must have length equal to input rank")
    else:
        s = [sampling] * 3
    s = np.asarray(s, dtype=np.float64)
    if not (np.isfinite(s).all() and (s > 0).all()):
        raise ValueError("distance_transform_edt: sampling must be positive and finite, got %r" % (s.tolist(),))
    return (ctypes.c_double * 3)(*s)


def _edt_ft(input, sampling, return_distances, return_indices, distances, indices, device):
    """distance_transform_edt through SciPy's feature transform (``vrg_edt_ft`` / ``vrg_edt_ft_device``).  The input is
    taken in C order on the caller's axes: a transposed view would run the passes in the other order and break ties
    differently from SciPy."""
    torch = _cuda_torch(input)
    out_type = torch.Tensor if torch is not None else np.ndarray  # SciPy writes in place into arrays only
    dt_inplace, ft_inplace = isinstance(distances, out_type), isinstance(indices, out_type)
    errors = []  # SciPy's _distance_transform_arg_check
    if not return_distances and not return_indices:
        errors.append("at least one of return_distances/return_indices must be True")
    if dt_inplace and not return_distances:
        errors.append("return_distances must be True if distances is supplied")
    if ft_inplace and not return_indices:
        errors.append("return_indices must be True if indices is supplied")
    if errors:
        raise RuntimeError(", ".join(errors))
    if torch is not None:
        if input.dim() != 3:
            raise ValueError("3-D volumes only, got shape %r" % (tuple(input.shape),))
        shape = tuple(input.shape)
        f64, i32 = torch.float64, torch.int32
    else:
        input = np.asarray(input)
        if input.ndim != 3:
            raise ValueError("3-D volumes only, got shape %r" % (input.shape,))
        shape = input.shape
        f64, i32 = np.float64, np.int32
    s = _sampling3(sampling)
    for out, inplace, want_shape, want_dtype, name, dtname in (
            (indices, ft_inplace, (3,) + shape, i32, "indices", "int32"),
            (distances, dt_inplace, shape, f64, "distances", "float64")):
        if not inplace:
            continue
        if tuple(out.shape) != want_shape:
            raise RuntimeError("%s array has wrong shape" % name)
        if out.dtype != want_dtype:
            raise RuntimeError("%s array must be %s" % (name, dtname))
        if torch is not None and out.device != input.device:
            raise RuntimeError("%s must be on %s, the input's device" % (name, input.device))
    lib = nat.load()
    shp = (nat.i64 * 3)(*shape)  # kept alive across the call
    m = (input != 0).to(torch.uint8).contiguous() if torch is not None else np.ascontiguousarray(input != 0, dtype=np.uint8)

    def target(out, inplace, sh, dtype):
        """where the kernel writes an output: the caller's array when it is C-contiguous, else a new one (copied over)"""
        if torch is not None:
            return out if inplace and out.is_contiguous() else torch.empty(sh, dtype=dtype, device=m.device)
        return out if inplace and out.flags.c_contiguous and out.flags.writeable else np.empty(sh, dtype=dtype)

    dt = target(distances, dt_inplace, shape, f64) if return_distances else None
    ft = target(indices, ft_inplace, (3,) + shape, i32) if return_indices else None
    sp = None if s is None else ctypes.addressof(s)
    if torch is not None:
        with torch.cuda.device(m.device):
            nat.check(lib.vrg_edt_ft_device(m.device.index, m.data_ptr(), ctypes.addressof(shp), sp,
                                            None if dt is None else dt.data_ptr(), None if ft is None else ft.data_ptr(),
                                            _stream(torch, m)))
    else:
        nat.check(lib.vrg_edt_ft(device, m.ctypes.data, ctypes.addressof(shp), sp,
                                 None if dt is None else dt.ctypes.data, None if ft is None else ft.ctypes.data))
    result = []
    if return_distances:
        if dt_inplace:
            if dt is not distances:
                distances[...] = dt
        else:
            result.append(dt)
    if return_indices:
        if ft_inplace:
            if ft is not indices:
                indices[...] = ft
        else:
            result.append(ft)
    if len(result) == 2:
        return tuple(result)
    return result[0] if result else None


def labelVolume(volume, minSize=1, maxHop=3, device: int = 0):
    """GVV:108-136: 26-connected components (``skimage.measure.label(volume, return_num=True, connectivity=maxHop)``).

    Exact for binary volumes (background 0, one foreground value), which is what the reference passes; a volume with several
    distinct non-zero values raises ``ValueError`` (skimage would label per value).

    Returns ``(labeled, labelResult)``: ``labeled`` holds 0 on the background and 1..K on the components, numbered in
    raster order of their first voxel; ``labelResult`` is ``[(label, size), ...]`` over every label present, the
    background entry ``(0, n0)`` included, exactly as the reference builds it from ``np.bincount`` (``minSize`` is
    accepted and, as in the reference, not applied: its filter is commented out at GVV:132).
    """
    if maxHop != 3:
        raise ValueError("labelVolume: only maxHop=3 (26-connectivity), the value the reference uses (GVV:196)")
    torch = _cuda_torch(volume)
    if torch is not None:
        return _label_tensor(torch, volume)
    vol = np.asarray(volume)
    nz = vol != 0
    # skimage.measure.label joins neighbours of EQUAL value: two touching regions with different non-zero values get different
    # labels there.  This drop-in labels the non-zero mask, which is the same thing only for two-valued volumes -- all the
    # reference ever passes (GVV:195 binarises first; skeletonization.py:108 passes a 0/1 mask).  Anything else is refused.
    if nz.any():
        vals = vol[nz]
        if vals.min() != vals.max():
            raise ValueError("labelVolume: the volume holds more than one non-zero value; skimage.measure.label would split "
                             "touching regions of different value, this drop-in is exact for binary (0 / v) volumes only")
    b = np.ascontiguousarray(nz, dtype=np.uint8)
    n = ctypes.c_int64(0)
    labeled = np.empty(b.shape, dtype=np.int32)
    sizes = np.zeros(max(1, b.size // 2 + 1), dtype=np.int64) if b.size < (1 << 22) else None
    lib = nat.load()
    shp = _shape3(b)  # kept alive across the calls
    if sizes is not None:
        nat.check(lib.vrg_label_components(device, b.ctypes.data, ctypes.addressof(shp), labeled.ctypes.data,
                                           ctypes.byref(n), sizes.ctypes.data, sizes.size))
        sizes = sizes[: n.value]
    else:  # component count unknown in advance: ask twice rather than reserve a voxel-sized buffer
        nat.check(lib.vrg_label_components(device, b.ctypes.data, ctypes.addressof(shp), labeled.ctypes.data,
                                           ctypes.byref(n), None, 0))
        sizes = np.bincount(labeled.ravel(), minlength=n.value + 1)[1:].astype(np.int64)
    n_bg = int(b.size - sizes.sum())
    result = ([(0, n_bg)] if n_bg else []) + [(k + 1, int(s)) for k, s in enumerate(sizes)]
    return labeled, result


def _label_tensor(torch, vol):
    """labelVolume on a CUDA tensor: int32 labels stay on the device, ``labelResult`` is the same host list."""
    if vol.dim() != 3:
        raise ValueError("3-D volumes only, got shape %r" % (tuple(vol.shape),))
    nz = vol != 0
    vals = vol[nz]
    if vals.numel() and bool(vals.min() != vals.max()):
        raise ValueError("labelVolume: the volume holds more than one non-zero value; skimage.measure.label would split "
                         "touching regions of different value, this drop-in is exact for binary (0 / v) volumes only")
    b = nz.to(torch.uint8).contiguous()  # raster order of the caller's axes, as on the host path
    n = ctypes.c_int64(0)
    labeled = torch.empty(b.shape, dtype=torch.int32, device=b.device)
    sizes = np.zeros(max(1, b.numel() // 2 + 1), dtype=np.int64) if b.numel() < (1 << 22) else None
    shp = (nat.i64 * 3)(*b.shape)
    with torch.cuda.device(b.device):
        nat.check(nat.load().vrg_label_components_device(
            b.device.index, b.data_ptr(), ctypes.addressof(shp), labeled.data_ptr(), ctypes.byref(n),
            sizes.ctypes.data if sizes is not None else None, sizes.size if sizes is not None else 0, _stream(torch, b)))
    if sizes is not None:
        sizes = sizes[: n.value]
    else:
        sizes = torch.bincount(labeled.flatten().to(torch.int64), minlength=n.value + 1)[1:].cpu().numpy()
    n_bg = int(b.numel() - sizes.sum())
    result = ([(0, n_bg)] if n_bg else []) + [(k + 1, int(s)) for k, s in enumerate(sizes)]
    return labeled, result


def maskVolume(volume, mask):
    """GVV:86-106: copy of ``volume`` with the voxels outside ``mask`` set to 0 (elementwise; CUDA tensors stay on their
    device)."""
    if _cuda_torch(volume, mask) is not None:
        new = volume.clone()
        new[mask == 0] = 0
        return new
    new = np.array(volume, copy=True)
    new[np.asarray(mask) == 0] = 0
    return new


def vesselnessToVesselMask(vesselnessVolume, brainVolumeMask, edgeDistance=10, edgeFraction=0.8, fraction=0.7,
                           minComponentSize=150, device: int = 0, return_info: bool = False):
    """The body of the reference's ``main()`` between loading and saving, GVV:183-200 + 216:

    * voxels within ``edgeDistance`` of the brain-mask boundary (EDT of ``brainVolumeMask``) whose vesselness is
      ``<= min + edgeFraction * (max - min)`` are zeroed, then all voxels ``<= min + fraction * (max - min)``;
    * the rest is binarised, labelled with 26-connectivity, and components of at most ``minComponentSize`` voxels
      are removed.

    Returns the uint8 vessel mask (what GVV:216 saves as ``vesselVolumeMask.nii.gz``); prints the reference's
    ``'Number of voxels in segmentation: N'`` line (GVV:211).  CUDA tensors in (both), a CUDA tensor out.
    """
    torch = _cuda_torch(vesselnessVolume, brainVolumeMask)
    if torch is not None:
        v, transposed = _tensor_view(torch, vesselnessVolume, torch.float64)
        b, tb = _tensor_view(torch, brainVolumeMask != 0, torch.uint8)
        if tb != transposed:
            b = b.permute(2, 1, 0).contiguous()
        if v.shape != b.shape:
            raise ValueError("vesselness %r and brain mask %r differ in shape" % (tuple(v.shape), tuple(b.shape)))
        out = torch.empty(v.shape, dtype=torch.uint8, device=v.device)
    else:
        v, transposed = _isotropic_view(vesselnessVolume, np.float64)
        b, tb = _isotropic_view(np.asarray(brainVolumeMask) != 0, np.uint8)
        if tb != transposed:
            b = np.ascontiguousarray(b.T)
        if v.shape != b.shape:
            raise ValueError("vesselness %r and brain mask %r differ in shape" % (v.shape, b.shape))
        out = np.empty(v.shape, dtype=np.uint8)
    info = (nat.i64 * 2)()
    thr = (ctypes.c_double * 2)()
    shp = _shape3(v) if torch is None else (nat.i64 * 3)(*v.shape)  # kept alive across the call
    if torch is not None:
        with torch.cuda.device(v.device):
            nat.check(nat.load().vrg_vessel_mask_device(v.device.index, v.data_ptr(), b.data_ptr(), ctypes.addressof(shp),
                                                        float(edgeDistance), float(edgeFraction), float(fraction),
                                                        int(minComponentSize), out.data_ptr(), ctypes.addressof(info),
                                                        ctypes.addressof(thr), _stream(torch, v)))
    else:
        nat.check(nat.load().vrg_vessel_mask(device, v.ctypes.data, b.ctypes.data, ctypes.addressof(shp),
                                             float(edgeDistance), float(edgeFraction), float(fraction),
                                             int(minComponentSize), out.ctypes.data, ctypes.addressof(info),
                                             ctypes.addressof(thr)))
    print('Number of voxels in segmentation: {}'.format(int(info[0])))
    out = (out.permute(2, 1, 0) if torch is not None else out.T) if transposed else out
    if return_info:
        return out, {"voxels": int(info[0]), "components": int(info[1]), "thresholds": (thr[0], thr[1])}
    return out

