"""Host-side handle around the C-ABI (include/vrg_b200.h): one z-slab of the volume on one GPU.

This is plumbing only -- every compute step is a kernel launch inside
``libvrg_b200.so``.  ``VRGEngine`` mirrors the phases of the reference
function (Code/variationalRegionGrowing.py): upload (VRG:40-46), init branch of
``update`` (VRG:129-155), the iteration loop (VRG:58-117) and the outputs (VRG:96).
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _native as nat


class VRGEngine:
    def __init__(self, shape, H=2.25, max_segment_size=5000, iter_max=200, device=0,
                 intensity="f64_band", z_begin=0, z_end=None, max_seconds=0.0):
        self.lib = nat.load()
        shape = tuple(int(s) for s in shape)
        if len(shape) != 3:
            raise ValueError("VRGEngine needs a 3-D shape (Z, Y, X)")
        self.shape = shape
        self.z_begin = int(z_begin)
        self.z_end = shape[0] if z_end is None else int(z_end)
        self.ext_lo = max(0, self.z_begin - nat.HALO)
        self.ext_hi = min(shape[0], self.z_end + nat.HALO)
        cfg = nat.Config()
        cfg.shape[:] = shape
        cfg.z_begin, cfg.z_end = self.z_begin, self.z_end
        cfg.device = int(device)
        cfg.intensity_mode = nat.INTENSITY_MODES[intensity] if isinstance(intensity, str) else int(intensity)
        cfg.H = float(H)
        cfg.iter_max = int(iter_max)
        cfg.max_segment_size = int(min(max_segment_size, 2 ** 62))
        cfg.max_seconds = float(max_seconds or 0.0)
        self.cfg = cfg
        self.device = int(device)
        self._h = nat.vp()
        nat.check(self.lib.vrg_create(ctypes.byref(cfg), ctypes.byref(self._h)))

    # -- lifetime -------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.vrg_destroy(self._h)
            self._h = nat.vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_stream(self, cuda_stream: int):
        nat.check(self.lib.vrg_set_stream(self._h, nat.vp(cuda_stream)))

    # -- inputs ---------------------------------------------------------------------------
    @property
    def own_planes(self):
        return self.z_end - self.z_begin

    def _ext(self, a, dtype):
        a = np.ascontiguousarray(a, dtype=dtype)
        n_ext = self.ext_hi - self.ext_lo
        if a.shape == self.shape:
            a = a[self.ext_lo:self.ext_hi]
        if a.shape != (n_ext,) + self.shape[1:]:
            raise ValueError("expected the whole volume %s or the extended slab (%d planes), got %s"
                             % (self.shape, n_ext, a.shape))
        return np.ascontiguousarray(a)

    def upload(self, data, value_map):
        d = self._ext(data, np.float64)
        v = self._ext(value_map, np.uint8)
        nat.check(self.lib.vrg_upload(self._h, d.ctypes.data, v.ctypes.data))

    def upload_value_map(self, value_map):
        v = self._ext(value_map, np.uint8)
        nat.check(self.lib.vrg_upload_value_map(self._h, v.ctypes.data))

    def upload_device(self, data_ptr: int, value_map_ptr: int):
        nat.check(self.lib.vrg_upload_device(self._h, nat.vp(data_ptr or None), nat.vp(value_map_ptr or None)))

    def attach_device(self, data_ptr: int, value_map_ptr: int):
        """Zero-copy: run on the caller's device-resident extended slab (fp64 data, uint8 valueMap)."""
        nat.check(self.lib.vrg_attach_device(self._h, nat.vp(data_ptr), nat.vp(value_map_ptr)))

    def attach_device_typed(self, data_ptr: int, value_map_ptr: int, value_map_dtype: int):
        """Zero-copy like ``attach_device``, the valueMap in its own dtype (``nat.DTYPE_*``): vrg_init reads it as it is."""
        nat.check(self.lib.vrg_attach_device_typed(self._h, nat.vp(data_ptr), nat.vp(value_map_ptr), int(value_map_dtype)))

    def attach_state_typed(self, data_ptr: int, seg_map_ptr: int, seg_map_dtype: int, value_map_ptr: int, value_map_dtype: int):
        """update()'s inputs on the device: fp64 data attached zero-copy, the state built from segmentedMap (== 1) and valueMap
        (== 4), each in its own dtype (``nat.DTYPE_*``), into the handle's own map on its stream."""
        nat.check(self.lib.vrg_attach_state_typed(self._h, nat.vp(data_ptr), nat.vp(seg_map_ptr), int(seg_map_dtype),
                                                  nat.vp(value_map_ptr), int(value_map_dtype)))

    # -- levels -----------------------------------------------------------------------------
    def scan_levels(self) -> np.ndarray:
        n = nat.i64(0)
        nat.check(self.lib.vrg_scan_levels(self._h, ctypes.byref(n)))
        out = np.empty(n.value, dtype=np.float64)
        nat.check(self.lib.vrg_get_levels(self._h, out.ctypes.data, out.size))
        return out

    def set_levels(self, levels):
        lv = np.ascontiguousarray(levels, dtype=np.float64)
        nat.check(self.lib.vrg_set_levels(self._h, lv.ctypes.data, lv.size))

    # -- run --------------------------------------------------------------------------------
    def init(self):
        nat.check(self.lib.vrg_init(self._h))

    def run(self) -> dict:
        r = nat.Result()
        nat.check(self.lib.vrg_run(self._h, ctypes.byref(r)))
        return self._res(r)

    def poll(self) -> dict:
        r = nat.Result()
        nat.check(self.lib.vrg_poll(self._h, ctypes.byref(r)))
        return self._res(r)

    def _res(self, r):
        out = {k: int(getattr(r, k)) for k, _ in nat.Result._fields_}
        n = nat.i64(0)
        nat.check(self.lib.vrg_dense_refresh_sweeps(self._h, ctypes.byref(n)))
        out["dense_refresh_sweeps"] = int(n.value)  # f64_dense: sweeps that read the intensities (the rest read the kept bits)
        return out

    def enqueue_decide(self):
        nat.check(self.lib.vrg_enqueue_decide(self._h))

    def enqueue_cancel(self):
        nat.check(self.lib.vrg_enqueue_cancel(self._h))

    def enqueue_absorb(self):
        nat.check(self.lib.vrg_enqueue_absorb(self._h))

    def enqueue_flip(self):
        nat.check(self.lib.vrg_enqueue_flip(self._h))

    def enqueue_advance(self):
        nat.check(self.lib.vrg_enqueue_advance(self._h))

    def enqueue_table(self):
        nat.check(self.lib.vrg_enqueue_table(self._h))

    def apply_flips(self, coords) -> dict:
        """One update() with caller-chosen flips (VRG:124,156-259): ``coords`` = rows of (z, y, x)."""
        c = np.ascontiguousarray(coords, dtype=np.int64).reshape(-1, 3)
        r = nat.Result()
        nat.check(self.lib.vrg_apply_flips(self._h, c.ctypes.data if c.size else None, c.shape[0], ctypes.byref(r)))
        return self._res(r)

    def apply_flips_device(self, rows_ptr, n: int) -> dict:
        """``apply_flips`` with ``n`` int64 rows (z, y, x) in device memory, checked on the device before anything changes."""
        r = nat.Result()
        nat.check(self.lib.vrg_apply_flips_device(self._h, nat.vp(rows_ptr or None), int(n), ctypes.byref(r)))
        return self._res(r)

    def profile(self, enable=True):
        nat.check(self.lib.vrg_profile(self._h, int(bool(enable))))

    def get_profile(self) -> dict:
        ms = (ctypes.c_double * 2)()
        n = (nat.i64 * 2)()
        nat.check(self.lib.vrg_get_profile(self._h, ctypes.addressof(ms), ctypes.addressof(n)))
        return {"decide_ms": ms[0], "decide_launches": int(n[0]), "cancel_ms": ms[1], "cancel_launches": int(n[1])}

    def get_tail_profile(self) -> dict:
        """Mean microseconds per phase of the fused tail kernel (first / last block of its grid), see vrg_get_tail_profile."""
        us = (ctypes.c_double * 14)()
        n = nat.i64(0)
        nat.check(self.lib.vrg_get_tail_profile(self._h, ctypes.addressof(us), ctypes.byref(n)))
        names = ("cancel", "barrier1", "phase2", "barrier2", "phase3", "pipe_halo_push", "pipe_counters")
        return {"launches": int(n.value), "first_block_us": {k: us[i] for i, k in enumerate(names)},
                "last_block_us": {k: us[7 + i] for i, k in enumerate(names)}}

    def use_separate_global_stats(self):
        nat.check(self.lib.vrg_use_separate_global_stats(self._h))

    def p2p_connect(self, rank: int, world: int, all_gather_bytes):
        """Peer-memory transport: export this rank's IPC handles, gather everyone's with ``all_gather_bytes``
        (a callable: bytes -> list of bytes in rank order), and map the peers' buffers."""
        mine = ctypes.create_string_buffer(nat.P2P_HANDLE_BYTES)
        nat.check(self.lib.vrg_p2p_export(self._h, int(world), ctypes.addressof(mine)))
        everyone = all_gather_bytes(bytes(mine.raw))
        blob = ctypes.create_string_buffer(b"".join(everyone), nat.P2P_HANDLE_BYTES * int(world))
        nat.check(self.lib.vrg_p2p_connect(self._h, int(rank), int(world), ctypes.addressof(blob)))

    def params_signature(self) -> int:
        sig = ctypes.c_uint64(0)
        nat.check(self.lib.vrg_params_signature(self._h, ctypes.byref(sig)))
        return int(sig.value)

    def buffer(self, which):
        p, n = nat.vp(), nat.i64()
        nat.check(self.lib.vrg_buffer_info(self._h, which, ctypes.byref(p), ctypes.byref(n)))
        return p.value, n.value

    def plane_geometry(self):
        a, b, c = nat.i64(), nat.i64(), nat.i64()
        nat.check(self.lib.vrg_plane_geometry(self._h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        return a.value, b.value, c.value

    # -- outputs ----------------------------------------------------------------------------
    def labels(self) -> np.ndarray:
        out = np.empty((self.own_planes,) + self.shape[1:], dtype=np.uint8)
        nat.check(self.lib.vrg_download_labels(self._h, out.ctypes.data))
        return out

    def segmented_map(self) -> np.ndarray:
        out = np.empty((self.own_planes,) + self.shape[1:], dtype=np.uint8)
        nat.check(self.lib.vrg_download_segmented_map(self._h, out.ctypes.data))
        return out

    def segmented_map_i64(self, out=None) -> np.ndarray:
        """segmentedMap in the reference's dtype (int64 0/1, VRG:45-46), own planes."""
        if out is None:
            out = np.empty((self.own_planes,) + self.shape[1:], dtype=np.int64)
        assert out.dtype == np.int64 and out.flags.c_contiguous and out.size == self.own_planes * self.shape[1] * self.shape[2]
        nat.check(self.lib.vrg_download_segmented_map_i64(self._h, out.ctypes.data))
        return out

    def count_nonzero(self) -> int:
        """np.count_nonzero of the own planes of the intensity volume, counted on the device (VRG:95)."""
        n = nat.i64(0)
        nat.check(self.lib.vrg_count_nonzero(self._h, ctypes.byref(n)))
        return int(n.value)

    def labels_hash(self) -> int:
        """Position-sensitive 64-bit hash of the own planes' labels; slab hashes add up (mod 2^64) to the whole volume's."""
        v = ctypes.c_uint64(0)
        nat.check(self.lib.vrg_labels_hash(self._h, ctypes.byref(v)))
        return int(v.value)

    def labels_device(self, dev_ptr: int):
        nat.check(self.lib.vrg_labels_device(self._h, nat.vp(dev_ptr)))

    def labels_device_typed(self, dev_ptr: int, dtype: int, segmented_only: bool = False):
        """Own planes' labels 0..4 (or the 0/1 segmented map) as ``dtype`` (``nat.DTYPE_*``) into a device buffer, on the
        handle's stream (no synchronisation)."""
        nat.check(self.lib.vrg_labels_device_typed(self._h, nat.vp(dev_ptr), int(dtype), int(bool(segmented_only))))

    def segmented_device(self, rows_ptr, cap: int) -> int:
        """Rows (z, y, x) of the own planes' segmented voxels, C order, compacted on the device into ``rows_ptr`` (int64,
        ``cap`` rows; None: count only).  Returns their number; rows beyond ``cap`` are not written."""
        n = nat.i64(0)
        nat.check(self.lib.vrg_segmented_device(self._h, nat.vp(rows_ptr or None), int(cap), ctypes.byref(n)))
        return int(n.value)

    def band_rows_device(self, which: int, rows_ptr, cap: int) -> int:
        """``segmented_device`` for ``which`` = 0 (segmented), 1 (inner band, label 1) or 2 (outer band, label 2)."""
        n = nat.i64(0)
        nat.check(self.lib.vrg_band_rows_device(self._h, int(which), nat.vp(rows_ptr or None), int(cap), ctypes.byref(n)))
        return int(n.value)

    def band_sums_device(self, pin_ptr: int, pout_ptr: int):
        """update()'s innerProb / outerProb of the current table into two float64 device buffers of the own planes (C order),
        on the handle's stream (no synchronisation)."""
        nat.check(self.lib.vrg_band_sums_device(self._h, nat.vp(pin_ptr), nat.vp(pout_ptr)))

    def segmented(self, at_most=None) -> np.ndarray:
        """Rows (z, y, x) of the segmented voxels of the own planes, C order.  ``at_most``: an upper bound of their number
        (e.g. the run's ``n_in``) saves the counting pass over the bit-plane."""
        n = nat.i64(0)
        if at_most is None:
            nat.check(self.lib.vrg_download_segmented(self._h, None, 0, ctypes.byref(n)))
            at_most = n.value
        out = np.empty((int(at_most), 3), dtype=np.int64)
        if at_most:
            nat.check(self.lib.vrg_download_segmented(self._h, out.ctypes.data, int(at_most), ctypes.byref(n)))
            if n.value > at_most:  # the bound was wrong: once more with the count
                return self.segmented()
        return out[: n.value]

    def trace(self) -> np.ndarray:
        cap = int(self.cfg.iter_max) + 2
        out = np.zeros((cap, 3), dtype=np.int64)
        n = nat.i64(0)
        nat.check(self.lib.vrg_get_trace(self._h, out.ctypes.data, cap, ctypes.byref(n)))
        return out[: n.value].copy()

    def band_sums(self):
        """Continuous mode: (flat voxel index, pin/n_in, pout/n_out) of every band voxel at the last decision."""
        n = nat.i64(0)
        nat.check(self.lib.vrg_get_band_sums(self._h, None, None, None, 0, ctypes.byref(n)))
        vox = np.empty(n.value, dtype=np.int64)
        pin, pout = np.empty(n.value), np.empty(n.value)
        if n.value:
            nat.check(self.lib.vrg_get_band_sums(self._h, vox.ctypes.data, pin.ctypes.data, pout.ctypes.data, n.value,
                                                 ctypes.byref(n)))
        return vox, pin, pout

    def table(self):
        """(levels, pin, pout) of the most recent decision table (VRG:79-82)."""
        r = self.poll()
        L = r["n_levels"]
        lv, pin, pout = (np.zeros(L, dtype=np.float64) for _ in range(3))
        nat.check(self.lib.vrg_get_table(self._h, pin.ctypes.data, pout.ctypes.data, L))
        nat.check(self.lib.vrg_get_table_levels(self._h, lv.ctypes.data, L))
        return lv, pin, pout
