#!/usr/bin/env python
"""Fixtures for the feature transform of distance_transform_edt (tests/test_gpu_edt_ft.py): SciPy's own
``distance_transform_edt(mask, sampling=s, return_indices=True)`` -- int32 indices and float64 distances -- for unit
spacing and for an anisotropic spacing, on masks chosen for what decides the feature transform:

    lattice      zeros on a lattice: most voxels have several equally near zero voxels (ties)
    vessel_tree  thin tubes in a background volume: the vessel-radius case, foreground of a few voxels across
    ellipsoid    a solid ellipsoid: long stacks in every pass
    line_x       1 x 1 x n and n x 1 x 1: one-voxel-thin volumes along either end of the pass order
    line_z
    odd_x        random blobs with an odd row length (partial tiles of the x pass)

    python tests/golden/edt_ft/make_golden_ft.py   (writes the .npz files next to this script)
"""
import os

import numpy as np
from scipy import ndimage as ndi

HERE = os.path.dirname(os.path.abspath(__file__))
SAMPLING = (1.3, 0.5, 0.7)


def masks():
    rng = np.random.default_rng(20261022)
    lat = np.ones((12, 14, 17), np.uint8)
    lat[::3, ::4, ::2] = 0
    lat[5, 6, 7] = 0
    yield "lattice", lat

    tree = np.zeros((20, 24, 29), np.uint8)
    z, y, x = np.meshgrid(np.arange(20), np.arange(24), np.arange(29), indexing="ij")
    for (p, q, r) in (((2, 3, 1), (17, 20, 27), 2.2), ((10, 12, 14), (3, 21, 6), 1.5), ((10, 12, 14), (18, 2, 25), 1.0)):
        p, q = np.array(p, float), np.array(q, float)
        d = q - p
        t = np.clip(((z - p[0]) * d[0] + (y - p[1]) * d[1] + (x - p[2]) * d[2]) / (d @ d), 0, 1)
        dist2 = (z - p[0] - t * d[0]) ** 2 + (y - p[1] - t * d[1]) ** 2 + (x - p[2] - t * d[2]) ** 2
        tree[dist2 <= r * r] = 1
    yield "vessel_tree", tree

    e = ((((z - 9.5) / 8.7) ** 2 + ((y - 11.5) / 10.2) ** 2 + ((x - 14.0) / 13.1) ** 2) <= 1.0).astype(np.uint8)
    yield "ellipsoid", e

    line = np.ones((1, 1, 37), np.uint8)
    line[0, 0, [0, 9, 10, 30]] = 0
    yield "line_x", line
    yield "line_z", np.ascontiguousarray(line.reshape(37, 1, 1))

    blobs = ndi.gaussian_filter(rng.random((9, 10, 31)), 1.2)
    yield "odd_x", (blobs > np.quantile(blobs, 0.35)).astype(np.uint8)


def main():
    for name, m in masks():
        assert (m == 0).any() and (m != 0).any(), name
        out = {"mask": m, "sampling": np.array(SAMPLING)}
        for tag, s in (("unit", None), ("sampled", SAMPLING)):
            dt, ft = ndi.distance_transform_edt(m, sampling=s, return_indices=True)
            out["dt_" + tag], out["ft_" + tag] = dt, ft
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
        print(name, m.shape, int(m.sum()))


if __name__ == "__main__":
    main()
