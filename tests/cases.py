"""Seeded op-level test cases shared by oracle/make_golden.py (reference CUDA ext on a B200),
tests/test_oracle_golden.py (C oracle vs golden, CPU) and tests/test_ops_gpu.py (our CUDA vs both).

Every case is a dict of numpy inputs; `sha` pins the exact input bytes so a drifting RNG is
caught instead of silently comparing different problems.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from spacap3d_b200.scenes import make_scene_xyz  # noqa: E402


def sha(*arrays):
    h = hashlib.sha1()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(str(a.dtype).encode() + str(a.shape).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def _lattice(n_side, spacing=0.25, offset=0.0):
    g = np.arange(n_side, dtype=np.float32) * np.float32(spacing) - np.float32(offset)
    p = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    return np.ascontiguousarray(p, np.float32)


# ------------------------------------------------------------------ FPS ---------------------
def fps_cases():
    c = {}
    rng = np.random.default_rng(101)
    c["tiny_n9"] = (rng.standard_normal((2, 9, 3)).astype(np.float32), 4)
    c["n1"] = (rng.standard_normal((1, 1, 3)).astype(np.float32), 3)
    c["n2"] = (rng.standard_normal((2, 2, 3)).astype(np.float32), 2)
    c["n300_T256"] = (rng.uniform(-2, 2, (2, 300, 3)).astype(np.float32), 64)
    c["n513"] = (rng.uniform(-2, 2, (1, 513, 3)).astype(np.float32), 200)
    c["n1000_T512"] = (rng.uniform(-3, 3, (3, 1000, 3)).astype(np.float32), 256)
    c["m_gt_n"] = (rng.uniform(-1, 1, (2, 20, 3)).astype(np.float32), 32)
    # duplicates: 600 distinct points resampled to 2048, npoint beyond #distinct => zero-distance ties
    base = rng.uniform(-3, 3, (2, 600, 3)).astype(np.float32)
    pick = rng.integers(0, 600, (2, 2048))
    dup = np.take_along_axis(base, pick[..., None].repeat(3, -1), 1)
    c["dup_2048"] = (np.ascontiguousarray(dup), 1024)
    # lattice: massive exact ties between distinct points (tie-break = bit-reversed thread id, F4)
    lat = _lattice(16, 0.25, 1.875)
    c["lattice_4096"] = (np.stack([lat, lat[::-1].copy()], 0), 512)
    lat5 = _lattice(5, 0.5, 1.0)
    c["lattice_125"] = (lat5[None].copy(), 125)
    # near-origin skip (F5): |p|^2 <= 1e-3 never selected / never updated; index 0 itself near origin
    near = rng.uniform(-0.02, 0.02, (2, 1500, 3)).astype(np.float32)
    far = rng.uniform(-2, 2, (2, 1500, 3)).astype(np.float32)
    mix = np.where(rng.random((2, 1500, 1)) < 0.4, near, far).astype(np.float32)
    mix[0, 0] = [0.001, -0.002, 0.0005]
    # points sitting right at the threshold |p|^2 ~ 1e-3
    thr = np.sqrt(np.float32(1e-3) / np.float32(3.0))
    for t in range(40):
        mix[1, 10 + t] = np.float32(thr) * (1 + (t - 20) * 1e-7) * np.array([1, 1, 1], np.float32)
    c["origin_mix"] = (np.ascontiguousarray(mix), 700)
    c["all_skipped"] = (rng.uniform(-0.01, 0.01, (2, 64, 3)).astype(np.float32), 8)
    # the BASELINE shape: 40k-point room scenes, one with duplicates (resampled with replacement)
    sc = np.stack([make_scene_xyz(11, 40000, with_replacement=False),
                   make_scene_xyz(12, 40000, with_replacement=True)], 0)
    c["scene_40k"] = (sc, 2048)
    return c


def fps_large_cases():
    """Clouds large enough (N >= 8192) for the library's Morton-sorted, culled FPS kernel; checked against
    the oracle (itself pinned on fps_cases) rather than against stored reference outputs."""
    c = {}
    rng = np.random.default_rng(202)
    # exact ties everywhere: 24^3 lattice, forwards and reversed
    lat = _lattice(24, 0.25, 2.875)
    c["lattice_13824"] = (np.stack([lat, lat[::-1].copy()], 0), 700)
    # heavy duplication: 700 distinct points resampled to 16384, npoint beyond #distinct
    base = rng.uniform(-3, 3, (2, 700, 3)).astype(np.float32)
    pick = rng.integers(0, 700, (2, 16384))
    c["dup_16384"] = (np.ascontiguousarray(np.take_along_axis(base, pick[..., None].repeat(3, -1), 1)), 1024)
    # near-origin skip inside a large cloud, first point itself skipped in scene 0
    near = rng.uniform(-0.02, 0.02, (2, 10000, 3)).astype(np.float32)
    far = rng.uniform(-2, 2, (2, 10000, 3)).astype(np.float32)
    mix = np.where(rng.random((2, 10000, 1)) < 0.3, near, far).astype(np.float32)
    mix[0, 0] = [0.001, -0.002, 0.0005]
    c["origin_mix_10000"] = (np.ascontiguousarray(mix), 600)
    # size edges of the culled kernel: smallest N, largest N of an 8x256x20 cluster, one past it
    c["n8192"] = (rng.uniform(-3, 3, (1, 8192, 3)).astype(np.float32), 300)
    c["n40960"] = (rng.uniform(-4, 4, (1, 40960, 3)).astype(np.float32), 512)
    c["n40961"] = (rng.uniform(-4, 4, (1, 40961, 3)).astype(np.float32), 256)
    # degenerate extents: all points on a plane / on a line / identical
    plane = rng.uniform(-3, 3, (1, 9000, 3)).astype(np.float32)
    plane[..., 2] = 1.5
    line = np.zeros((1, 9000, 3), np.float32)
    line[..., 0] = rng.uniform(-5, 5, (1, 9000)).astype(np.float32)
    line[..., 1] = 0.25
    c["plane_line_9000"] = (np.concatenate([plane, line], 0), 400)
    c["identical_8500"] = (np.full((1, 8500, 3), 0.75, np.float32), 70)
    # clustered (very non-uniform density) cloud
    cen = rng.uniform(-4, 4, (1, 12, 3))
    which = rng.integers(0, 12, (1, 20000))
    pts = np.take_along_axis(cen, which[..., None].repeat(3, -1), 1) + rng.normal(0, 0.05, (1, 20000, 3))
    c["clusters_20000"] = (pts.astype(np.float32), 1024)
    return c


def fps_follow_on(xyz, idx, npoint):
    """new_xyz gathered with idx, as the SA module does (pointnet2_modules.py:240-242)."""
    return np.take_along_axis(xyz, idx[..., None].astype(np.int64).repeat(3, -1), 1)[:, :npoint]


# ------------------------------------------------------------------ ball query --------------
def ball_query_cases():
    """name -> (new_xyz, xyz, radius, nsample)"""
    c = {}
    rng = np.random.default_rng(202)
    xyz = rng.uniform(-1, 1, (2, 500, 3)).astype(np.float32)
    new = rng.uniform(-1.5, 1.5, (2, 70, 3)).astype(np.float32)  # some centres have empty balls
    c["rand_small_r"] = (new, xyz, 0.15, 16)
    c["rand_big_r"] = (new, xyz, 5.0, 32)            # every ball full after 32 points
    c["nsample1"] = (new, xyz, 0.4, 1)
    c["nsample_gt_n"] = (new[:, :10].copy(), xyz[:, :20].copy(), 0.8, 48)
    lat = _lattice(8, 0.25, 0.875)
    c["lattice_boundary"] = (lat[None, ::7].copy(), lat[None].copy(), 0.25, 8)  # d2 == r2 exactly: not a hit
    c["lattice_boundary2"] = (lat[None, ::5].copy(), lat[None].copy(), 0.5, 64)
    c["n33"] = (rng.uniform(-1, 1, (3, 5, 3)).astype(np.float32),
                rng.uniform(-1, 1, (3, 33, 3)).astype(np.float32), 0.9, 7)
    sc = np.stack([make_scene_xyz(21, 40000, with_replacement=False),
                   make_scene_xyz(22, 40000, with_replacement=True)], 0)
    # centres: a strided subset of the cloud itself (what FPS would return is checked elsewhere)
    new_sc = np.ascontiguousarray(sc[:, ::40][:, :1000])
    c["scene_sa1"] = (new_sc, sc, 0.2, 64)
    sub = np.ascontiguousarray(sc[:, ::20])            # 2000 pts
    c["scene_sa2"] = (np.ascontiguousarray(sub[:, ::2]), sub, 0.4, 32)
    c["scene_sa4"] = (np.ascontiguousarray(sub[:, ::8][:, :256]), np.ascontiguousarray(sub[:, :512]), 1.2, 16)
    # --- cases that take the uniform-grid path (N >= 4096 and N*M >= 2^22) -------------------------
    rng = np.random.default_rng(909)
    big = rng.uniform(-2, 2, (2, 6000, 3)).astype(np.float32)
    cen = rng.uniform(-2.6, 2.6, (2, 800, 3)).astype(np.float32)          # some centres outside the bbox
    c["grid_rand_r03"] = (cen, big, 0.3, 32)
    c["grid_rand_tiny_r"] = (cen, big, 0.02, 8)                            # mostly empty balls
    c["grid_rand_huge_r"] = (cen, big, 1.5, 64)                            # > 512 hits per centre: fallback scan
    c["grid_rand_r_gt_extent"] = (cen, big, 9.0, 16)                       # one cell
    lat = _lattice(17, 0.25, 2.0)                                          # 4913 points, spacing == radius
    c["grid_lattice_boundary"] = (np.ascontiguousarray(lat[None, ::5][:, :900]), lat[None].copy(), 0.25, 16)
    c["grid_lattice_r05"] = (np.ascontiguousarray(lat[None, ::5][:, :900]) + np.float32(0.125), lat[None].copy(), 0.5, 48)
    flat = big.copy(); flat[..., 2] = np.float32(0.5)                      # degenerate (zero) extent in z
    c["grid_flat"] = (np.ascontiguousarray(flat[:, ::7][:, :750]), flat, 0.25, 24)
    c["scene_sa1_ns16"] = (new_sc, sc, 0.35, 16)                           # more hits than slots
    return c


# ------------------------------------------------------------------ three_nn ----------------
def three_nn_cases():
    """name -> (unknown, known)"""
    c = {}
    rng = np.random.default_rng(303)
    c["fp1"] = (rng.uniform(-3, 3, (2, 512, 3)).astype(np.float32),
                rng.uniform(-3, 3, (2, 256, 3)).astype(np.float32))
    c["fp2"] = (rng.uniform(-3, 3, (2, 1024, 3)).astype(np.float32),
                rng.uniform(-3, 3, (2, 512, 3)).astype(np.float32))
    c["m2"] = (rng.standard_normal((1, 17, 3)).astype(np.float32),
               rng.standard_normal((1, 2, 3)).astype(np.float32))
    c["m1"] = (rng.standard_normal((2, 5, 3)).astype(np.float32),
               rng.standard_normal((2, 1, 3)).astype(np.float32))
    lat = _lattice(6, 0.5, 1.25)
    c["lattice_ties"] = (lat[None, ::3].copy() + np.float32(0.25), lat[None].copy())
    known = rng.uniform(-1, 1, (1, 300, 3)).astype(np.float32)
    c["subset_zero_dist"] = (known[:, ::2].copy(), known)    # unknown is a subset: d = 0 exactly
    return c


# ------------------------------------------------------------------ index ops ---------------
def gather_cases():
    """name -> (points (B,C,N), idx (B,M))"""
    rng = np.random.default_rng(404)
    c = {}
    c["xyz"] = (rng.standard_normal((2, 3, 1000)).astype(np.float32),
                rng.integers(0, 1000, (2, 256)).astype(np.int32))
    c["c7_dups"] = (rng.standard_normal((3, 7, 50)).astype(np.float32),
                    rng.integers(0, 50, (3, 120)).astype(np.int32))
    c["m1"] = (rng.standard_normal((1, 2, 9)).astype(np.float32), np.array([[4]], np.int32))
    return c


def group_cases():
    """name -> (points (B,C,N), idx (B,np,ns))"""
    rng = np.random.default_rng(505)
    c = {}
    c["sa_like"] = (rng.standard_normal((2, 16, 2048)).astype(np.float32),
                    rng.integers(0, 2048, (2, 128, 32)).astype(np.int32))
    c["c3"] = (rng.standard_normal((2, 3, 500)).astype(np.float32),
               rng.integers(0, 500, (2, 33, 7)).astype(np.int32))
    c["c1_ns1"] = (rng.standard_normal((1, 1, 10)).astype(np.float32),
                   rng.integers(0, 10, (1, 5, 1)).astype(np.int32))
    idx = rng.integers(0, 300, (2, 64, 16)).astype(np.int32)
    idx[:, :, 5:] = idx[:, :, :1]                     # ball-query style padding: one index repeated
    c["padded"] = (rng.standard_normal((2, 130, 300)).astype(np.float32), idx)
    c["odd"] = (rng.standard_normal((1, 5, 77)).astype(np.float32),
                rng.integers(0, 77, (1, 13, 3)).astype(np.int32))
    return c


def group_grad_big_cases():
    """name -> (idx (B,np,ns), C, N): shapes that take the list-based (atomic-free) backward."""
    rng = np.random.default_rng(515)
    c = {}

    def padded(B, N, npoint, ns, fill):
        idx = rng.integers(0, N, (B, npoint, ns)).astype(np.int32)
        cnt = rng.integers(1, ns + 1, (B, npoint, 1))
        first = np.minimum(idx[:, :, :1], fill)            # hubs: low indices collect the padding
        return np.where(np.arange(ns)[None, None, :] < cnt, idx, first).astype(np.int32)

    c["sa2_like_two_partitions"] = (padded(2, 2048, 1024, 32, 40), 9, 2048)       # S=32768 -> H=2, CT=1
    c["sa3_like"] = (padded(2, 1024, 512, 16, 25), 10, 1024)                      # S=8192  -> H=1, CT=2
    c["sa4_like_ct4"] = (padded(3, 512, 256, 16, 10), 7, 512)                     # S=4096  -> CT=4, C%4 != 0
    c["three_partitions"] = (padded(1, 3000, 1000, 60, 100), 6, 3000)             # S=60000 -> H=3 (N <= 512*C)
    c["odd_unaligned"] = (padded(2, 333, 77, 13, 5), 5, 333)                      # S=1001: no bulk copy
    c["one_hub"] = (np.zeros((1, 64, 16), np.int32) + 7, 6, 50)                   # every position -> point 7
    # N > 8192: one list per point over all positions + point-owned gather (atomic cursors: order not deterministic)
    c["large_cloud"] = (padded(2, 20000, 512, 64, 300), 9, 20000)                 # S=32768, CT=8 + a 1-channel tile
    c["large_cloud_hubs"] = (padded(1, 9000, 300, 64, 3), 8, 9000)                # four hubs with very long lists
    return c


def interp_cases():
    """name -> (points (B,C,m), idx (B,n,3), weight (B,n,3))"""
    rng = np.random.default_rng(606)
    c = {}
    for name, (B, C, m, n) in {"fp1": (2, 256, 256, 512), "odd": (1, 5, 7, 13), "c1": (2, 1, 3, 4)}.items():
        w = rng.uniform(0.01, 1, (B, n, 3)).astype(np.float32)
        w = (w / w.sum(-1, keepdims=True)).astype(np.float32)
        c[name] = (rng.standard_normal((B, C, m)).astype(np.float32),
                   rng.integers(0, m, (B, n, 3)).astype(np.int32), w)
    # the reference's own test fixture (pointnet2_test.py:18-30)
    c["ref_test"] = (rng.standard_normal((1, 2, 4)).astype(np.float32),
                     np.array([[[0, 1, 2], [1, 2, 3]]], np.int32),
                     np.array([[[1, 1, 1], [2, 2, 2]]], np.float32))
    return c


def ball_query_extra_cases():
    """Ball-query cases without golden vectors (checked against the oracle and the live reference ext): long thin
    clouds whose uniform grid has many hundreds of cells along one axis, where the fp32 cell arithmetic is least
    accurate (round-1 advisor finding), also far away from the origin."""
    rng = np.random.default_rng(909)
    c = {}
    for name, (length, off, r) in {"corridor_900_cells": (180.0, 0.0, 0.2), "corridor_far_from_origin": (150.0, 3000.0, 0.2),
                                   "corridor_2000_cells": (100.0, -50.0, 0.05)}.items():
        pts = rng.uniform(0, 1, (1, 12000, 3)).astype(np.float64)
        pts[..., 0] = pts[..., 0] * length + off
        pts[..., 1] *= 0.6
        pts[..., 2] *= 0.3
        xyz = pts.astype(np.float32)
        new = np.ascontiguousarray(xyz[:, ::12]).copy()
        new[:, ::3, 0] += np.float32(r * 0.999)             # centres whose ball reaches into the next cells
        c[name] = (new, xyz, r, 16)
    return c


def interp_big_cases():
    """Larger interpolation shapes (no golden vectors: checked against the oracle and the live reference ext):
    FP2's, config 5's x4 cloud, and a ragged one (n % 4 != 0, channel count not a multiple of the tile)."""
    rng = np.random.default_rng(707)
    c = {}
    for name, (B, C, m, n) in {"fp2": (2, 256, 512, 1024), "config5_x4": (1, 40, 2048, 4096),
                               "ragged": (3, 33, 100, 1022)}.items():
        w = rng.uniform(0.01, 1, (B, n, 3)).astype(np.float32)
        w = (w / w.sum(-1, keepdims=True)).astype(np.float32)
        c[name] = (rng.standard_normal((B, C, m)).astype(np.float32),
                   rng.integers(0, m, (B, n, 3)).astype(np.int32), w)
    return c


def grad_for(tag, shape):
    """Deterministic upstream gradient for a named case."""
    seed = int(hashlib.sha1(tag.encode()).hexdigest()[:8], 16)
    return np.random.default_rng(seed).standard_normal(shape).astype(np.float32)
