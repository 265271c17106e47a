"""The bucketed FPS sampler takes the runner-up a2 of a round as the next pick when that is provably what the
sequential algorithm does (csrc/fps.cu, fps_bucket_kernel).  These clouds send it through every branch of that
rule: a2 accepted, rejected by the distance test, by the second key of the pick's bucket, by a tie at the runner-up,
the last pick of a call at odd and even npoint, and selectable points running out.

Every cloud is built so that each bucket of the sampler is one cell of its 32^3 Hilbert grid: the box is
[-16, 16]^3 (cells are unit cubes), and every occupied cell holds exactly one bucket's worth of points (32 below
20,481 points, 64 above).  Coordinates are multiples of 1/64, so every squared distance is exact in fp32 and the
numpy replay below computes what the kernel computes.  The CPU test asserts that each case reaches its branches;
the GPU test that the sampler equals the oracle, new_xyz included, and flags strict sequences exactly."""
import functools

import numpy as np
import pytest

import cases
import oracle

GRID = 64                                   # coordinate resolution: 1/64


def _cells(rng, n):
    """n distinct cells of the 32^3 grid, none of them next to the origin (|p|^2 <= 1e-3 is never selected), with
    (0,0,0) and (31,31,31) among them so that the box is exactly [-16, 16]^3."""
    codes = set()
    near = {15, 16}
    while len(codes) < n - 2:
        c = tuple(int(v) for v in rng.integers(0, 32, 3))
        if c in ((0, 0, 0), (31, 31, 31)) or all(v in near for v in c):
            continue
        codes.add(c)
    return [(0, 0, 0)] + sorted(codes) + [(31, 31, 31)]


def _cloud(seed, ncell, dup=0, plain=0):
    """ncell clusters of one bucket each, of distinct points but for these: the first `dup` points of every cluster
    are repeated in place of its last ones, and the last `plain` clusters hold one point repeated."""
    rng = np.random.default_rng(seed)
    per = 32 if ncell * 32 <= 20480 else 64
    pts = []
    for i, c in enumerate(_cells(rng, ncell)):
        n = 1 if i >= ncell - plain else per
        off = rng.choice(GRID ** 3, n, replace=False)
        off = np.stack([off // GRID ** 2, off // GRID % GRID, off % GRID], 1)
        if i == 0:
            off[0] = 0                                       # (-16, -16, -16)
        if i == ncell - 1:
            off[0] = GRID                                    # (16, 16, 16): cell 31 holds [15, 16]
        cl = np.repeat(off, per // n, 0)
        if dup:
            cl[per - dup:] = cl[:dup]
        pts.append(np.asarray(c, np.float32) - 16 + cl.astype(np.float32) / GRID)
    xyz = np.concatenate(pts, 0)
    return xyz[rng.permutation(len(xyz))]


@functools.lru_cache(None)
def two_pick_cases():
    """name -> (xyz (B, N, 3), npoints, branches the rounds must reach)"""
    c = {}
    # random clusters in every compiled shape: 32-point buckets in one / two table slots per lane, 64-point ones.
    # 129 cells, not 128: 4,096 points or fewer go to the single-CTA sampler
    c["random_4128"] = (_cloud(1, 129)[None], (2, 3, 4, 5, 512, 513),
                        {"accept", "dist", "key2", "last", "accept_final"})
    c["random_19200"] = (_cloud(2, 600)[None], (700, 701), {"accept", "dist", "key2"})
    c["random_25600"] = (_cloud(3, 400)[None], (600,), {"accept", "dist", "key2"})
    c["random_40960"] = (_cloud(4, 640)[None], (511,), {"accept", "dist", "key2"})
    # a duplicated point at the top of a bucket: key2 == key, a tie wherever it is the runner-up
    c["duplicates_4128"] = (_cloud(5, 129, dup=8)[None], (800,), {"accept", "tie", "key2"})
    # fewer distinct points than picks: the keys run down to "distance 0" mid-call; scene 1 has no selectable point
    few = _cloud(6, 129, plain=64)
    skipped = np.random.default_rng(6).uniform(-0.01, 0.01, few.shape).astype(np.float32)
    c["running_out_4128"] = (np.stack([few, skipped], 0), (2200,), {"accept", "exhausted", "none"})
    return c


def _bucket(xyz):
    """Bucket of every point: its cell (the clouds above hold one bucket per occupied cell).  This restates the grid
    of fps_morton_sort_kernel in csrc/fps.cu -- 32 cells per axis over the cloud's bounding box -- for a box of exactly
    [-16, 16]^3, where a cell is a unit cube."""
    cell = np.clip(np.floor(xyz.astype(np.float64) + 16), 0, 31).astype(np.int64)
    return (cell[:, 0] * 32 + cell[:, 1]) * 32 + cell[:, 2]


def _assert_one_bucket_per_cell(xyz):
    """The replay's premise: the box is [-16, 16]^3 and every occupied cell holds exactly one bucket (32 points up to
    20,480, 64 above, fb_bucket_size in csrc/fps.cu), so the sort cannot split a cell between buckets."""
    np.testing.assert_array_equal(xyz.min(0), [-16, -16, -16])
    np.testing.assert_array_equal(xyz.max(0), [16, 16, 16])
    _, counts = np.unique(_bucket(xyz), return_counts=True)
    assert (counts == (32 if len(xyz) <= 20480 else 64)).all()


def replay(xyz, npoint, picks):
    """The bucketed sampler's rounds on one scene, in exact arithmetic: the branch each round takes and whether
    every pick was the strict unique maximum.  `picks` are the oracle's; a taken runner-up must be the next one."""
    p = xyz.astype(np.float64)
    sel = (p * p).sum(1) > 1e-3
    t = np.where(sel, 1e10, -1.0)                            # -1: key 0, never selected
    bucket = _bucket(xyz)

    def apply(k):
        np.minimum(t, ((p - p[k]) ** 2).sum(1), out=t, where=sel)

    def strict_pick(k):
        m = t.max()
        return bool(m >= 0 and t[k] == m and (t == m).sum() == 1)

    labels, strict = [], True
    apply(0)
    j = 1
    while j < npoint:
        if t.max() < 0:                                      # nothing selectable: point 0, one pick
            labels.append("none")
            strict = False
            assert picks[j] == 0
            apply(0)
            j += 1
            continue
        a1 = picks[j]
        assert t[a1] == t.max()
        strict = strict and strict_pick(a1)
        a2, label = None, "last"
        if j + 1 < npoint:
            in_a1 = bucket == bucket[a1]
            key2 = np.sort(t[in_a1])[-2]                     # second-largest value of the pick's bucket
            out = np.where(in_a1, -1.0, t)
            ck = out.max()
            if ck <= 0:
                label = "exhausted"                          # a2 at distance 0 would tie a1 after its update
            elif key2 >= ck:
                label = "key2"
            elif (out == ck).sum() > 1:
                label = "tie"
            else:
                a2 = int(out.argmax())
                label = "dist" if ((p[a2] - p[a1]) ** 2).sum() < t[a2] else "accept"
                if label == "accept" and j + 2 == npoint:
                    label = "accept_final"
                if label == "dist":
                    a2 = None
        labels.append(label)
        apply(a1)
        if a2 is not None:
            assert picks[j + 1] == a2 and strict_pick(a2)
            apply(a2)
            j += 2
        else:
            j += 1
    return labels, strict


def _params():
    return [(name, m) for name, (_, ms, _) in two_pick_cases().items() for m in ms]


def test_replay_reaches_every_branch():
    """Each constructed cloud reaches the branches it is built for (and a taken runner-up is always the next
    sequential pick); over all npoints of a cloud, a call ends both on a lone last pick and on a taken runner-up."""
    for name, (xyz, npoints, want) in two_pick_cases().items():
        assert 4096 < xyz.shape[1] <= 40960, name            # the bucketed sampler's range
        seen = set()
        for m in npoints:
            picks = oracle.furthest_point_sampling(xyz, m)
            for b in range(xyz.shape[0]):
                if (xyz[b].astype(np.float64) ** 2).sum(1).max() > 1e-3:     # not the scene of skipped points only
                    _assert_one_bucket_per_cell(xyz[b])
                labels, _ = replay(xyz[b], m, picks[b])
                seen.update(labels)
        assert want <= seen, (name, sorted(want - seen))


@pytest.fixture(scope="module")
def ext():
    from spacap3d_b200 import _ext
    return _ext


@pytest.mark.gpu
@pytest.mark.parametrize("name,npoint", _params())
def test_bucket_sampler_two_picks(ext, name, npoint):
    import torch
    xyz, _, _ = two_pick_cases()[name]
    want = oracle.furthest_point_sampling(xyz, npoint)
    with ext.launch_options(fps_algo=ext.FPS_BUCKET):
        idx, new_xyz, strict = ext.furthest_point_sampling_with_xyz(torch.from_numpy(xyz).cuda(), npoint,
                                                                    want_strict=True)
    np.testing.assert_array_equal(idx.cpu().numpy(), want)
    np.testing.assert_array_equal(new_xyz.cpu().numpy(), cases.fps_follow_on(xyz, want, npoint))
    flags = [int(replay(xyz[b], npoint, want[b])[1]) for b in range(xyz.shape[0])]
    assert strict.cpu().numpy().tolist() == flags
