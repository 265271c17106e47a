"""CPU: the C oracle (oracle/pointnet2_oracle.c) against the golden vectors in
tests/golden/ref_ops.npz, which are outputs of the REFERENCE's own CUDA extension (rebuilt
unmodified for sm_100a, run on a B200 by oracle/make_golden.py).  This is what pins the oracle.

Bar: bit-exact for every index tensor and every pure copy (gather/group forward, three_nn
distances, three_interpolate forward), which the file stores as digests of dtype, shape and bytes;
1e-6-relative for the atomically accumulated gradients, whose summation order on the GPU is arbitrary.
"""
import numpy as np
import pytest

import cases
import oracle


def _check_sha(golden, key, *arrays):
    assert str(golden[key]) == cases.sha(*arrays), "input generator drifted for " + key


def _assert_bits(golden, key, got):
    assert cases.sha(got) == str(golden[key]), "differs from the reference's output bit for bit: " + key


@pytest.mark.parametrize("name", list(cases.fps_cases().keys()))
def test_fps_matches_reference(golden, name):
    xyz, m = cases.fps_cases()[name]
    _check_sha(golden, f"fps/{name}/sha", xyz, np.int64(m))
    _assert_bits(golden, f"fps/{name}/idx", oracle.furthest_point_sampling(xyz, m))


@pytest.mark.parametrize("name", list(cases.ball_query_cases().keys()))
def test_ball_query_matches_reference(golden, name):
    new_xyz, xyz, r, ns = cases.ball_query_cases()[name]
    _check_sha(golden, f"ball_query/{name}/sha", new_xyz, xyz, np.float32(r), np.int64(ns))
    _assert_bits(golden, f"ball_query/{name}/idx", oracle.ball_query(new_xyz, xyz, r, ns))


@pytest.mark.parametrize("name", list(cases.three_nn_cases().keys()))
def test_three_nn_matches_reference(golden, name):
    unknown, known = cases.three_nn_cases()[name]
    _check_sha(golden, f"three_nn/{name}/sha", unknown, known)
    d2, idx = oracle.three_nn(unknown, known)
    _assert_bits(golden, f"three_nn/{name}/idx", idx)
    _assert_bits(golden, f"three_nn/{name}/dist2", d2)


@pytest.mark.parametrize("name", list(cases.gather_cases().keys()))
def test_gather_matches_reference(golden, name):
    pts, idx = cases.gather_cases()[name]
    out = oracle.gather_points(pts, idx)
    g = cases.grad_for("gather/" + name, out.shape)
    _check_sha(golden, f"gather/{name}/sha", pts, idx, g)
    _assert_bits(golden, f"gather/{name}/out", out)
    want = golden[f"gather/{name}/grad"]
    np.testing.assert_allclose(oracle.gather_points_grad(g, idx, pts.shape[2]), want,
                               rtol=1e-6, atol=1e-6 * max(1.0, np.abs(want).max()))


@pytest.mark.parametrize("name", list(cases.group_cases().keys()))
def test_group_matches_reference(golden, name):
    pts, idx = cases.group_cases()[name]
    out = oracle.group_points(pts, idx)
    g = cases.grad_for("group/" + name, out.shape)
    _check_sha(golden, f"group/{name}/sha", pts, idx, g)
    _assert_bits(golden, f"group/{name}/out", out)
    want = golden[f"group/{name}/grad"]
    np.testing.assert_allclose(oracle.group_points_grad(g, idx, pts.shape[2]), want,
                               rtol=1e-5, atol=2e-6 * max(1.0, np.abs(want).max()))


@pytest.mark.parametrize("name", list(cases.interp_cases().keys()))
def test_interpolate_matches_reference(golden, name):
    pts, idx, w = cases.interp_cases()[name]
    out = oracle.three_interpolate(pts, idx, w)
    g = cases.grad_for("interp/" + name, out.shape)
    _check_sha(golden, f"interp/{name}/sha", pts, idx, w, g)
    _assert_bits(golden, f"interp/{name}/out", out)   # same FMA order => same bits
    want = golden[f"interp/{name}/grad"]
    np.testing.assert_allclose(oracle.three_interpolate_grad(g, idx, w, pts.shape[2]), want,
                               rtol=1e-5, atol=2e-6 * max(1.0, np.abs(want).max()))


def test_golden_provenance(golden):
    assert "B200" in str(golden["meta/gpu"])


# ------------------------------------------------------------- known-answer tests (semantics) ---
def test_opt_n_threads_matches_integer_rule():
    """cuda_utils.h:15-19 uses log()/log(2.0); the product computes the same value with integers."""
    for n in list(range(1, 3000)) + [4095, 4096, 4097, 39999, 40000, 65535, 65536, 200000]:
        t = 1
        while t * 2 <= n and t * 2 <= 512:
            t *= 2
        assert oracle.opt_n_threads(n) == t, n


def test_fps_tie_break_is_bit_reversed_thread_id():
    """SURVEY F4: with all distances tied the block tree prefers the smallest bit-reversed
    thread id, NOT the lowest index."""
    # 4 points: p0 at origin-ish far corner, the rest all at the same distance from p0
    xyz = np.array([[[1, 1, 1], [2, 1, 1], [1, 2, 1], [1, 1, 2]]], np.float32)
    idx = oracle.furthest_point_sampling(xyz, 2)
    # T=4: thread ids 1,2,3 tie; bit-reversed (2 bits) -> 2,1,3 => thread 2 wins
    assert idx.tolist() == [[0, 2]]


def test_fps_skips_points_near_origin():
    xyz = np.array([[[0.5, 0, 0], [0.01, 0.01, 0.01], [0.6, 0, 0], [-3, 0, 0]]], np.float32)
    idx = oracle.furthest_point_sampling(xyz, 4)
    assert 1 not in idx[0, 1:].tolist()            # |p|^2 = 3e-4 <= 1e-3: never selected
    assert idx[0, 0] == 0 and idx[0, 1] == 3


def test_ball_query_padding_and_empty():
    xyz = np.array([[[0, 0, 0], [0.1, 0, 0], [5, 5, 5], [0.05, 0, 0]]], np.float32)
    new = np.array([[[0, 0, 0], [9, 9, 9]]], np.float32)
    idx = oracle.ball_query(new, xyz, 0.2, 5)
    assert idx[0, 0].tolist() == [0, 1, 3, 0, 0]   # ascending hits, padded with the first
    assert idx[0, 1].tolist() == [0, 0, 0, 0, 0]   # empty ball: zeros (F9)


def test_three_nn_fewer_than_three_known():
    d2, idx = oracle.three_nn(np.zeros((1, 1, 3), np.float32), np.ones((1, 2, 3), np.float32))
    assert np.isinf(d2[0, 0, 2]) and idx[0, 0].tolist() == [0, 1, 0]
    assert d2[0, 0, 0] == 3.0 and d2[0, 0, 1] == 3.0
