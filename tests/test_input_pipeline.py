"""Input pipeline (SURVEY row N4): oracle vs the reference's own outputs (CPU), host RNG restatement vs the reference's
draw order (CPU), device kernels vs golden / oracle (GPU)."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import cases  # noqa: E402
import cases_input  # noqa: E402
from oracle import input_pipeline as oi  # noqa: E402
from spacap3d_b200 import input_pipeline as ip  # noqa: E402

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "input_ref.npz"))
NAMES = list(cases_input.CASES.keys())


def _draw(c):
    return ip.draw_item(np.random.RandomState(c["seed"]), c["verts"].shape[0], c["P"], c["augment"])


def test_oracle_floor_height_equals_numpy_percentile():
    for i, z in enumerate(cases_input.percentile_inputs()):
        assert oi.floor_height(z) == GOLD["percentile/%d" % i], i


@pytest.mark.parametrize("name", NAMES)
def test_draw_item_follows_reference_rng_order(name):
    c = cases_input.case(name)
    choices, aug = _draw(c)
    np.testing.assert_array_equal(choices, GOLD[name + "/choices"])
    assert (aug is not None) == c["augment"]


@pytest.mark.parametrize("name", NAMES)
def test_oracle_equals_reference(name):
    c = cases_input.case(name)
    choices, aug = _draw(c)
    fh = oi.floor_height(c["verts"][:, 2]) if c["use_height"] else None
    if fh is not None:
        assert fh == GOLD[name + "/floor_height"]
    pc = oi.prepare_point_cloud(c["verts"], choices, c["multiview"] if c["use_multiview"] else None, fh, aug,
                                c["use_color"], c["use_normal"])
    assert cases.sha(pc) == str(GOLD[name + "/point_clouds"])
    votes, mask = oi.vote_labels(pc, c["inst"][choices], c["sem"][choices])
    np.testing.assert_array_equal(votes, GOLD[name + "/vote_label"])
    np.testing.assert_array_equal(mask, GOLD[name + "/vote_label_mask"])
    boxes = np.zeros((ip.MAX_NUM_OBJ, 6))
    nb = min(c["bboxes"].shape[0], ip.MAX_NUM_OBJ)
    boxes[:nb] = c["bboxes"][:ip.MAX_NUM_OBJ, 0:6]
    if aug is not None:
        boxes = oi.augment_boxes(boxes, aug)
    np.testing.assert_array_equal(boxes, GOLD[name + "/target_bboxes"])
    assert nb == GOLD[name + "/num_bbox"]


def test_sem_mask_matches_nyu40ids():
    m = ip.sem_mask_of()
    assert [i for i in range(64) if (m >> i) & 1] == list(oi.NYU40IDS)


# ---- device ------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_device_floor_height_equals_numpy():
    from spacap3d_b200 import _ext
    for i, z in enumerate(cases_input.percentile_inputs()):
        tab = np.zeros((z.shape[0], 3), np.float32)
        tab[:, 2] = z
        got = _ext.scene_floor_height(torch.from_numpy(tab).cuda()).cpu().numpy()[0]
        assert got == GOLD["percentile/%d" % i], (i, got, GOLD["percentile/%d" % i])


def _store(cs):
    st = ip.DeviceSceneStore("cuda")
    for i, c in enumerate(cs):
        st.add_scene("s%d" % i, c["verts"], c["inst"], c["sem"], c["bboxes"], c["multiview"])
    return st.finalize()


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_device_batch_equals_reference(name):
    """Two items of the same scene with different draws through DeviceSceneStore.make_batch == the reference's
    __getitem__ statements (golden) for item 0 and the numpy oracle for item 1."""
    c = cases_input.case(name)
    filler = cases_input.case("replace_eval")                                # the scene is NOT first in the table
    if c["use_multiview"]:
        filler["multiview"] = np.ones((filler["verts"].shape[0], 128), np.float32)
    store = _store([filler, c])
    d0 = _draw(c)
    d1 = ip.draw_item(np.random.RandomState(c["seed"] + 100), c["verts"].shape[0], c["P"], c["augment"])
    out = store.make_batch(["s1", "s1"], [d0, d1], use_color=c["use_color"], use_normal=c["use_normal"],
                           use_multiview=c["use_multiview"], use_height=c["use_height"])
    assert int(out["_instance_overflow"].item()) == 0
    pc = out["point_clouds"].cpu().numpy()
    # fp64 rotation products rounded to fp32: identical unless BLAS' dgemm and the kernel's fma chain round an fp64
    # intermediate differently AND that flips the fp32 rounding; never observed -> exact comparison
    assert cases.sha(pc[0]) == str(GOLD[name + "/point_clouds"])             # stored as a digest of the exact bytes
    np.testing.assert_array_equal(out["vote_label"][0].cpu().numpy(), GOLD[name + "/vote_label"])
    np.testing.assert_array_equal(out["vote_label_mask"][0].cpu().numpy(), GOLD[name + "/vote_label_mask"])
    np.testing.assert_allclose(out["target_bboxes"][0].cpu().numpy(), GOLD[name + "/target_bboxes"], rtol=1e-13,
                               atol=1e-15)
    np.testing.assert_array_equal(out["center_label"][0].cpu().numpy(), GOLD[name + "/center_label"])
    assert int(out["num_bbox"][0]) == int(GOLD[name + "/num_bbox"])
    # item 1 against the oracle
    fh = oi.floor_height(c["verts"][:, 2]) if c["use_height"] else None
    want = oi.prepare_point_cloud(c["verts"], d1[0], c["multiview"] if c["use_multiview"] else None, fh, d1[1],
                                  c["use_color"], c["use_normal"])
    np.testing.assert_array_equal(pc[1], want)
    votes, mask = oi.vote_labels(want, c["inst"][d1[0]], c["sem"][d1[0]])
    np.testing.assert_array_equal(out["vote_label"][1].cpu().numpy(), votes)
    np.testing.assert_array_equal(out["vote_label_mask"][1].cpu().numpy(), mask)


@pytest.mark.gpu
def test_device_batch_full_size_properties():
    """BASELINE size (8 items x 40 k of 50 k vertices, 135 channels): oracle comparison on one item, and
    size-independent properties on all: un-augmented xyz are exact row copies, votes point at the instance centre."""
    v, inst, sem, bb, mv = cases_input.make_scene(50000, 60, 77, multiview=True)
    st = ip.DeviceSceneStore("cuda")
    st.add_scene("big", v, inst, sem, bb, mv)
    st.finalize()
    draws = [ip.draw_item(np.random.RandomState(s), 50000, 40000, True) for s in range(8)]
    out = st.make_batch(["big"] * 8, draws, use_color=True, use_normal=True, use_multiview=True, use_height=True)
    pc = out["point_clouds"].cpu().numpy()
    assert pc.shape == (8, 40000, 3 + 3 + 3 + 128 + 1)
    fh = oi.floor_height(v[:, 2])
    want = oi.prepare_point_cloud(v, draws[3][0], mv, fh, draws[3][1], True, True)
    np.testing.assert_array_equal(pc[3], want)
    for b in range(8):
        ch = draws[b][0]
        np.testing.assert_array_equal(pc[b, :, 9:137], mv[ch])               # multiview rows are pure gathers
        np.testing.assert_array_equal(pc[b, :, 6:9], v[ch, 6:9])
        np.testing.assert_array_equal(pc[b, :, 137], v[ch, 2] - fh)
    votes = out["vote_label"].cpu().numpy()
    mask = out["vote_label_mask"].cpu().numpy()
    for b in (0, 7):
        il = inst[draws[b][0]]
        for i in np.unique(il)[:10]:
            ind = np.where(il == i)[0]
            if mask[b, ind[0]]:
                ctr = pc[b, ind, :3] + votes[b, ind, :3]                      # x + (centre - x) = centre for every member
                assert np.abs(ctr - ctr[0]).max() < 1e-5
            else:
                assert not votes[b, ind].any()
    eval_out = st.make_batch(["big"], [ip.draw_item(np.random.RandomState(5), 50000, 40000, False)], use_height=True,
                             want_votes=False)
    np.testing.assert_array_equal(eval_out["point_clouds"][0, :, :3].cpu().numpy(),
                                  v[eval_out["choices"][0].cpu().numpy(), :3])


@pytest.mark.gpu
def test_device_sampler_draws_valid_subsets():
    ch = ip.draw_batch_device([5000, 1500, 3000], 2000, generator=torch.Generator("cuda").manual_seed(1)).cpu().numpy()
    assert ch.shape == (3, 2000) and ch.dtype == np.int32
    for row, m in zip(ch, (5000, 1500, 3000)):
        assert row.min() >= 0 and row.max() < m
    assert len(np.unique(ch[0])) == 2000 and len(np.unique(ch[2])) == 2000      # without replacement when M >= P
    assert len(np.unique(ch[1])) < 1500                                        # with replacement when M < P


def test_store_rejects_missing_multiview():
    st = ip.DeviceSceneStore("cpu")
    st.multiview = None
    with pytest.raises(RuntimeError, match="multiview"):
        st.make_batch([], [], use_multiview=True)


@pytest.mark.gpu
def test_store_feeds_detector():
    """Row N4 -> the hot path: a batch assembled on the device goes straight into the detector (same layout as the
    reference's data_dict['point_clouds']); the device sampler and the numpy-stream sampler both work."""
    from spacap3d_b200.detector import VoteNetDetector
    st = ip.DeviceSceneStore("cuda")
    for i in range(2):
        v, inst, sem, bb, _ = cases_input.make_scene(24000, 30, 300 + i)
        st.add_scene("s%d" % i, v, inst, sem, bb)
    st.finalize()
    torch.manual_seed(0)
    model = VoteNetDetector(input_feature_dim=1).cuda().eval()
    draws = [ip.draw_item(np.random.RandomState(s), 24000, 20000, True) for s in range(2)]
    dev_choices = ip.draw_batch_device([24000, 24000], 20000, generator=torch.Generator("cuda").manual_seed(3))
    for d in (draws, (dev_choices, np.stack([x[1] for x in draws]))):
        batch = st.make_batch(["s0", "s1"], d, use_height=True)
        assert batch["point_clouds"].shape == (2, 20000, 4)
        with torch.no_grad():
            out = model({"point_clouds": batch["point_clouds"]})
        assert out["bbox_corner"].shape == (2, 256, 8, 3) and torch.isfinite(out["center"]).all()
        assert batch["vote_label"].shape == (2, 20000, 9) and batch["vote_label_mask"].sum() > 0
