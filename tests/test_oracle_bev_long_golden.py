"""Crowd mode of the BEV oracle (long_image_plan, bev_long_merge) against tests/golden/bev_long.npz, the outputs of the
reference's own BEV.process_long_image (tests/golden/make_golden_bev_long.py)."""
import os

import numpy as np
import pytest

from oracle import bev_oracle as B
from oracle import bev_long_oracle as BL
from romp_b200 import synth


@pytest.fixture(scope="module")
def z(golden_dir):
    return np.load(os.path.join(golden_dir, "bev_long.npz"))


def shapes(z):
    return [i for i in range(8) if f"s{i}_shape" in z.files]


def per_crop(z, p, S):
    """the fixture's raw single_image_forward outputs, one dict (or None) per crop"""
    crop = z[p + "raw_crop"]
    out = []
    for c in range(S):
        m = crop == c
        out.append(None if not m.any() else {"cam": z[p + "raw_cam"][m], "smpl_thetas": z[p + "raw_thetas"][m],
                                             "smpl_betas": z[p + "raw_betas"][m], "params_pred": z[p + "raw_params_pred"][m],
                                             "center_confs": z[p + "raw_conf"][m]})
    return out


def test_plan_matches_reference(z):
    sizes = []
    for i in shapes(z):
        p = f"s{i}_"
        h, w = z[p + "shape"].tolist()
        plan, pad = BL.long_image_plan(h, w)
        assert np.array_equal(plan, z[p + "plan"]) and pad == int(z[p + "pad"]), (h, w)
        assert plan[-1, 1] - plan[-1, 0] < h == plan[0, 1] - plan[0, 0]          # the narrow last crop
        sizes.append(len(plan))
    assert 14 in sizes and 24 in sizes and max(sizes) > 32


def test_merge_reproduces_reference_survivors(z):
    pa, ps = synth.smpl_pack(0, num_betas=11), synth.smpl_pack(1)
    for i in shapes(z):
        p = f"s{i}_"
        h, w = z[p + "shape"].tolist()
        plan, pad = BL.long_image_plan(h, w)
        out = BL.bev_long_merge(per_crop(z, p, len(plan)), plan, pad, h, w, pa, ps)
        surv = z[p + "survivors"]
        assert np.array_equal(out["params_pred"].numpy(), z[p + "raw_params_pred"][surv]), (h, w)     # same people, same order
        assert np.array_equal(out["center_confs"].numpy(), z[p + "center_confs"])
        for k in ("cam", "cam_trans", "smpl_thetas", "joints"):
            assert np.abs(out[k].numpy() - z[p + k]).max() < 1e-5, (h, w, k)
        assert np.abs(out["verts"][:, z["vsel"]].numpy() - z[p + "verts_sel"]).max() < 1e-5
        assert np.abs(out["pj2d_org"].numpy() - z[p + "pj2d_org"]).max() < 2e-2          # pixels of a >= 1024 wide image
        assert not out["pred_batch_ids"].any()


def test_fixture_exercises_every_filter(z):
    """512x1024: boundary exclusions, crop 1's missing left test, per-crop and global duplicates and outliers, a baby"""
    p = "s0_"
    assert z[p + "shape"].tolist() == [512, 1024]
    crop, surv = z[p + "raw_crop"], set(z[p + "survivors"].tolist())
    dropped = crop[[r for r in range(len(crop)) if r not in surv]].tolist()
    assert sorted(set(dropped)) == [0, 2, 4, 6, 8, 9]                   # left, right, global dup, crop outlier, crop dup, global outlier
    assert (z[p + "raw_betas"][sorted(surv), 10] > 0.8).any()
    assert (z[p + "raw_betas"][:, 10] > 0.8).sum() >= 2


def test_empty_crops_contribute_nothing(z):
    """The reference raises on an empty non-trailing crop; here the crop is skipped and nobody else changes."""
    pa, ps = synth.smpl_pack(0, num_betas=11), synth.smpl_pack(1)
    p = "s0_"
    h, w = z[p + "shape"].tolist()
    plan, pad = BL.long_image_plan(h, w)
    pc = per_crop(z, p, len(plan))
    pc[10] = None
    out = BL.bev_long_merge(pc, plan, pad, h, w, pa, ps)
    surv = [r for r in z[p + "survivors"] if z[p + "raw_crop"][r] != 10]
    assert np.array_equal(out["params_pred"].numpy(), z[p + "raw_params_pred"][surv])
    assert BL.bev_long_merge([None] * len(plan), plan, pad, h, w, pa, ps) is None
