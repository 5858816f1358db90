"""BEV crowd mode on the GPU (BEV.process_long_image, all through the C ABI): batched crop preprocessing, the per-crop
and global post stages against the reference's own results (tests/golden/bev_long.npz), end to end, and edge cases."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

from oracle import bev_oracle as B
from oracle import bev_long_oracle as BL
from oracle import preproc_oracle as P
from oracle import romp_oracle as O
from romp_b200 import _lib, synth
from romp_b200.bev import BEV, bev_settings

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
from make_golden_bev_long import SHAPES  # noqa: E402

pytestmark = pytest.mark.gpu
P_ = lambda t: C.c_void_p(t.data_ptr())


@pytest.fixture(scope="module")
def z(golden_dir):
    return np.load(os.path.join(golden_dir, "bev_long.npz"))


@pytest.fixture(scope="module")
def packs():
    return synth.bev_crowd_state_dict(0), synth.smpl_pack(0, num_betas=11), synth.smpl_pack(1)


def make(packs, precision="fp32", max_batch=32, extra=()):
    s = bev_settings(["--precision", precision, "--max_batch", str(max_batch), *extra])
    return BEV(s, state_dict=packs[0], smpla_pack=packs[1], smil_pack=packs[2])


def shape_index(z, shape):
    return next(i for i in range(8) if f"s{i}_shape" in z.files and tuple(z[f"s{i}_shape"].tolist()) == shape)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("h,w", [(512, 1024), (512, 2048), (437, 1311), (300, 2100), (31, 97)])
def test_crop_preprocess_bit_exact(h, w):
    lib = _lib.load()
    img = np.random.RandomState(h + w).randint(0, 256, (h, w, 3)).astype(np.uint8)
    plan, pad = BL.long_image_plan(h, w)
    S = len(plan)
    d = torch.from_numpy(img).cuda()
    pd = torch.from_numpy(plan.reshape(-1).copy()).cuda()
    out = torch.full((S, 512, 512, 3), 7, dtype=torch.uint8, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.b200romp_preprocess_crops_bgr(P_(d), h, w, 3 * w, pad, P_(pd), 0, S, 512, P_(out), st))
    part = torch.zeros((3, 512, 512, 3), dtype=torch.uint8, device="cuda")      # a later chunk: crops 2..4
    _lib.check(lib.b200romp_preprocess_crops_bgr(P_(d), h, w, 3 * w, pad, P_(pd), 2, 3, 512, P_(part), st))
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    padded = np.zeros((h, w + 2 * pad, 3), np.uint8)
    padded[:, pad:pad + w] = img
    for c, (l, r) in enumerate(plan):
        assert np.array_equal(got[c], P.img_preprocess(padded[:, l:r])[0][0]), f"crop {c} of {S}"
    assert np.array_equal(part.cpu().numpy(), got[2:5])


# ---------------------------------------------------------------------------------------------------------------------
def fill_raw(m, z, p, rows, batch_ids):
    """raw per-crop outputs of the reference (single_image_forward) written into the post stage's input buffers"""
    b, n = m.buf, len(rows)
    t = lambda k: torch.from_numpy(np.ascontiguousarray(z[p + k][rows])).cuda()
    b["thetas"][:n] = t("raw_thetas"); b["betas"][:n] = t("raw_betas"); b["cam"][:n] = t("raw_cam")
    b["params_pred"][:n] = t("raw_params_pred"); b["conf"][:n] = t("raw_conf")
    b["cam_trans"][:n] = B.cam_to_trans(torch.from_numpy(z[p + "raw_cam"][rows])).cuda()
    b["batch_ids"][:n] = torch.as_tensor(batch_ids, dtype=torch.int64).cuda()
    b["count"][0] = n


@pytest.mark.parametrize("shape", list(SHAPES))
def test_long_post_stage_golden(packs, z, shape):
    """SMPL-A/SMIL, boundary exclusion, per-crop filters, cam conversion, merge and the global filters on the fixture's
    raw per-crop outputs, crops in chunks of 16: the reference's survivors in its order."""
    p = f"s{shape_index(z, shape)}_"
    h, w = shape
    plan, pad = BL.long_image_plan(h, w)
    S, chunk = len(plan), 16
    m = make(packs, "fp32", chunk)
    m._long_alloc(S * 64)
    crop = z[p + "raw_crop"]
    with torch.cuda.stream(m.stream):
        m._long_begin(plan)
        for c0 in range(0, S, chunk):
            nb = min(chunk, S - c0)
            rows = np.flatnonzero((crop >= c0) & (crop < c0 + nb))
            fill_raw(m, z, p, rows, crop[rows] - c0)
            m._long_chunk(plan, pad, c0, nb, h, w)
        m._long_finish(h, w)
        out = m._long_collect()
    surv = z[p + "survivors"]
    assert np.array_equal(out["params_pred"], z[p + "raw_params_pred"][surv])
    assert np.array_equal(out["center_confs"], z[p + "center_confs"])
    assert np.abs(out["cam"] - z[p + "cam"]).max() < 1e-6
    assert np.abs(out["cam_trans"] - z[p + "cam_trans"]).max() < 1e-4 * np.abs(z[p + "cam_trans"]).max()
    assert np.abs(out["verts"][:, z["vsel"]] - z[p + "verts_sel"]).max() < 1e-4
    assert np.abs(out["joints"] - z[p + "joints"]).max() < 1e-4
    assert np.abs(out["pj2d_org"] - z[p + "pj2d_org"]).max() < 5e-2
    assert np.array_equal(out["smpl_thetas"], z[p + "smpl_thetas"]) and not out["pred_batch_ids"].any()


# ---------------------------------------------------------------------------------------------------------------------
def planted(z, shape):
    h, w = shape
    S = len(BL.long_image_plan(h, w)[0])
    return synth.synthetic_wide_image(h, w, int(z["image_seed"])), synth.bev_planted_crops(S, SHAPES[shape], int(z["volume_seed"]))


def oracle_on_gpu_crops(m, packs, shape):
    """the oracle's merge applied to the GPU's own per-crop outputs (max_batch >= S: one chunk, self.buf holds every crop)"""
    h, w = shape
    plan, pad = BL.long_image_plan(h, w)
    b = m.buf
    n = int(b["count"].item())
    pp, bid, conf = b["params_pred"][:n].cpu(), b["batch_ids"][:n].cpu().numpy(), b["conf"][:n].cpu()
    pk = O.pack_params(pp, num_betas=11)
    pc = [None if not (bid == c).any() else
          {"cam": pk["cam"][bid == c], "smpl_thetas": pk["smpl_thetas"][bid == c], "smpl_betas": pk["smpl_betas"][bid == c],
           "params_pred": pp[bid == c], "center_confs": conf[bid == c]} for c in range(len(plan))]
    return BL.bev_long_merge(pc, plan, pad, h, w, packs[1], packs[2])


def test_end_to_end_fp32_matches_reference(packs, z):
    shape = (512, 1024)
    p = f"s{shape_index(z, shape)}_"
    img, vol = planted(z, shape)
    m = make(packs, "fp32", 32)
    out = m.process_long_image(img, center3d_override=torch.from_numpy(vol).cuda())
    assert set(out) == {"smpl_thetas", "smpl_betas", "cam", "cam_trans", "params_pred", "center_confs", "pred_batch_ids",
                        "verts", "joints", "pj2d_org"}
    assert np.array_equal(out["center_confs"], z[p + "center_confs"])            # same people, same order
    assert np.abs(out["cam"] - z[p + "cam"]).max() < 2e-3
    assert np.abs(out["params_pred"] - z[p + "raw_params_pred"][z[p + "survivors"]]).max() < 5e-3


def test_end_to_end_bf16_matches_oracle_on_own_crops(packs, z):
    shape = (512, 1024)
    img, vol = planted(z, shape)
    m = make(packs, "bf16", 32)
    out = m.process_long_image(torch.from_numpy(img).cuda(), center3d_override=torch.from_numpy(vol).cuda())
    ref = oracle_on_gpu_crops(m, packs, shape)
    assert np.array_equal(out["params_pred"], ref["params_pred"].numpy())
    assert np.abs(out["cam"] - ref["cam"].numpy()).max() < 1e-5
    assert np.abs(out["verts"] - ref["verts"].numpy()).max() < 1e-4 and np.abs(out["joints"] - ref["joints"].numpy()).max() < 1e-4


def test_chunking_is_invisible(packs, z):
    """24 crops through max_batch 8 (three chunks) and 64 (one chunk): every conv tile lies within one frame and every
    later stage is per person or per crop, so the outputs are bit-identical."""
    img, vol = planted(z, (512, 2048))
    vol = torch.from_numpy(vol).cuda()
    a = make(packs, "bf16", 8).process_long_image(img, center3d_override=vol)
    b = make(packs, "bf16", 64).process_long_image(img, center3d_override=vol)
    assert set(a) == set(b) and len(a["cam"]) == 24
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_empty_middle_crop_and_empty_image(packs, z):
    shape = (512, 1024)
    img, vol = planted(z, shape)
    vol[5] = 0.0                                     # crop 5 detects nobody (the reference raises here)
    m = make(packs, "fp32", 32)
    out = m.process_long_image(img, center3d_override=torch.from_numpy(vol).cuda())
    ref = oracle_on_gpu_crops(m, packs, shape)
    assert (m.buf["batch_ids"][: int(m.buf["count"].item())] != 5).all()
    assert np.array_equal(out["params_pred"], ref["params_pred"].numpy())
    assert np.abs(out["cam"] - ref["cam"].numpy()).max() < 1e-5
    assert m.process_long_image(img, center3d_override=torch.zeros(14, 64, 128, 128).cuda()) is None


def test_global_merge_over_256_people(packs):
    shape = (512, 2048)
    h, w = shape
    S = len(BL.long_image_plan(h, w)[0])
    cells = [(c, 28 + (k % 8), 16 + 24 * (k // 4), 40 + 16 * (k % 4), 0.3 + 0.02 * k) for c in range(S) for k in range(20)]
    vol = synth.bev_planted_crops(S, cells, 1)
    m = make(packs, "fp32", 32)
    out = m.process_long_image(synth.synthetic_wide_image(h, w, 3), center3d_override=torch.from_numpy(vol).cuda())
    assert int(m._long["merged"].item()) > 256
    ref = oracle_on_gpu_crops(m, packs, shape)
    assert np.array_equal(out["params_pred"], ref["params_pred"].numpy())
    assert np.abs(out["cam"] - ref["cam"].numpy()).max() < 1e-5


def test_crowd_off_takes_the_normal_path(packs, monkeypatch):
    m = make(packs, "fp32", 1, extra=("--crowd",))
    monkeypatch.setattr(BEV, "process_long_image", lambda *a, **k: (_ for _ in ()).throw(AssertionError("crowd mode used")))
    img = synth.synthetic_wide_image(256, 640, 1)
    from romp_b200.main import img_preprocess
    frame, pad = img_preprocess(img)
    ref = m.forward_batch(torch.from_numpy(frame), offsets=pad, img_max_side=640.0)
    out = m(img)
    assert (out is None) == (ref is None)
    if out is not None:
        for k in out:
            assert np.array_equal(out[k], ref[k]), k


def test_unsupported_options_raise(packs):
    img = synth.synthetic_wide_image(128, 512, 2)
    m = make(packs, "fp32", 4)
    with pytest.raises(NotImplementedError, match="render"):
        m.process_long_image(img, show_patch_results=True)
    m2 = make(packs, "fp32", 4, extra=("--calc_smpl",))
    with pytest.raises(ValueError, match="calc_smpl"):
        m2(img)
