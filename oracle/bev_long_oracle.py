"""CPU oracle of BEV's crowd mode (BEV.process_long_image, simple_romp/bev/main.py:184-258, bev/split2process.py).
TEST INFRASTRUCTURE ONLY.

Builds on oracle/bev_oracle.py (model, SMPL-A/SMIL, projection, remove_outlier) and adds the crop plan, the conf-based
variant of suppressing_redundant_prediction_via_projection (bev/post_parser.py:167-198) and the merge of the per-crop
results.  Pinned by tests/golden/bev_long.npz, produced by the reference's own process_long_image
(tests/golden/make_golden_bev_long.py).
"""
from __future__ import annotations

import numpy as np
import torch

from . import romp_oracle as R
from .bev_oracle import bev_model, cam_to_trans, perspective_project, remove_outlier, smpla_forward

_t = R._t


def suppress_redundant(pj2d, cam, img_shape, thresh, conf_based=False, center_confs=None):
    """suppressing_redundant_prediction_via_projection, bev/post_parser.py:167-198 -> indices that survive.  Every pair
    closer than the threshold is judged at once; the loser is the smaller scale, or with ``conf_based`` (crowd mode,
    :191-193) the lower ``center_confs``.  The threshold is compared in fp32, like torch against a Python scalar."""
    n = len(pj2d)
    if n <= 1:
        return list(range(n))
    pj2d, cam = _t(pj2d), _t(cam)
    dist = torch.norm(pj2d.unsqueeze(1) - pj2d.unsqueeze(0), p=2, dim=-1).mean(-1)
    sc = cam[:, 0] * 2
    mx = torch.max(sc.unsqueeze(1).expand(n, n), sc.unsqueeze(0).expand(n, n))
    dn = dist / mx
    dn[torch.triu(torch.ones_like(dn), diagonal=1) < 0.5] = 10000.0
    i0, i1 = torch.where(dn < thresh * max(img_shape) / 640)
    key = _t(center_confs) if conf_based else sc
    removed = set(torch.where(key[i0] < key[i1], i0, i1).tolist())
    return [i for i in range(n) if i not in removed]


def long_image_plan(h, w, overlap=0.8):
    """padding_image_overlap + get_image_split_plan (split2process.py:6-39) -> (crop boxes int32 [S,2] = [left, right)
    in padded columns, pad).  The last crop starts at W-h but keeps the right edge of crop S-2 (:33-37), so it is
    narrower than h."""
    pad = int(h * overlap)                                     # :8
    W = w + 2 * pad
    S = int(np.ceil((W / h - 1) / (1 - overlap))) + 1          # :26-27
    step = (1 - overlap) * h
    boxes, right = [], None
    for i in range(S):
        if i == S - 1:
            left = W - h
        else:
            left = step * i
            right = left + h
        boxes.append([left, right])
    return np.array(boxes).astype(np.int32), pad


def _f32(x):
    return float(np.float32(x))


@torch.no_grad()
def bev_long_merge(per_crop, plan, pad, h, w, pack_a, pack_smil, nms_thresh=20, rel_scale_thresh=1.6, trace=None):
    """Steps 3-8 of process_long_image (bev/main.py:195-258) on the per-crop outputs of single_image_forward
    (``per_crop[c]``: None or a dict with cam, smpl_thetas, smpl_betas, params_pred, center_confs).

    Differs from the reference where it fails: an empty crop contributes nothing (the reference's croped_images /
    outputs_list indexing misaligns and raises as soon as a non-trailing crop is empty), and no survivor at all returns
    None (the reference raises KeyError).  Thresholds are compared in fp32 like torch against Python scalars.
    ``trace`` (a dict) receives the global stage's decisive quantities for the fixture generator.
    Returns the merged dict (crop order) or None."""
    S = len(plan)
    outs = []
    for c in range(S):
        o = per_crop[c]
        if o is None or len(o["cam"]) == 0:
            outs.append(None)
            continue
        o = {k: _t(o[k]).clone() for k in ("cam", "smpl_thetas", "smpl_betas", "params_pred", "center_confs")}
        o["verts"], o["joints"] = smpla_forward(pack_a, pack_smil, o["smpl_betas"], o["smpl_thetas"])      # :203
        outs.append(o)
    sel = lambda o, m: {k: v[m] for k, v in o.items()}
    cw = [int(plan[c, 1] - plan[c, 0]) for c in range(S)]
    ratio = [(plan[c, 1] - plan[c + 1, 0]) / h / 2 for c in range(S - 1)]                                  # :213-214
    for c in range(S):                                          # left-boundary exclusion, crop-pixel projection :209-218
        o = outs[c]
        if o is None:
            continue
        if c != S - 1:
            o = outs[c] = sel(o, ~(o["cam"][:, 2] > (1 - ratio[c] + 0)))                                     # split2process.py:43
        o["cam_trans"] = cam_to_trans(o["cam"])
        o["pj2d_org"] = R.to_org_image(perspective_project(o["joints"], o["cam_trans"]), [0, h, 0, cw[c], h, cw[c]])
    for c in range(1, S - 1):                                   # right-boundary exclusion of crop c+1; crop 1 never :221-226
        if outs[c + 1] is not None:
            o = outs[c + 1]
            outs[c + 1] = sel(o, ~(o["cam"][:, 2] < (ratio[c] - 1 - 0)))                                     # split2process.py:45
    for c in range(S):                                          # per-crop filters :228-232
        o = outs[c]
        if o is None:
            continue
        k = suppress_redundant(o["pj2d_org"], o["cam"], [h, cw[c]], nms_thresh, conf_based=True, center_confs=o["center_confs"])
        o = sel(o, k)
        outs[c] = sel(o, remove_outlier(o["cam_trans"], o["cam"], rel_scale_thresh, scale_thresh=1))
    merged = []
    for c in range(S):                                          # convert_crop_cam_params2full_image + collect :242-249
        o = outs[c]
        if o is None or len(o["cam"]) == 0:
            continue
        left, right = int(plan[c, 0]) - pad, int(plan[c, 1]) - pad
        cam = o["cam"] * _f32(max(right - left, h) / max(h, w))                                              # split2process.py:51-52
        cam[:, 2] = cam[:, 2] + _f32((left + right) / 2 / (w / 2) - 1)                                       # :56-57
        o["cam"] = cam
        o["crop_ids"] = torch.full((len(cam),), c, dtype=torch.int64)
        merged.append(o)
    if not merged:
        return None
    out = {k: torch.cat([o[k] for o in merged]) for k in merged[0] if k not in ("cam_trans", "pj2d_org")}
    out["cam_trans"] = cam_to_trans(out["cam"])                                                              # :253
    out["pj2d_org"] = R.to_org_image(perspective_project(out["joints"], out["cam_trans"]),
                                     [(w - h) // 2, w - (w - h) // 2, 0, w, h, w])                           # split2process.py:16-21
    k = suppress_redundant(out["pj2d_org"], out["cam"], (h, w, 3), nms_thresh, conf_based=True, center_confs=out["center_confs"])
    if trace is not None:
        pj, sc = out["pj2d_org"], out["cam"][:, 0] * 2
        dn = torch.norm(pj[:, None] - pj[None], dim=-1).mean(-1) / torch.maximum(sc[:, None], sc[None])
        trace.update(merged=out, dn_over_thr=dn / (nms_thresh * max(h, w) / 640), kept_after_nms=k)
    out = sel(out, k)                                                                                        # :255
    out = sel(out, remove_outlier(out["cam_trans"], out["cam"], rel_scale_thresh, scale_thresh=0.5))        # :256
    if len(out["cam"]) == 0:
        return None
    out["pred_batch_ids"] = torch.zeros(len(out["cam"]), dtype=torch.int64)
    return out


@torch.no_grad()
def bev_long_forward(sd, pack_a, pack_smil, image_bgr, thresh=0.08, nms_thresh=20, rel_scale_thresh=1.6, overlap=0.8,
                     center3d_override=None):
    """BEV.process_long_image (bev/main.py:184-258): pad, split, run BEVv1 + pack_params_dict on every crop
    (single_image_forward :123-135), then ``bev_long_merge``.  ``center3d_override`` [S,64,128,128] replaces each crop's
    3-D centre map.  Returns (merged dict or None, per-crop outputs)."""
    from .preproc_oracle import img_preprocess
    h, w = image_bgr.shape[:2]
    plan, pad = long_image_plan(h, w, overlap)
    padded = np.zeros((h, w + 2 * pad, 3), np.uint8)                                                         # split2process.py:6-13
    padded[:, pad:pad + w] = image_bgr
    per_crop = []
    for c, (left, right) in enumerate(plan):
        frame = img_preprocess(padded[:, left:right])[0]
        o = bev_model(sd, frame, thresh, None if center3d_override is None else _t(center3d_override)[c:c + 1])
        if o is None:
            per_crop.append(None)
            continue
        pk = R.pack_params(o["params_pred"], num_betas=11)
        per_crop.append({"cam": pk["cam"], "smpl_thetas": pk["smpl_thetas"], "smpl_betas": pk["smpl_betas"],
                         "params_pred": o["params_pred"], "center_confs": o["center_confs"]})
    return bev_long_merge(per_crop, plan, pad, h, w, pack_a, pack_smil, nms_thresh, rel_scale_thresh), per_crop
