"""Golden fixture of BEV's crowd mode (bev/main.py:184-258, bev/split2process.py), produced by calling the REFERENCE's
own ``BEV.process_long_image`` unbound on a stub ``self`` (build container only):

    python tests/golden/make_golden_bev_long.py

The stub carries the reference BEVv1 on the synthetic BEV weights (``synth.bev_crowd_state_dict``: a person's cam is
close to the 3-D coordinate of its planted cell, and some people are babies), whose 3-D centre-map parse is replaced by the planted volume of the
current crop, the reference SMPLA_parser on the synthetic packs, and the crowd settings.  ``single_image_forward`` is
wrapped to record each crop's raw outputs.  OpenCV runs with IPP off (DESIGN 4.8).  Importing bev.main needs a stub
``vis_human`` and a no-op ``romp.utils.download_model`` (its module-level ``bev_settings([])`` asks for the missing
checkpoint); the real download function is never called.  Only outputs are stored, in tests/golden/bev_long.npz.
"""
import importlib
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)

IMAGE_SEED = 21
VOLUME_SEED = 4
N_VSEL = 64
# (h, w) -> planted cells (crop, z, y, x, centre value).  With the damped cam offsets a cell (z, y, x) gives
# cam ~ (anchor[z], y/64-1, x/64-1); the boundary tests compare cam_x with +-0.6 (overlap 0.8).
SHAPES = {
    (512, 1024): [
        (0, 27, 64, 60, 0.90),                          # kept
        (0, 27, 64, 116, 0.70),                         # left exclusion (cam_x ~ 0.81 > 0.6)
        (1, 27, 40, 12, 0.80),                          # crop 1 is never tested on its left edge: kept
        (1, 30, 80, 70, 0.60),
        (2, 30, 90, 10, 0.75),                          # right exclusion (cam_x ~ -0.84 < -0.6)
        (2, 32, 60, 64, 0.50),
        (3, 33, 60, 64, 0.85), (3, 31, 60, 67, 0.55),
        (4, 35, 30, 80, 0.65), (5, 35, 30, 54, 0.66),   # one person seen by crops 4 and 5 (crops are 25.6 cells apart)
        (6, 60, 100, 90, 0.45), (6, 28, 50, 40, 0.62), (6, 29, 60, 60, 0.61), (6, 30, 70, 80, 0.64),   # crop outlier
        (7, 3, 64, 64, 0.55),                           # very close person
        (8, 30, 64, 64, 0.85), (8, 28, 64, 67, 0.55),   # per-crop duplicate: the higher confidence has the smaller scale
        (9, 50, 64, 64, 0.52),                          # alone in its crop, far behind everybody: global outlier
        (10, 29, 64, 64, 0.57),
        (11, 29, 64, 64, 0.58),
        (12, 31, 64, 64, 0.59),
        (13, 33, 64, 64, 0.63),
    ],
    (512, 2048): [(c, 26 + c % 8, 64, 64, 0.5 + 0.01 * c) for c in range(24)],
    (437, 1311): [(c, 27 + c % 6, 64, 64, 0.5 + 0.01 * c) for c in range(19)],
    (300, 2100): [(c, 27 + c % 7, 64, 64, 0.4 + 0.01 * c) for c in range(40)],
}


def load_bev_main():
    from make_golden import load_reference
    load_reference()
    U = importlib.import_module("romp.utils")
    sys.modules["vis_human"] = types.SimpleNamespace(setup_renderer=None, rendering_romp_bev_results=None)
    U.download_model = lambda *a, **k: None            # before the import: bev_settings([]) runs at module level
    return importlib.import_module("bev.main"), importlib.import_module("bev.model"), importlib.import_module("bev.post_parser")


def run_reference(BM, M, PP, shape, cells, sd, parser):
    from romp_b200 import synth
    h, w = shape
    image = synth.synthetic_wide_image(h, w, IMAGE_SEED)
    model = M.BEVv1(center_thresh=0.08).eval()
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=False)
    S = 1 + max(c for c, *_ in cells)
    vol = synth.bev_planted_crops(S, cells, VOLUME_SEED)
    state = {"crop": 0}
    parse = model.centermap_parser.parse_3dcentermap

    def planted_parse(_center_maps_3d):
        c = state["crop"]
        state["crop"] += 1
        return parse(torch.from_numpy(vol[c:c + 1]))

    model.centermap_parser.parse_3dcentermap = planted_parse
    raw = []

    class Stub:
        settings = types.SimpleNamespace(overlap_ratio=0.8, center_thresh=0.08, nms_thresh=20, relative_scale_thresh=1.6,
                                         render_mesh=False, show_patch_results=False, renderer="sim3dr")
        result_keys = ["smpl_thetas", "smpl_betas", "cam", "cam_trans", "params_pred", "center_confs", "pred_batch_ids"]
        tdevice = torch.device("cpu")

        def __init__(self):
            self.model, self.smpl_parser = model, parser

        def single_image_forward(self, image):
            out, pad_info = BM.BEV.single_image_forward(self, image)
            raw.append(None if out is None else {k: v.clone() for k, v in out.items()})
            return out, pad_info

    with torch.no_grad():
        out = BM.BEV.process_long_image(Stub(), image, show_patch_results=False)
    assert state["crop"] == S == len(raw)
    return image, out, raw


def margins(raw, shape):
    """Print every decisive quantity of the crowd-mode filters next to its threshold (oracle restatement on the
    reference's raw per-crop outputs)."""
    from oracle import bev_oracle as B
    from oracle import bev_long_oracle as BL
    from romp_b200 import synth
    h, w = shape
    plan, pad = BL.long_image_plan(h, w)
    pa, ps = synth.smpl_pack(0, num_betas=11), synth.smpl_pack(1)
    S = len(plan)
    ratio = [(plan[c, 1] - plan[c + 1, 0]) / h / 2 for c in range(S - 1)]
    worst = []
    for c, o in enumerate(raw):
        x = o["cam"][:, 2].numpy()
        if c != S - 1:
            worst.append(np.abs(x - (1 - ratio[c])).min())
        if c >= 2:
            worst.append(np.abs(x - (ratio[c - 1] - 1)).min())
        cw = plan[c, 1] - plan[c, 0]
        if len(x) > 1:
            v, j = B.smpla_forward(pa, ps, o["smpl_betas"], o["smpl_thetas"])
            pj = B.R.to_org_image(B.perspective_project(j, B.cam_to_trans(o["cam"])), [0, h, 0, cw, h, cw])
            dist = torch.norm(pj[:, None] - pj[None], dim=-1).mean(-1)
            sc = o["cam"][:, 0] * 2
            dn = dist / torch.maximum(sc[:, None], sc[None])
            iu = np.triu_indices(len(x), 1)
            thr = 20 * max(h, cw) / 640
            print(f"  crop {c}: cam_x {np.round(x, 3).tolist()} scale {np.round(o['cam'][:, 0].numpy(), 3).tolist()} "
                  f"pair dn/thr {np.round(dn.numpy()[iu] / thr, 3).tolist()}")
            worst.append(np.abs(dn.numpy()[iu] - thr).min() / thr)
        else:
            print(f"  crop {c}: cam_x {np.round(x, 3).tolist()} scale {np.round(o['cam'][:, 0].numpy(), 3).tolist()}")
    print(f"  smallest boundary / per-crop NMS margin {min(worst):.4f}")
    print("  betas[:, 10] (baby > 0.8):", [np.round(o["smpl_betas"][:, 10].numpy(), 3).tolist() for o in raw])
    tr = {}
    BL.bev_long_merge(raw, plan, pad, h, w, pa, ps, trace=tr)
    dn = tr["dn_over_thr"].numpy()
    iu = np.triu_indices(len(dn), 1)
    crops = tr["merged"]["crop_ids"].numpy()
    close = [(int(crops[i]), int(crops[j]), round(float(dn[i, j]), 3)) for i, j in zip(*iu) if dn[i, j] < 2]
    print(f"  global pairs (crop i, crop j, dn/thr) below 2: {close};  smallest |dn/thr - 1| {np.abs(dn[iu] - 1).min():.4f}")
    t = tr["merged"]["cam_trans"][tr["kept_after_nms"]]
    n = len(t)
    d = torch.sort(torch.norm(t[:, None] - t[None], dim=-1)).values[:, 1:-1].mean(1)
    rel = d / ((d.sum() - d) / (n - 1))
    print("  global rel / 1.6:", np.round(rel.numpy() / 1.6, 3).tolist())
    print("  global scales / 0.5:", np.round(tr["merged"]["cam"][tr["kept_after_nms"], 0].numpy() / 0.5, 3).tolist())


def main():
    from romp_b200 import synth
    import cv2
    cv2.ipp.setUseIPP(False)
    torch.set_num_threads(os.cpu_count())
    BM, M, PP = load_bev_main()
    sd = synth.bev_crowd_state_dict(0)
    tt = lambda d: {k: torch.from_numpy(np.asarray(v)) for k, v in d.items()}
    with tempfile.TemporaryDirectory() as d:
        torch.save(tt(synth.smpl_pack(0, num_betas=11)), os.path.join(d, "a.pth"))
        torch.save(tt(synth.smpl_pack(1)), os.path.join(d, "s.pth"))
        parser = PP.SMPLA_parser(os.path.join(d, "a.pth"), os.path.join(d, "s.pth"))
    only = [tuple(int(v) for v in a.split("x")) for a in sys.argv[1:]]
    rs = np.random.RandomState(5)
    vsel = np.sort(rs.choice(6890, N_VSEL, replace=False))
    store = {"image_seed": IMAGE_SEED, "volume_seed": VOLUME_SEED, "vsel": vsel}
    for si, (shape, cells) in enumerate(SHAPES.items()):
        if only and shape not in only:
            continue
        h, w = shape
        image, out, raw = run_reference(BM, M, PP, shape, cells, sd, parser)
        from oracle import bev_oracle as B
        from oracle import bev_long_oracle as BL
        plan, pad = BL.long_image_plan(h, w)
        print(f"{h}x{w}: {len(plan)} crops, {sum(len(o['cam']) for o in raw)} detections, {len(out['cam'])} survivors")
        margins(raw, shape)
        cat = lambda k: torch.cat([o[k] for o in raw]).numpy()
        rp = cat("params_pred")
        surv = [int(np.flatnonzero((rp == p).all(1))[0]) for p in out["params_pred"].numpy()]
        print("  survivors (raw rows):", surv)
        p = f"s{si}_"
        store.update({p + "shape": np.array(shape), p + "cells": np.array(cells, np.float32),
                      p + "raw_crop": np.concatenate([np.full(len(o["cam"]), c) for c, o in enumerate(raw)]),
                      p + "raw_cam": cat("cam"), p + "raw_thetas": cat("smpl_thetas"), p + "raw_betas": cat("smpl_betas"),
                      p + "raw_params_pred": rp, p + "raw_conf": cat("center_confs"), p + "survivors": np.array(surv),
                      p + "cam": out["cam"].numpy(), p + "cam_trans": out["cam_trans"].numpy(),
                      p + "center_confs": out["center_confs"].numpy(), p + "smpl_thetas": out["smpl_thetas"].numpy(),
                      p + "joints": out["joints"].numpy(), p + "pj2d_org": out["pj2d_org"].numpy(),
                      p + "verts_sel": out["verts"][:, vsel].numpy(), p + "pred_batch_ids": out["pred_batch_ids"].numpy()})
        # the reference's plan, as returned by its own split2process functions
        SP = importlib.import_module("bev.split2process")
        padded, _, pad_ref = SP.padding_image_overlap(image, overlap_ratio=0.8)
        store[p + "plan"] = SP.get_image_split_plan(padded, overlap_ratio=0.8)[:, :2]
        store[p + "pad"] = np.array(pad_ref)
    if not only:
        path = os.path.join(HERE, "bev_long.npz")
        np.savez_compressed(path, **store)
        print(path, os.path.getsize(path))


if __name__ == "__main__":
    main()
