"""Drop-in call surface of ``simple_romp``'s BEV (bev/main.py) on the B200 hot path.

``bev_settings`` mirrors bev/main.py:27-87 (same flags and defaults, including the quirk that ``crowd`` defaults to
True and therefore overrides the thresholds with ``long_conf_dict``), ``BEV(settings)(image_bgr) -> dict | None``
mirrors bev/main.py:91-181: normal images, and with ``crowd`` images of aspect ratio >= 2 through the sliding-window
``process_long_image`` (bev/main.py:184-258); ``forward_batch`` is the batched entry point.
Per-frame semantics of the two post filters (bev/post_parser.py:167-222) are preserved by applying them per
``pred_batch_ids`` group on the device.  Python only allocates buffers and sequences library calls.
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
import os.path as osp
import sys

import numpy as np
import torch

from . import _lib, graph
from ._lib import BF16, F32, U8
from .main import MAX_PERSON, SMPLParser, _ptr, img_preprocess

conf_dict = {1: [0.25, 20, 2], 2: [0.1, 20, 1.6]}                    # bev/main.py:24-25
long_conf_dict = {1: [0.12, 20, 1.5, 0.46], 2: [0.08, 20, 1.6, 0.8]}
model_dict = {1: "BEV_ft_agora.pth", 2: "BEV.pth"}
N_PARAMS = 146                                                       # 3 cam + 22*6 + 11 betas, bev/model.py:116


def bev_settings(input_args=sys.argv[1:]):
    """Same flags/defaults as bev/main.py:27-87; no downloads, no prints."""
    model_id = 2
    home = osp.join(osp.expanduser("~"), ".romp")
    p = argparse.ArgumentParser(description="BEV (B200-native hot path)")
    p.add_argument("-m", "--mode", type=str, default="image")
    p.add_argument("--model_id", type=int, default=2)
    p.add_argument("-i", "--input", type=str, default=None)
    p.add_argument("-o", "--save_path", type=str, default=osp.join(osp.expanduser("~"), "BEV_results"))
    p.add_argument("--crowd", action="store_false")
    p.add_argument("--GPU", type=int, default=0)
    p.add_argument("--overlap_ratio", type=float, default=long_conf_dict[model_id][3])
    p.add_argument("--center_thresh", type=float, default=conf_dict[model_id][0])
    p.add_argument("--nms_thresh", type=float, default=conf_dict[model_id][1])
    p.add_argument("--relative_scale_thresh", type=float, default=conf_dict[model_id][2])
    p.add_argument("--show_largest", action="store_true")
    p.add_argument("--show_patch_results", action="store_true")
    p.add_argument("--calc_smpl", action="store_false")
    p.add_argument("--renderer", type=str, default="sim3dr")
    p.add_argument("--render_mesh", action="store_false")
    p.add_argument("--show", action="store_true")
    p.add_argument("--show_items", type=str, default="mesh,mesh_bird_view")
    p.add_argument("--save_video", action="store_true")
    p.add_argument("--frame_rate", type=int, default=24)
    p.add_argument("--smpl_path", type=str, default=osp.join(home, "SMPLA_NEUTRAL.pth"))
    p.add_argument("--smil_path", type=str, default=osp.join(home, "smil_packed_info.pth"))
    p.add_argument("--model_path", type=str, default=osp.join(home, model_dict[model_id]))
    p.add_argument("-t", "--temporal_optimize", action="store_true")
    p.add_argument("-sc", "--smooth_coeff", type=float, default=3.0)
    p.add_argument("--webcam_id", type=int, default=0)
    p.add_argument("--precision", type=str, default="bf16", choices=["bf16", "tf32", "fp32"])
    p.add_argument("--max_batch", type=int, default=32)
    args = p.parse_args(input_args)
    if args.model_id != 2:                                            # bev/main.py:59-63
        args.model_path = osp.join(home, model_dict[args.model_id])
        args.center_thresh, args.nms_thresh = conf_dict[args.model_id][0], conf_dict[args.model_id][1]
        args.relative_scale_thresh = conf_dict[model_id][2]
    if args.crowd:                                                    # :81-85 (crowd defaults to True)
        args.center_thresh, args.nms_thresh = long_conf_dict[args.model_id][0], long_conf_dict[args.model_id][1]
        args.relative_scale_thresh, args.overlap_ratio = long_conf_dict[model_id][2], long_conf_dict[args.model_id][3]
    return args


def long_image_plan(h, w, overlap):
    """padding_image_overlap + get_image_split_plan (bev/split2process.py:6-39) -> (int32 [S,2] crop columns [left, right)
    of the image padded by ``pad`` zero columns on each side, pad).  Every crop spans the full height h; the last one
    starts at W-h but keeps the right edge of crop S-2 (:33-37), so it is narrower than h."""
    pad = int(h * overlap)
    W = w + 2 * pad
    S = int(np.ceil((W / h - 1) / (1 - overlap))) + 1
    step = (1 - overlap) * h
    boxes, right = [], None
    for i in range(S):
        left = W - h if i == S - 1 else step * i
        if i != S - 1:
            right = left + h
        boxes.append([left, right])
    return np.array(boxes).astype(np.int32), pad


class BEV(torch.nn.Module):
    """``BEV(settings)(image_bgr)`` - the contract of simple_romp/bev/main.py:91-181 for normal images."""

    result_keys = ["smpl_thetas", "smpl_betas", "cam", "cam_trans", "params_pred", "center_confs", "pred_batch_ids"]   # :115

    def __init__(self, settings, state_dict=None, smpla_pack=None, smil_pack=None):
        super().__init__()
        self.settings = s = settings
        if not torch.cuda.is_available() or s.GPU < 0:
            raise RuntimeError("romp_b200.BEV needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        if getattr(s, "temporal_optimize", False) or getattr(s, "show", False) or getattr(s, "show_largest", False):
            raise NotImplementedError("temporal smoothing / display are outside the B200 hot path (SURVEY.md section 2)")
        # NB the reference renders by default (render_mesh is store_false, bev/main.py:44); rendering is out of scope and
        # simply not performed here.
        self.lib = _lib.load()
        self.device_index = int(s.GPU)
        self.tdevice = torch.device("cuda", self.device_index)
        torch.cuda.set_device(self.tdevice)
        self.precision = getattr(s, "precision", "bf16")
        self._staging = {}
        self.max_batch = B = int(getattr(s, "max_batch", 32))
        if state_dict is None:
            state_dict = torch.load(s.model_path, map_location="cpu")          # bev/main.py:101 (strict=False)
        self._sd = state_dict
        self._nets = {}
        self.stream = torch.cuda.Stream(device=self.tdevice)
        w = graph.bev_weights(state_dict)
        self._w_keep = w
        fp = C.POINTER(C.c_float)
        bw = _lib.BevWeights(*[w[k].ctypes.data_as(fp) for k in ("center_ref", "cam_ref", "coordmap", "anchors", "embed",
                                                                   "w0", "b0", "w1", "b1", "w2", "b2")])
        self.h = self.lib.b200romp_bev_create(self.device_index, C.byref(bw))
        if not self.h:
            raise RuntimeError("b200romp_bev_create: " + self.lib.b200romp_last_error().decode())
        self.calc_smpl = bool(s.calc_smpl)
        if self.calc_smpl:
            if smpla_pack is None:
                smpla_pack = torch.load(s.smpl_path, map_location="cpu")
            if smil_pack is None:
                smil_pack = torch.load(s.smil_path, map_location="cpu")
            self.smpla = SMPLParser(smpla_pack, self.device_index, n_betas=11, shape_key="smpla_shapedirs")   # post_parser.py:259
            self.smil = SMPLParser(smil_pack, self.device_index, n_betas=10)                                     # :258
        self._alloc(B)

    def _net(self, in_dtype):
        if in_dtype not in self._nets:
            self._nets[in_dtype] = graph.build_bev(self._sd, self.device_index, self.precision, in_dtype, self.max_batch)
        return self._nets[in_dtype]

    def _alloc(self, B):
        dev, cap = self.tdevice, B * MAX_PERSON
        self.cap = cap
        act = torch.bfloat16 if self.precision == "bf16" else torch.float32
        self.act_code = BF16 if self.precision == "bf16" else F32
        z = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, device=dev)
        i64, i32 = torch.int64, torch.int32
        self.buf = dict(
            maps_fv=z(B, 4, 128, 128), fv_feats=z(B, 128, 128, 128, dtype=act), img_feats=z(B, 128, 128, graph.bev_feats_channels(self.precision), dtype=act),
            bv_in=z(B, 1, 128, 2560, dtype=act), bv_out=z(B, 1, 128, 128, dtype=act),
            c3d_tmp=z(B, 64, 128, 128), center3d=z(B, 64, 128, 128),
            parse_ws=torch.zeros(int(self.lib.b200romp_bev_parse_workspace_bytes(B)), dtype=torch.uint8, device=dev),
            count=z(1, dtype=i32), batch_ids=z(cap, dtype=i64), czyx=z(cap, 3, dtype=i64), conf=z(cap),
            params_pred=z(cap, N_PARAMS), cam_czyx=z(cap, 3, dtype=i64), cam=z(cap, 3), thetas=z(cap, 72), betas=z(cap, 11),
            cam_trans=z(cap, 3), pj2d_org=z(cap, 71, 2), keep=z(cap, dtype=i32), sel=z(cap, dtype=i32), count2=z(1, dtype=i32),
        )
        if self.calc_smpl:
            self.buf.update(verts=z(cap, 6890, 3), joints=z(cap, 71, 3), verts_smil=z(cap, 6890, 3), joints_smil=z(cap, 71, 3),
                            smpl_ws=z(cap, self.smpla.ws_floats))
        # compacted outputs (after the per-frame post filters)
        self.out = {k: torch.zeros_like(self.buf[k]) for k in ("batch_ids", "conf", "params_pred", "cam", "thetas", "betas",
                                                               "cam_trans", "pj2d_org")}
        if self.calc_smpl:
            self.out.update(verts=torch.zeros_like(self.buf["verts"]), joints=torch.zeros_like(self.buf["joints"]))
        self.count_host = torch.zeros(2, dtype=torch.int32).pin_memory()

    # ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def run_model(self, frames_dev, center3d_override=None):
        """BEVv1.forward (bev/model.py:232-250) + pack_params_dict / cam_trans (bev/main.py:128-129); no host sync."""
        B = frames_dev.shape[0]
        assert frames_dev.is_cuda and frames_dev.is_contiguous() and tuple(frames_dev.shape[1:]) == (512, 512, 3)
        assert B <= self.max_batch
        in_dtype = {torch.uint8: U8, torch.float32: F32}[frames_dev.dtype]
        g1, io1, g2, io2 = self._net(in_dtype)
        lib, b, sp, ac = self.lib, self.buf, C.c_void_p(self.stream.cuda_stream), self.act_code
        ck = _lib.check
        ck(lib.b200romp_net_bind(g1.net, io1["frames"], _ptr(frames_dev)))
        ck(lib.b200romp_net_bind(g1.net, io1["maps_fv"], _ptr(b["maps_fv"])))
        ck(lib.b200romp_net_bind(g1.net, io1["fv_feats"], _ptr(b["fv_feats"])))
        ck(lib.b200romp_net_bind(g1.net, io1["img_feats"], _ptr(b["img_feats"])))
        ck(lib.b200romp_net_run(g1.net, B, sp), "net_run(g1)")
        ck(lib.b200romp_bev_bv_input(_ptr(b["maps_fv"]), _ptr(b["img_feats"]), ac, b["img_feats"].shape[-1], B, _ptr(b["bv_in"]), ac, sp),
           "bv_input")
        ck(lib.b200romp_net_bind(g2.net, io2["bv_in"], _ptr(b["bv_in"])))
        ck(lib.b200romp_net_bind(g2.net, io2["bv_out"], _ptr(b["bv_out"])))
        ck(lib.b200romp_net_run(g2.net, B, sp), "net_run(g2)")
        ck(lib.b200romp_bev_center3d(self.h, _ptr(b["maps_fv"]), _ptr(b["bv_out"]), ac, B, _ptr(b["c3d_tmp"]), _ptr(b["center3d"]), sp),
           "center3d")
        c3d = b["center3d"] if center3d_override is None else center3d_override
        ck(lib.b200romp_bev_parse3d(_ptr(c3d), B, float(self.settings.center_thresh), self.cap, _ptr(b["count"]), _ptr(b["batch_ids"]),
                                    _ptr(b["czyx"]), _ptr(b["conf"]), _ptr(b["parse_ws"]), sp), "parse3d")
        ck(lib.b200romp_bev_regress(self.h, _ptr(b["maps_fv"]), _ptr(b["bv_out"]), ac, _ptr(b["fv_feats"]), ac, B * MAX_PERSON,
                                    _ptr(b["count"]), _ptr(b["batch_ids"]), _ptr(b["czyx"]), _ptr(b["params_pred"]),
                                    _ptr(b["cam_czyx"]), _ptr(b["cam"]), _ptr(b["thetas"]), _ptr(b["betas"]), _ptr(b["cam_trans"]), sp),
           "regress")

    @torch.no_grad()
    def run_post(self, B, offsets, img_max_side=512.0):
        """SMPLA_parser + projection + the two per-frame filters (bev/main.py:172-180), then row compaction."""
        lib, b, o, sp = self.lib, self.buf, self.out, C.c_void_p(self.stream.cuda_stream)
        cap = B * MAX_PERSON
        off = (C.c_float * 6)(*[float(v) for v in offsets])
        if not self.calc_smpl:
            return
        st = self.stream.cuda_stream
        self.smpla.forward(b["betas"], b["thetas"], cap, b["count"], True, b["smpl_ws"], b["verts"], b["joints"], st)
        self.smil.forward(b["betas"], b["thetas"], cap, b["count"], True, b["smpl_ws"], b["verts_smil"], b["joints_smil"], st)
        _lib.check(lib.b200romp_bev_post(_ptr(b["betas"]), _ptr(b["verts_smil"]), _ptr(b["joints_smil"]), _ptr(b["verts"]),
                                         _ptr(b["joints"]), _ptr(b["cam"]), _ptr(b["cam_trans"]), _ptr(b["batch_ids"]), B, cap,
                                         _ptr(b["count"]), off, float(self.settings.nms_thresh),
                                         float(self.settings.relative_scale_thresh), float(img_max_side), _ptr(b["pj2d_org"]),
                                         _ptr(b["keep"]), _ptr(b["sel"]), _ptr(b["count2"]), sp), "bev_post")
        for k, dst in o.items():
            src = b["conf"] if k == "conf" else b[k]
            row = src[0].numel() * src.element_size()
            _lib.check(lib.b200romp_gather_rows(_ptr(src), row, _ptr(b["sel"]), _ptr(b["count2"]), cap, _ptr(dst), sp), "gather_rows")

    def collect(self, to_numpy=True):
        with torch.cuda.stream(self.stream):
            self.count_host[0:1].copy_(self.buf["count"], non_blocking=True)
            self.count_host[1:2].copy_(self.buf["count2"], non_blocking=True)
        self.stream.synchronize()
        n_det, n = int(self.count_host[0]), int(self.count_host[1])
        if n_det == 0:
            return None
        if not self.calc_smpl:
            b = self.buf
            out = {"smpl_thetas": b["thetas"][:n_det], "smpl_betas": b["betas"][:n_det], "cam": b["cam"][:n_det],
                   "cam_trans": b["cam_trans"][:n_det], "params_pred": b["params_pred"][:n_det],
                   "center_confs": b["conf"][:n_det], "pred_batch_ids": b["batch_ids"][:n_det]}
        else:
            o = self.out
            out = {"smpl_thetas": o["thetas"][:n], "smpl_betas": o["betas"][:n], "cam": o["cam"][:n], "cam_trans": o["cam_trans"][:n],
                   "params_pred": o["params_pred"][:n], "center_confs": o["conf"][:n], "pred_batch_ids": o["batch_ids"][:n],
                   "verts": o["verts"][:n], "joints": o["joints"][:n], "pj2d_org": o["pj2d_org"][:n]}
        if to_numpy:
            with torch.cuda.stream(self.stream):
                out = {k: v.contiguous().cpu().numpy() for k, v in out.items()}
        return out

    @torch.no_grad()
    def forward_batch(self, frames, offsets=None, to_numpy=True, center3d_override=None, img_max_side=512.0):
        if isinstance(frames, np.ndarray):
            frames = torch.from_numpy(frames)
        B = frames.shape[0]
        # device-resident inputs come from the caller's current stream: order self.stream after it (no host sync)
        cur = torch.cuda.current_stream(self.tdevice)
        for t in (frames, center3d_override):
            if isinstance(t, torch.Tensor) and t.is_cuda:
                if cur != self.stream:
                    self.stream.wait_stream(cur)
                t.record_stream(self.stream)
        key = (frames.dtype, B)
        if key not in self._staging:                  # stable pointer -> one cached CUDA graph per (dtype, B)
            self._staging[key] = torch.empty((B, 512, 512, 3), dtype=frames.dtype, device=self.tdevice)
        fd = self._staging[key]
        with torch.cuda.stream(self.stream):
            fd.copy_(frames, non_blocking=True)
            self.run_model(fd, center3d_override)
            self.run_post(B, offsets if offsets is not None else [0, 512, 0, 512, 512, 512], img_max_side)
        return self.collect(to_numpy)

    # ------------------------------------------------------------------------------------------
    _long_fields = ("thetas", "betas", "cam", "params_pred", "conf", "verts", "joints")

    def _long_alloc(self, mcap):
        """Merged buffers of crowd mode for up to ``mcap`` people (S crops x 64), grown on demand."""
        if getattr(self, "_long", None) is not None and self._long["mcap"] >= mcap:
            return self._long
        self._long = None
        dev, b = self.tdevice, self.buf
        z = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype, device=dev)
        L = {"mcap": mcap, "cam_full": z(self.cap, 3), "flags": z(2 * self.cap, dtype=torch.int32), "base": z(1, dtype=torch.int32),
             "merged": z(1, dtype=torch.int32), "cam_trans": z(mcap, 3), "pj2d_org": z(mcap, 71, 2),
             "ws": z(3 * mcap + 1, dtype=torch.int32), "sel": z(mcap, dtype=torch.int32), "count_out": z(1, dtype=torch.int32),
             "plan": z(2 * mcap, dtype=torch.int32), "plan_host": torch.zeros(2 * mcap, dtype=torch.int32).pin_memory()}
        L["m"] = {k: z(mcap, *b[k].shape[1:]) for k in self._long_fields}
        L["o"] = {k: z(mcap, *b[k].shape[1:]) for k in self._long_fields + ("cam_trans", "pj2d_org")}
        self._long = L
        return L

    def _long_upload(self, img):
        """raw HxWx3 uint8 image -> device, on self.stream, without a host sync: a host image goes through a pinned buffer
        (free again: every call ends with the stream synchronised by ``collect``)."""
        if img.is_cuda:
            cur = torch.cuda.current_stream(self.tdevice)
            if cur != self.stream:
                self.stream.wait_stream(cur)
            img.record_stream(self.stream)
            return img.contiguous()
        n = img.numel()
        if getattr(self, "_raw_host", None) is None or self._raw_host.numel() < n:
            self._raw_host = torch.empty(max(n, 1 << 22), dtype=torch.uint8).pin_memory()
            self._raw_dev = torch.empty(self._raw_host.numel(), dtype=torch.uint8, device=self.tdevice)
        self._raw_host[:n].copy_(img.reshape(-1))
        raw = self._raw_dev[:n]
        raw.copy_(self._raw_host[:n], non_blocking=True)
        return raw

    @torch.no_grad()
    def process_long_image(self, full_image, show_patch_results=False, center3d_override=None, to_numpy=True):
        """BEV.process_long_image (bev/main.py:184-258): crowd mode for images with w/h >= 2.  The image is padded by
        int(h * overlap_ratio) zero columns on each side and cut into S overlapping full-height crops
        (bev/split2process.py); the crops run as batches of <= max_batch through the batched BEV path, every per-crop
        and merge step runs on the device, and the only host synchronisation is the final person count.

        full_image: HxWx3 uint8 BGR, numpy or tensor (host or device).  center3d_override [S,64,128,128] replaces each
        crop's 3-D centre map (tests).  Returns the dict of ``forward_batch`` (pred_batch_ids all 0, full-image cam /
        cam_trans / pj2d_org) or None.  Deliberate differences to the reference: a crop without detections contributes
        nothing (the reference's crop bookkeeping misaligns and raises), and an image without survivors returns None
        (the reference raises KeyError)."""
        if show_patch_results:
            raise NotImplementedError("show_patch_results renders every crop; rendering is outside the B200 hot path")
        if not self.calc_smpl:
            raise ValueError("crowd mode (images with w/h >= 2 and --crowd on) needs SMPL: the crops are merged on projected "
                             "joints, so build BEV with calc_smpl on")
        img = torch.from_numpy(np.ascontiguousarray(full_image)) if isinstance(full_image, np.ndarray) else full_image
        assert img.dtype == torch.uint8 and img.dim() == 3 and img.shape[2] == 3, "image must be HxWx3 uint8 (BGR)"
        h, w = int(img.shape[0]), int(img.shape[1])
        plan, pad = long_image_plan(h, w, float(self.settings.overlap_ratio))
        S = len(plan)
        assert S >= 2 and int((plan[:, 1] - plan[:, 0]).max()) <= h, "crowd mode needs w/h >= 2"
        L = self._long_alloc(S * MAX_PERSON)
        if center3d_override is not None:
            center3d_override = torch.as_tensor(center3d_override, dtype=torch.float32, device=self.tdevice)
            assert tuple(center3d_override.shape) == (S, 64, 128, 128), "center3d_override must be [S,64,128,128]"
        cur = torch.cuda.current_stream(self.tdevice)
        if center3d_override is not None and cur != self.stream:
            self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            raw = self._long_upload(img)
            self._long_begin(plan)
            for c0 in range(0, S, self.max_batch):
                nb = min(self.max_batch, S - c0)
                key = (torch.uint8, nb)
                if key not in self._staging:
                    self._staging[key] = torch.empty((nb, 512, 512, 3), dtype=torch.uint8, device=self.tdevice)
                fd = self._staging[key]
                _lib.check(self.lib.b200romp_preprocess_crops_bgr(_ptr(raw), h, w, 3 * w, pad, _ptr(L["plan"]), c0, nb, 512, _ptr(fd),
                                                                  C.c_void_p(self.stream.cuda_stream)), "preprocess_crops_bgr")
                self.run_model(fd, None if center3d_override is None else center3d_override[c0:c0 + nb])
                self._long_chunk(plan, pad, c0, nb, h, w)
            self._long_finish(h, w)
        return self._long_collect(to_numpy)

    def _long_begin(self, plan):
        L = self._long
        L["plan_host"][:plan.size].copy_(torch.from_numpy(plan.reshape(-1)))
        L["plan"][:plan.size].copy_(L["plan_host"][:plan.size], non_blocking=True)
        L["merged"].zero_()

    def _long_chunk(self, plan, pad, c0, nb, h, w):
        """Crops c0 .. c0+nb-1, detected and regressed into self.buf (batch_ids = crop - c0): SMPL-A / SMIL, then
        bev/main.py:203-249 on the device, survivors appended to the merged buffers."""
        lib, b, L, sp, ck = self.lib, self.buf, self._long, C.c_void_p(self.stream.cuda_stream), _lib.check
        s, st = self.settings, self.stream.cuda_stream
        self.smpla.forward(b["betas"], b["thetas"], self.cap, b["count"], True, b["smpl_ws"], b["verts"], b["joints"], st)
        self.smil.forward(b["betas"], b["thetas"], self.cap, b["count"], True, b["smpl_ws"], b["verts_smil"], b["joints_smil"], st)
        crop_thr = float(s.nms_thresh) * h / 640          # nms_thresh * max(crop h, crop w) / 640 (post_parser.py:186-187)
        ck(lib.b200romp_bev_long_crops(_ptr(b["betas"]), _ptr(b["verts_smil"]), _ptr(b["joints_smil"]), _ptr(b["verts"]),
                                       _ptr(b["joints"]), _ptr(b["cam"]), _ptr(b["cam_trans"]), _ptr(b["conf"]), _ptr(b["batch_ids"]),
                                       nb, self.cap, _ptr(b["count"]), _ptr(L["plan"]), len(plan), c0, h, w, pad, crop_thr,
                                       float(s.relative_scale_thresh), _ptr(b["pj2d_org"]), _ptr(L["cam_full"]), _ptr(L["flags"]),
                                       _ptr(b["sel"]), _ptr(b["count2"]), _ptr(L["base"]), _ptr(L["merged"]), L["mcap"], sp),
           "bev_long_crops")
        for k in self._long_fields:
            src = L["cam_full"] if k == "cam" else b[k]
            ck(lib.b200romp_gather_rows_at(_ptr(src), src[0].numel() * 4, _ptr(b["sel"]), _ptr(b["count2"]), _ptr(L["base"]),
                                           self.cap, _ptr(L["m"][k]), sp), "gather_rows_at")

    def _long_finish(self, h, w):
        """bev/main.py:253-256 over all merged people, survivors gathered into the output buffers."""
        lib, L, m, sp, ck = self.lib, self._long, self._long["m"], C.c_void_p(self.stream.cuda_stream), _lib.check
        s, mcap = self.settings, self._long["mcap"]
        full_thr = float(s.nms_thresh) * max(h, w, 3) / 640                # image.shape has 3 entries (main.py:255)
        ck(lib.b200romp_bev_long_merge(_ptr(m["joints"]), _ptr(m["cam"]), _ptr(m["conf"]), mcap, _ptr(L["merged"]), h, w, full_thr,
                                       float(s.relative_scale_thresh), _ptr(L["cam_trans"]), _ptr(L["pj2d_org"]), _ptr(L["ws"]),
                                       _ptr(L["sel"]), _ptr(L["count_out"]), sp), "bev_long_merge")
        for k, dst in L["o"].items():
            src = L[k] if k in ("cam_trans", "pj2d_org") else m[k]
            ck(lib.b200romp_gather_rows(_ptr(src), src[0].numel() * 4, _ptr(L["sel"]), _ptr(L["count_out"]), mcap, _ptr(dst), sp),
               "gather_rows")
        self.count_host[0:1].copy_(L["count_out"], non_blocking=True)

    def _long_collect(self, to_numpy=True):
        self.stream.synchronize()                                           # the one host synchronisation of a wide image
        n = int(self.count_host[0])
        if n == 0:
            return None
        o = self._long["o"]
        out = {"smpl_thetas": o["thetas"][:n], "smpl_betas": o["betas"][:n], "cam": o["cam"][:n], "cam_trans": o["cam_trans"][:n],
               "params_pred": o["params_pred"][:n], "center_confs": o["conf"][:n],
               "pred_batch_ids": torch.zeros(n, dtype=torch.int64, device=self.tdevice), "verts": o["verts"][:n],
               "joints": o["joints"][:n], "pj2d_org": o["pj2d_org"][:n]}
        if to_numpy:
            out = {k: v.cpu().numpy() for k, v in out.items()}
        return out

    @torch.no_grad()
    def forward(self, image, signal_ID=0, **kwargs):
        """image: HxWx3 uint8 BGR.  bev/main.py:139-156; with ``crowd`` (the default) an image of aspect ratio >= 2 goes
        through ``process_long_image``."""
        if image.shape[1] / image.shape[0] >= 2 and self.settings.crowd:
            return self.process_long_image(image, show_patch_results=getattr(self.settings, "show_patch_results", False))
        inp, pad = img_preprocess(image)
        out = self.forward_batch(torch.from_numpy(inp), offsets=pad, img_max_side=float(max(image.shape[:2])))
        if out is None:
            print("No person detected!")                                       # bev/model.py:239
            return None
        return out

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.b200romp_bev_destroy(self.h)
        except Exception:
            pass
