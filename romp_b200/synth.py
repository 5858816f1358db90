"""Deterministic synthetic parameters for the ROMP hot path.

The released checkpoint (``ROMP.pkl``) and the licensed SMPL model file are not
available offline, so the benchmarks and parity tests run on seeded synthetic
parameters that have exactly the reference's schema:

* ``romp_state_dict(seed)``  -> dict with the 1851 keys / shapes of
  ``ROMPv1().state_dict()`` (reference: simple_romp/romp/model.py:420-481).
* ``smpl_pack(seed)``        -> dict with the keys written by
  simple_romp/romp/pack_smpl_info.py:70-111 and read by
  simple_romp/romp/smpl.py:41-59.

Everything is drawn from ``numpy.random.RandomState`` so the values do not depend
on the torch version.  BatchNorm statistics are randomised so that BN folding is
really exercised.
"""
from __future__ import annotations

import numpy as np

# --------------------------------------------------------------------------------------
# HRNet-W32 + ROMP head parameter enumeration (names and shapes only)
# --------------------------------------------------------------------------------------
STAGE_CFG = {
    2: dict(modules=1, channels=[32, 64]),
    3: dict(modules=4, channels=[32, 64, 128]),
    4: dict(modules=3, channels=[32, 64, 128, 256]),
}
BLOCKS_PER_BRANCH = 4
HEAD_OUT = {1: 142, 2: 1, 3: 3}   # final_layers index -> output channels (params, center, cam)


def _conv(specs, name, cout, cin, k, bias=False):
    specs.append((name + ".weight", (cout, cin, k, k), "conv_w"))
    if bias:
        specs.append((name + ".bias", (cout,), "conv_b", cin * k * k))


def _bn(specs, name, c):
    specs.append((name + ".weight", (c,), "bn_w"))
    specs.append((name + ".bias", (c,), "bn_b"))
    specs.append((name + ".running_mean", (c,), "bn_m"))
    specs.append((name + ".running_var", (c,), "bn_v"))
    specs.append((name + ".num_batches_tracked", (), "bn_n"))


def romp_param_specs():
    """Ordered (name, shape, kind, ...) list equal to ROMPv1().state_dict() order."""
    s = []
    p = "backbone."
    _conv(s, p + "conv1", 64, 3, 3); _bn(s, p + "bn1", 64)
    _conv(s, p + "conv2", 64, 64, 3); _bn(s, p + "bn2", 64)
    # layer1: 4 Bottlenecks, first has a 1x1 downsample 64->256
    for i in range(4):
        q = f"{p}layer1.{i}."
        cin = 64 if i == 0 else 256
        _conv(s, q + "conv1", 64, cin, 1); _bn(s, q + "bn1", 64)
        _conv(s, q + "conv2", 64, 64, 3); _bn(s, q + "bn2", 64)
        _conv(s, q + "conv3", 256, 64, 1); _bn(s, q + "bn3", 256)
        if i == 0:
            _conv(s, q + "downsample.0", 256, 64, 1); _bn(s, q + "downsample.1", 256)
    # transition1: [256] -> [32, 64]
    _conv(s, p + "transition1.0.0", 32, 256, 3); _bn(s, p + "transition1.0.1", 32)
    _conv(s, p + "transition1.1.0.0", 64, 256, 3); _bn(s, p + "transition1.1.0.1", 64)

    def stage(idx):
        cfg = STAGE_CFG[idx]
        ch = cfg["channels"]
        nb = len(ch)
        for m in range(cfg["modules"]):
            q = f"{p}stage{idx}.{m}."
            for b in range(nb):
                for k in range(BLOCKS_PER_BRANCH):
                    r = f"{q}branches.{b}.{k}."
                    _conv(s, r + "conv1", ch[b], ch[b], 3); _bn(s, r + "bn1", ch[b])
                    _conv(s, r + "conv2", ch[b], ch[b], 3); _bn(s, r + "bn2", ch[b])
            multi = not (idx == 4 and m == cfg["modules"] - 1)
            for i in range(nb if multi else 1):
                for j in range(nb):
                    r = f"{q}fuse_layers.{i}.{j}."
                    if j > i:
                        _conv(s, r + "0", ch[i], ch[j], 1); _bn(s, r + "1", ch[i])
                    elif j < i:
                        for k in range(i - j):
                            cout = ch[i] if k == i - j - 1 else ch[j]
                            _conv(s, f"{r}{k}.0", cout, ch[j], 3); _bn(s, f"{r}{k}.1", cout)

    stage(2)
    _conv(s, p + "transition2.2.0.0", 128, 64, 3); _bn(s, p + "transition2.2.0.1", 128)
    stage(3)
    _conv(s, p + "transition3.3.0.0", 256, 128, 3); _bn(s, p + "transition3.3.0.1", 256)
    stage(4)
    for h in (1, 2, 3):
        q = f"final_layers.{h}."
        _conv(s, q + "0.0", 64, 34, 3, bias=True); _bn(s, q + "0.1", 64)
        for blk in range(2):
            r = f"{q}1.{blk}.0."
            _conv(s, r + "conv1", 64, 64, 3); _bn(s, r + "bn1", 64)
            _conv(s, r + "conv2", 64, 64, 3); _bn(s, r + "bn2", 64)
        _conv(s, q + "2", HEAD_OUT[h], 64, 1, bias=True)
    return s


def romp_state_dict(seed: int = 0, gain: float = 0.55):
    """Synthetic ROMPv1 state dict as numpy arrays (float32 / int64 scalars)."""
    rng = np.random.RandomState(seed)
    sd = {}
    for spec in romp_param_specs():
        name, shape, kind = spec[0], spec[1], spec[2]
        if kind == "conv_w":
            fan_in = shape[1] * shape[2] * shape[3]
            bound = gain * np.sqrt(3.0 / fan_in)          # unit-variance-preserving uniform
            v = rng.uniform(-bound, bound, size=shape)
        elif kind == "conv_b":
            bound = 1.0 / np.sqrt(spec[3])
            v = rng.uniform(-bound, bound, size=shape)
        elif kind == "bn_w":
            v = rng.uniform(0.5, 1.5, size=shape)
        elif kind == "bn_b":
            v = rng.normal(0.0, 0.1, size=shape)
        elif kind == "bn_m":
            v = rng.normal(0.0, 0.1, size=shape)
        elif kind == "bn_v":
            v = rng.uniform(0.5, 1.5, size=shape)
        elif kind == "bn_n":
            sd[name] = np.array(1, dtype=np.int64)
            continue
        else:  # pragma: no cover
            raise ValueError(kind)
        sd[name] = v.astype(np.float32)
    return sd


# --------------------------------------------------------------------------------------
# Synthetic packed SMPL (schema: simple_romp/romp/pack_smpl_info.py:70-111)
# --------------------------------------------------------------------------------------
SMPL_PARENTS = np.array([-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14,
                         16, 17, 18, 19, 20, 21], dtype=np.int64)
NUM_VERTS = 6890
NUM_FACES = 13776


def smpl_pack(seed: int = 0, num_betas: int = 10, dense_weights: bool = False):
    """Synthetic packed SMPL with human-like magnitudes.

    v_template ~ a 1.7 m tall point cloud, shapedirs ~ cm scale, posedirs ~ mm-cm scale,
    skinning weights with 4 non-zeros per vertex (or dense if ``dense_weights``) that sum to 1,
    joint regressors as sparse convex combinations (stored dense like the reference).
    """
    rng = np.random.RandomState(seed + 7919)
    V = NUM_VERTS
    v_template = (rng.uniform(-1, 1, size=(V, 3)) * np.array([0.45, 0.85, 0.15])).astype(np.float32)
    shapedirs = (rng.normal(0, 0.01, size=(V, 3, num_betas))).astype(np.float32)
    posedirs = (rng.normal(0, 0.004, size=(207, V * 3))).astype(np.float32)

    def convex_rows(rows, nnz):
        m = np.zeros((rows, V), dtype=np.float64)
        for r in range(rows):
            idx = rng.choice(V, size=nnz, replace=False)
            w = rng.uniform(0.1, 1.0, size=nnz)
            m[r, idx] = w / w.sum()
        return m.astype(np.float32)

    J_regressor = convex_rows(24, 48)
    J_extra9 = convex_rows(9, 32)
    J_h36m17 = convex_rows(17, 64)
    if dense_weights:
        w = rng.uniform(0.0, 1.0, size=(V, 24)) ** 4
    else:
        w = np.zeros((V, 24), dtype=np.float64)
        for v in range(V):
            idx = rng.choice(24, size=4, replace=False)
            w[v, idx] = rng.uniform(0.05, 1.0, size=4)
    weights = (w / w.sum(1, keepdims=True)).astype(np.float32)
    extra_joints_index = rng.choice(V, size=21, replace=False).astype(np.int64)
    faces = rng.randint(0, V, size=(NUM_FACES, 3)).astype(np.int64)
    key = "shapedirs" if num_betas == 10 else "smpla_shapedirs"
    pack = {
        "kintree_table": SMPL_PARENTS.copy(),
        "J_regressor_extra9": J_extra9,
        "J_regressor_h36m17": J_h36m17,
        key: shapedirs,
        "posedirs": posedirs,
        "extra_joints_index": extra_joints_index,
        "f": faces,
        "v_template": v_template,
        "J_regressor": J_regressor,
        "weights": weights,
    }
    if num_betas != 10:
        pack["shapedirs"] = shapedirs[:, :, :10].copy()
    return pack


def synthetic_frames(batch: int, seed: int = 0, dtype=np.uint8):
    """[B,512,512,3] frames with values 0..255 (what img_preprocess produces, utils.py:26-30)."""
    rng = np.random.RandomState(seed + 104729)
    # low-frequency structure + noise so activations are not pure white noise
    base = rng.randint(0, 256, size=(batch, 64, 64, 3)).astype(np.float32)
    up = np.repeat(np.repeat(base, 8, axis=1), 8, axis=2)
    noise = rng.randint(-32, 33, size=(batch, 512, 512, 3)).astype(np.float32)
    x = np.clip(up + noise, 0, 255)
    return x.astype(dtype)


def plant_centers(batch: int, seed: int = 0, kmin: int = 1, kmax: int = 10, size: int = 64):
    """Center maps [B,1,size,size] with K_b ~ U{kmin..kmax} isolated peaks per frame.

    Peaks are >=3 cells apart (5x5 NMS keeps them all) and have distinct values in (0.3, 1.0)
    so that the top-k order has no ties (SURVEY section 8d cfg2).
    Returns (maps float32, list of per-frame [(flat_index, value)] sorted by value desc).
    """
    rng = np.random.RandomState(seed + 15485863)
    maps = np.zeros((batch, 1, size, size), dtype=np.float32)
    truth = []
    for b in range(batch):
        k = rng.randint(kmin, kmax + 1)
        cells = []
        tries = 0
        while len(cells) < k and tries < 10000:
            tries += 1
            y, x = rng.randint(0, size), rng.randint(0, size)
            if all(max(abs(y - cy), abs(x - cx)) >= 3 for cy, cx in cells):
                cells.append((y, x))
        vals = rng.uniform(0.3, 1.0, size=len(cells)).astype(np.float32)
        vals = np.unique(vals)[: len(cells)]
        rng.shuffle(vals)
        cur = []
        for (y, x), v in zip(cells, vals):
            maps[b, 0, y, x] = v
            cur.append((y * size + x, float(v)))
        cur.sort(key=lambda t: -t[1])
        truth.append(cur)
    return maps, truth


# --------------------------------------------------------------------------------------
# BEV head parameters (simple_romp/bev/model.py:104-187): enumeration + synthetic values
# --------------------------------------------------------------------------------------
def plant_centers_3d(batch: int, seed: int = 0, kmin: int = 1, kmax: int = 10, z_lo: int = 24, z_hi: int = 44, min_sep: int = 20):
    """BEV cfg3 workload: 3-D center maps [B,64,128,128] (low uniform background + K_b ~ U{kmin..kmax} planted peaks per
    frame) whose persons SURVIVE BEV's per-frame post-filters, so that the step really processes <= 10 kept persons
    per frame: depth levels z_lo..z_hi (scale anchors 1.08..0.45: `remove_outlier` only drops scales < 0.25,
    bev/post_parser.py:200-222) and >= min_sep cells (= 4*min_sep pixels) apart in the image plane, far beyond the
    duplicate-suppression radius nms_thresh * 512/640 * 2*scale pixels (bev/post_parser.py:167-198).
    Returns (volume float32, number of planted persons)."""
    rs = np.random.RandomState(seed + 32452843)
    vol = rs.uniform(0, 0.05, size=(batch, 64, 128, 128)).astype(np.float32)
    persons = 0
    for b in range(batch):
        k = rs.randint(kmin, kmax + 1)
        cells, tries = [], 0
        while len(cells) < k and tries < 20000:
            tries += 1
            y, x = rs.randint(8, 120), rs.randint(8, 120)
            if all(max(abs(y - cy), abs(x - cx)) >= min_sep for cy, cx in cells):
                cells.append((y, x))
        for (y, x) in cells:
            vol[b, rs.randint(z_lo, z_hi + 1), y, x] = rs.uniform(0.3, 1.0)
            persons += 1
    return vol, persons


def nms_peaks(center_maps):
    """Values and flat indices of the 5x5 local maxima of [B,1,S,S] maps (CenterMap.nms, post_parser.py:50-54), per frame."""
    cm = np.asarray(center_maps, np.float32)[:, 0]
    B, S, _ = cm.shape
    pad = np.full((B, S + 4, S + 4), -np.inf, np.float32)
    pad[:, 2:-2, 2:-2] = cm
    mx = np.max(np.stack([pad[:, dy:dy + S, dx:dx + S] for dy in range(5) for dx in range(5)]), 0)
    return [(cm[b][mx[b] == cm[b]], np.flatnonzero((mx[b] == cm[b]).ravel())) for b in range(B)]


def calibrate_center_head(sd, center_maps, max_per_frame: float = 10.0, thresh: float = 0.25):
    """Synthetic weights detect nobody (the raw center head hovers around 0), so the natural-detection tests and benches
    calibrate the LAST layer of the center head, ``final_layers.2.2`` (Conv2d 64->1 with bias, model.py:455-468): its
    bias is shifted so that between 1 and ``max_per_frame`` NMS peaks per frame (on average) of ``center_maps`` (the
    fp32 maps the un-shifted weights produce on the calibration frames) exceed ``thresh``.  The cut is placed in the
    middle of the WIDEST gap between consecutive pooled peak values in that rank range, so the detection set is as far
    from a threshold tie as the data allow ("tie-free inputs").  Returns (new state dict, shift, half-width of the
    gap = decision margin)."""
    peaks = np.sort(np.concatenate([v for v, _ in nms_peaks(center_maps)]))[::-1]
    B = np.asarray(center_maps).shape[0]
    lo, hi = max(1, B), min(len(peaks) - 1, int(max_per_frame * B))
    gaps = peaks[lo - 1:hi - 1] - peaks[lo:hi]
    j = int(np.argmax(gaps)) + lo                      # peaks[:j] fire, peaks[j:] do not
    cut = 0.5 * (float(peaks[j - 1]) + float(peaks[j]))
    out = dict(sd)
    out["final_layers.2.2.bias"] = (np.asarray(sd["final_layers.2.2.bias"], np.float32) + np.float32(thresh - cut)).astype(np.float32)
    return out, float(thresh - cut), 0.5 * float(gaps[j - lo])


def bev_damp_cam_offsets(sd, factor: float = 0.02):
    """cfg3 workload calibration.  With random weights the three cam-OFFSET producers of BEVv1 (det_head.1 channels 1..3,
    the upper 64 channels of bv_out_layers' last BatchNorm1d, and cam_map_refiner's residual branch; bev/model.py:200-213)
    emit O(1..10) noise on top of the 3-D coordinate map, so most planted people get huge scales and are removed as
    duplicates by suppressing_redundant_prediction_via_projection (distance normalised by 2*scale; round 1 kept 39 of 169).
    A trained model predicts small offsets; scaling those three outputs by ``factor`` makes cam ~ coordmap_3d[z, y, x], so
    people planted at distinct cells really are distinct people and survive the per-frame post-filters."""
    out = dict(sd)
    f = np.float32(factor)
    for k in ("det_head.1.weight", "det_head.1.bias"):
        v = np.array(out[k], np.float32, copy=True)
        v[1:4] *= f
        out[k] = v
    for k in ("bv_out_layers.2.bn2.weight", "bv_out_layers.2.bn2.bias"):
        v = np.array(out[k], np.float32, copy=True)
        v[64:] *= f
        out[k] = v
    for k in ("cam_map_refiner.0.bn2.weight", "cam_map_refiner.0.bn2.bias"):
        out[k] = np.array(out[k], np.float32, copy=True) * f
    return out


def bev_cam3dmap_anchor(fov=60, size=128):
    """get_cam3dmap_anchor, bev/model.py:77-87: 64 strictly decreasing scale anchors."""
    depth_level = np.array([1, 10, 20, 100], dtype=np.float32)
    ranges = (np.array([2 / 64., 25 / 64., 3 / 64., 2 / 64.], dtype=np.float32) * size).astype(np.int32)
    scale_level = 1 / np.tan(np.radians(fov / 2.)) / depth_level
    out, cache = [], 8
    for scale, r in zip(scale_level, ranges):
        out.append(cache - np.arange(1, r + 1) / r * (cache - scale))
        cache = scale
    return np.concatenate(out).astype(np.float32)


def bev_coordmap_3d(size=128):
    """get_3Dcoord_maps_halfz, bev/model.py:9-17 -> [1,64,size,size,3] with last dim (Z=anchor, Y, X)."""
    z = bev_cam3dmap_anchor(60, size)
    r = np.arange(size, dtype=np.float32) / size * 2 - 1
    D = len(z)
    out = np.zeros((1, D, size, size, 3), np.float32)
    out[..., 0] = z[None, :, None, None]
    out[..., 1] = r[None, None, :, None]
    out[..., 2] = r[None, None, None, :]
    return out


def bev_head_param_specs():
    s = []

    def conv(name, shape, bias=False):
        s.append((name + ".weight", shape, "conv_w"))
        if bias:
            s.append((name + ".bias", (shape[0],), "conv_b", int(np.prod(shape[1:]))))

    s.append(("coordmap_3d", (1, 64, 128, 128, 3), "coordmap"))
    s.append(("position_embeddings.weight", (128, 128), "embed"))
    for i, (o, c) in zip((0, 3, 6), ((512, 128), (512, 512), (143, 512))):
        conv(f"transformer.{i}", (o, c), bias=True)
    for head in ("det_head", "param_head"):
        q = head + ".0.0."
        conv(q + "conv1", (128, 32, 3, 3)); _bn(s, q + "bn1", 128)
        conv(q + "conv2", (128, 128, 3, 3)); _bn(s, q + "bn2", 128)
        conv(q + "downsample", (128, 32, 1, 1), bias=True)
        if head == "det_head":
            conv("det_head.1", (4, 128, 1, 1), bias=True)
    conv("bv_pre_layers.0", (16, 32, 1, 1), bias=True); _bn(s, "bv_pre_layers.1", 16)
    conv("bv_pre_layers.3", (16, 16, 3, 3), bias=True); _bn(s, "bv_pre_layers.4", 16)
    conv("bv_pre_layers.6", (16, 16, 1, 1), bias=True); _bn(s, "bv_pre_layers.7", 16)
    for i, (cin, cout) in enumerate(((2560, 512), (512, 512), (512, 128))):
        q = f"bv_out_layers.{i}."
        conv(q + "conv1", (cout, cin, 3)); _bn(s, q + "bn1", cout)
        conv(q + "conv2", (cout, cout, 3)); _bn(s, q + "bn2", cout)
    for name, c in (("center_map_refiner", 1), ("cam_map_refiner", 3)):
        q = name + ".0."
        conv(q + "conv1", (c, c, 3, 3, 3)); _bn(s, q + "bn1", c)
        conv(q + "conv2", (c, c, 3, 3, 3)); _bn(s, q + "bn2", c)
    return s


def bev_state_dict(seed: int = 0, gain: float = 0.55):
    """Synthetic BEVv1 state dict: ROMP's backbone keys + the BEV head keys (1871 entries like the reference)."""
    sd = {k: v for k, v in romp_state_dict(seed, gain).items() if k.startswith("backbone.")}
    rng = np.random.RandomState(seed + 31337)
    for spec in bev_head_param_specs():
        name, shape, kind = spec[0], spec[1], spec[2]
        if kind == "coordmap":
            sd[name] = bev_coordmap_3d(128)
        elif kind == "embed":
            v = rng.normal(0, 0.5, size=shape).astype(np.float32)
            v[0] = 0.0                                   # nn.Embedding(padding_idx=0), bev/model.py:132
            sd[name] = v
        elif kind == "conv_w":
            fan_in = int(np.prod(shape[1:]))
            bound = gain * np.sqrt(3.0 / fan_in) * (2.0 if len(shape) == 5 else 1.0)
            sd[name] = rng.uniform(-bound, bound, size=shape).astype(np.float32)
        elif kind == "conv_b":
            bound = 1.0 / np.sqrt(spec[3])
            sd[name] = rng.uniform(-bound, bound, size=shape).astype(np.float32)
        elif kind == "bn_w":
            sd[name] = rng.uniform(0.5, 1.5, size=shape).astype(np.float32)
        elif kind in ("bn_b", "bn_m"):
            sd[name] = rng.normal(0.0, 0.1, size=shape).astype(np.float32)
        elif kind == "bn_v":
            sd[name] = rng.uniform(0.5, 1.5, size=shape).astype(np.float32)
        elif kind == "bn_n":
            sd[name] = np.array(1, dtype=np.int64)
    return sd


# --------------------------------------------------------------------------------------
# ResNet-50 backbone variant of ROMP (BASELINE.json configs[0]; romp/lib/models/resnet_50.py:19-120)
# --------------------------------------------------------------------------------------
def resnet50_param_specs():
    s = []
    _conv(s, "backbone.conv1", 64, 3, 7); _bn(s, "backbone.bn1", 64)
    inplanes = 64
    for li, (planes, blocks) in enumerate(((64, 3), (128, 4), (256, 6), (512, 3)), start=1):
        for b in range(blocks):
            q = f"backbone.layer{li}.{b}."
            _conv(s, q + "conv1", planes, inplanes, 1); _bn(s, q + "bn1", planes)
            _conv(s, q + "conv2", planes, planes, 3); _bn(s, q + "bn2", planes)
            _conv(s, q + "conv3", planes * 4, planes, 1); _bn(s, q + "bn3", planes * 4)
            if b == 0:
                _conv(s, q + "downsample.0", planes * 4, inplanes, 1); _bn(s, q + "downsample.1", planes * 4)
            inplanes = planes * 4
    cin = 2048
    for i, planes in enumerate((256, 128, 64)):
        s.append((f"backbone.deconv_layers.{3 * i}.weight", (cin, planes, 4, 4), "conv_w"))   # ConvTranspose2d: [in,out,k,k]
        _bn(s, f"backbone.deconv_layers.{3 * i + 1}", planes)
        cin = planes
    for h in (1, 2, 3):                      # ROMP head on 64 + 2 coord channels (romp/lib/models/romp_model.py)
        q = f"final_layers.{h}."
        _conv(s, q + "0.0", 64, 66, 3, bias=True); _bn(s, q + "0.1", 64)
        for blk in range(2):
            r = f"{q}1.{blk}.0."
            _conv(s, r + "conv1", 64, 64, 3); _bn(s, r + "bn1", 64)
            _conv(s, r + "conv2", 64, 64, 3); _bn(s, r + "bn2", 64)
        _conv(s, q + "2", HEAD_OUT[h], 64, 1, bias=True)
    return s


def resnet50_state_dict(seed: int = 0, gain: float = 0.8):
    rng = np.random.RandomState(seed + 50)
    sd = {}
    for spec in resnet50_param_specs():
        name, shape, kind = spec[0], spec[1], spec[2]
        if kind == "conv_w":
            fan_in = int(np.prod(shape[1:])) if "deconv" not in name else shape[0] * 4   # 2x2 of the 4x4 taps hit each output
            bound = gain * np.sqrt(3.0 / fan_in)
            sd[name] = rng.uniform(-bound, bound, size=shape).astype(np.float32)
        elif kind == "conv_b":
            sd[name] = (rng.uniform(-1, 1, size=shape) / np.sqrt(spec[3])).astype(np.float32)
        elif kind == "bn_w":
            sd[name] = rng.uniform(0.5, 1.5, size=shape).astype(np.float32)
        elif kind in ("bn_b", "bn_m"):
            sd[name] = rng.normal(0.0, 0.1, size=shape).astype(np.float32)
        elif kind == "bn_v":
            sd[name] = rng.uniform(0.5, 1.5, size=shape).astype(np.float32)
        elif kind == "bn_n":
            sd[name] = np.array(1, dtype=np.int64)
    return sd


def synthetic_wide_image(h: int, w: int, seed: int = 0):
    """HxWx3 uint8 BGR image of any size with the texture of ``synthetic_frames`` (8-pixel blocks + noise): the input of
    BEV's crowd mode (w/h >= 2, bev/main.py:140-141)."""
    rng = np.random.RandomState(seed + 1299709)
    base = rng.randint(0, 256, size=(h // 8 + 1, w // 8 + 1, 3)).astype(np.float32)
    up = np.repeat(np.repeat(base, 8, axis=0), 8, axis=1)[:h, :w]
    noise = rng.randint(-32, 33, size=(h, w, 3)).astype(np.float32)
    return np.clip(up + noise, 0, 255).astype(np.uint8)


def bev_planted_crops(n_crops: int, cells, seed: int = 0):
    """Per-crop 3-D centre maps [n_crops,64,128,128] for crowd mode: a uniform background in [0, 0.05) (below every BEV
    centre threshold) plus the caller's cells ``(crop, z, y, x, value)``.  Cells of one crop should be >= 3 voxels apart
    in some axis so that the 5x5x5 max-pool NMS (bev/post_parser.py:44-66) keeps each of them."""
    rs = np.random.RandomState(seed + 49979687)
    vol = rs.uniform(0, 0.05, size=(n_crops, 64, 128, 128)).astype(np.float32)
    for c, z, y, x, v in cells:
        vol[int(c), int(z), int(y), int(x)] = np.float32(v)
    return vol


def bev_crowd_state_dict(seed: int = 0, beta10_shift: float = 0.6735):
    """Synthetic BEV weights of the crowd-mode tests and bench: ``bev_damp_cam_offsets`` (planted cells give
    cam ~ coordmap_3d[z, y, x]) plus a shift of the output bias of betas[10] (transformer.6 row 142, bev/model.py:116) so
    that some planted people are babies (betas[10] > 0.8 selects SMIL, bev/post_parser.py:260-268); the default shift
    puts the threshold in the widest gap of the crowd-mode fixture's values."""
    out = bev_damp_cam_offsets(bev_state_dict(seed))
    b = np.array(out["transformer.6.bias"], np.float32, copy=True)
    b[142] += np.float32(beta10_shift)
    out["transformer.6.bias"] = b
    return out
