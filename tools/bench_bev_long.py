"""Wide images per second of BEV's crowd mode (BEV.process_long_image, bev/main.py:184-258) on one GPU.

    python tools/bench_bev_long.py [--precision bf16] [--iters 20] [--warmup 3]

Workloads: 512x1024 (14 crops) and 512x2048 (24 crops) synthetic images, one planted person per crop (synthetic
weights detect nobody on their own).  ``batched`` is the library as shipped: the crops of an image go through the BEV
net as batches of <= max_batch (32), every per-crop and merge step on the device, one host sync per image.
``crop_by_crop`` is the same library driven with max_batch 1, i.e. one crop at a time like the reference's loop.
Each timed call ends with the host sync that reads the person count, so wall-clock time per call is device time plus
launch overhead.  Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from romp_b200 import synth  # noqa: E402
from romp_b200.bev import BEV, bev_settings, long_image_plan  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def rate(model, img, vol, iters, warmup):
    for _ in range(warmup):
        out = model.process_long_image(img, center3d_override=vol)
    t0 = time.perf_counter()
    for _ in range(iters):
        out = model.process_long_image(img, center3d_override=vol)
    dt = time.perf_counter() - t0
    return iters / dt, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--precision", default="bf16", choices=["bf16", "tf32", "fp32"])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_bev_long needs a GPU"
    sd, pa, ps = synth.bev_crowd_state_dict(0), synth.smpl_pack(0, num_betas=11), synth.smpl_pack(1)
    models = {mb: BEV(bev_settings(["--precision", a.precision, "--max_batch", str(mb)]), state_dict=sd, smpla_pack=pa, smil_pack=ps)
              for mb in (32, 1)}
    res = []
    for h, w in ((512, 1024), (512, 2048)):
        S = len(long_image_plan(h, w, 0.8)[0])
        img = synth.synthetic_wide_image(h, w, 0)
        vol = torch.from_numpy(synth.bev_planted_crops(S, [(c, 28 + c % 6, 64, 64, 0.5 + 0.01 * c) for c in range(S)], 0)).cuda()
        fast, out_b = rate(models[32], img, vol, a.iters, a.warmup)
        slow, out_s = rate(models[1], img, vol, max(3, a.iters // 2), 1)
        same = out_b is not None and out_s is not None and all(np.array_equal(out_b[k], out_s[k]) for k in out_b)
        res.append({"shape": f"{h}x{w}", "crops": S, "people": 0 if out_b is None else len(out_b["cam"]),
                    "batched_images_per_s": round(fast, 2), "batched_ms_per_image": round(1e3 / fast, 3),
                    "crop_by_crop_images_per_s": round(slow, 2), "speedup": round(fast / slow, 2), "outputs_identical": same})
    print(json.dumps({"workload": "bev_long", "precision": a.precision, "gpu": gpu_info(), "iters": a.iters, "results": res}))


if __name__ == "__main__":
    main()
