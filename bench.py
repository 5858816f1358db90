#!/usr/bin/env python
"""bench.py - ROMP hot-path throughput on B200 (contract: see the task statement / DESIGN.md section 6).

    python bench.py --gpus 1 --steps 10 --warmup 3                 # our arm  (frames/s, cfg2)
    python bench.py --impl reference --steps 2 --warmup 1          # reference arm: the CPU path on host cores
    torchrun --nproc-per-node N bench.py --gpus N ...              # frames sharded over N ranks (weak scaling)

A step = one pass of the whole hot path (backbone+heads -> parse -> SMPL -> projection) over one batch of 64
synthetic 512x512 frames per GPU (BASELINE.json configs[1]).  Weights are seeded synthetic parameters with
the reference's schema; person detections are planted (1..10 per frame) because random weights detect nobody.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_FRAME = 85_710_602_240          # ROMP HRNet-32 + heads @512x512 (SURVEY 8d, hooked on the reference)
SMPL_BYTES_PER_PERSON = 83_860
BATCH = 64
DUMP_LIMIT_BYTES = 63_000_000           # --dump-outputs stays under 64 MB, .npy headers included


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16=d.get("bf16_tflops_sustained", 1472.5), bf16_burst=d.get("bf16_tflops", 1717.1),
                    hbm=d.get("hbm_gbs", 6484.3), src="measured")
    return dict(bf16=1400.0, bf16_burst=1590.0, hbm=6650.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def oracle_fps(sample_frames, threads):
    """The reference's CPU path (oracle port: fp32 torch-CPU restatement) on `sample_frames` frames."""
    import torch
    from oracle import romp_oracle as O
    from romp_b200 import synth
    torch.set_num_threads(threads)
    sd, pack = synth.romp_state_dict(0), synth.smpl_pack(0)
    frames = synth.synthetic_frames(sample_frames, seed=0)
    planted, _ = synth.plant_centers(sample_frames, seed=0)
    t0 = time.perf_counter()
    out = O.romp_forward(sd, pack, frames, center_override=planted)
    dt = time.perf_counter() - t0
    return sample_frames / dt, 0 if out is None else len(out["cam"])


def best_thread_count():
    """torch CPU convs do not scale to every core of a big host: time one frame at a few thread counts and keep
    the fastest ("all the host threads it can use")."""
    n = os.cpu_count() or 8
    cands = sorted({n, max(8, n // 2), max(8, n // 4), min(n, 32)}, reverse=True)
    oracle_fps(1, cands[0])                       # first-touch warm-up (weights generation, allocator)
    best = max(cands, key=lambda t: oracle_fps(1, t)[0])
    return best


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = best_thread_count()
    sample = 4
    for _ in range(args.warmup):
        oracle_fps(1, cores)
    t0 = time.perf_counter()
    persons = 0
    for _ in range(args.steps):
        _, n = oracle_fps(sample, cores)
        persons += n
    dt = time.perf_counter() - t0
    fps = args.steps * sample / dt
    line = {
        "impl": "reference", "metric": "frames/sec 512x512 ROMP-HRNet32 (whole hot path)", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg2 ROMP HRNet-32 512x512, planted 1..10 persons/frame", "sample_frames_per_step": sample},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} frames/step of the cfg2 workload through oracle/romp_oracle.py (torch CPU fp32)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "persons_per_step": persons / max(args.steps, 1),
    }
    emit(line)


def _events():
    import torch
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def dump_outputs(path, arrays):
    """Write the result arrays of the last timed step as path/<name>.npy so that two builds can be compared output for
    output: integer arrays as float64 (exact), the rest as float32.  ``arrays`` maps names to numpy arrays or device
    tensors that all index persons along their first axis.  Above DUMP_LIMIT_BYTES in all, every array keeps the same
    rows: a seeded sample of the persons, in ascending order, taken on the device before the read-back."""
    import torch
    os.makedirs(path, exist_ok=True)
    if not arrays:
        return
    dtypes = {}
    for name, v in arrays.items():
        dt = (v[:0].cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)).dtype
        dtypes[name] = np.dtype(np.float64 if dt == np.float64 or dt.kind in "iub" else np.float32)
    n = len(next(iter(arrays.values())))
    row_bytes = sum(int(np.prod(v.shape[1:])) * dtypes[name].itemsize for name, v in arrays.items())
    rows = None
    if n * row_bytes > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // row_bytes, replace=False))
    for name, v in arrays.items():
        dt = dtypes[name]
        if rows is not None:
            v = v[torch.from_numpy(rows).to(v.device)] if isinstance(v, torch.Tensor) else v[rows]
        if isinstance(v, torch.Tensor):
            v = v.cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(v, dtype=dt))


def committed_traffic(precision):
    """DRAM bytes per conv-graph replay (batch 64) from the committed ncu capture of this bench command
    (profiles/r02_ncu_step_bytes.json, written by tools/ncu_step_bytes.py from an `ncu --metrics dram__bytes_*` pass)."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_step_bytes.json")
    if not os.path.exists(p):
        return None
    try:
        d = json.load(open(p))
        return d.get(precision, {}).get("conv_graph_dram_bytes_per_step")
    except Exception:
        return None


def pytorch_cuda_comparator(B, time_cap_s=60.0):
    """SURVEY 8d-ii comparator: the reference's conv path (oracle restatement, pinned to the reference's modules by the
    golden fixtures; /root/reference does not exist on the GPU box) as plain PyTorch eager on the SAME GPU with cuDNN,
    default flags (cudnn.allow_tf32 = True: TF32 convs, exactly what the reference runs), batch B.  A reported baseline."""
    import torch
    from oracle import romp_oracle as O
    from romp_b200 import synth
    dev = torch.device("cuda", torch.cuda.current_device())
    autotune = os.environ.get("B200ROMP_COMPARATOR_AUTOTUNE") == "1"     # cudnn.benchmark=True costs ~4 min of autotuning
    torch.backends.cudnn.benchmark = autotune
    sd = {k: torch.from_numpy(np.asarray(v)).to(dev) for k, v in synth.romp_state_dict(0).items()}
    frames = torch.from_numpy(synth.synthetic_frames(B, seed=0)).to(dev).float()
    t_start = time.perf_counter()
    with torch.no_grad():
        O.romp_maps(sd, frames)                              # warm-up (cuDNN heuristics / autotune, allocator)
        torch.cuda.synchronize()
        e0, e1 = _events()
        iters, total = 0, 0.0
        while iters < 5 and time.perf_counter() - t_start < time_cap_s:
            e0.record()
            O.romp_maps(sd, frames)
            e1.record()
            torch.cuda.synchronize()
            total += e0.elapsed_time(e1)
            iters += 1
    del sd, frames
    torch.cuda.empty_cache()
    if iters == 0:
        return None
    ms = total / iters
    return {"value": B / ms * 1e3, "unit": "frames/s", "ms_per_batch": ms, "iters": iters, "batch": B,
            "what": "oracle/romp_oracle.py romp_maps (HRNet-32 + heads only: no parse/SMPL/projection) under torch eager + cuDNN on "
                    "cuda:0, fp32 tensors, cudnn.allow_tf32=%s, cudnn.benchmark=%s" % (torch.backends.cudnn.allow_tf32, autotune)}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from romp_b200 import ROMP, romp_settings, shard, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B = args.batch
    steps, warm = args.steps, max(args.warmup, 3)
    sd, pack = synth.romp_state_dict(0), synth.smpl_pack(0)
    frames_host = torch.from_numpy(synth.synthetic_frames(B, seed=rank)).pin_memory()       # uint8 [B,512,512,3]
    planted_np, truth = synth.plant_centers(B, seed=rank)
    planted = torch.from_numpy(planted_np).cuda()
    persons = sum(len(t) for t in truth)
    frames_dev = frames_host.cuda()
    offsets = [0, 512, 0, 512, 512, 512]
    peaks = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def build(precision):
        s = romp_settings(["--GPU", str(local), "--precision", precision, "--max_batch", str(B)])
        return ROMP(s, state_dict=sd, smpl_pack=pack)

    def device_legs(model, gather, k_steps):
        """(seconds for k_steps whole-path steps incl. the per-step all-gather when sharded, seconds for k_steps conv graphs)"""
        stream = model.stream

        def step():
            with torch.cuda.stream(stream):
                model.run_maps(frames_dev)
                model.run_post(B, offsets, planted)
                if gather is not None:
                    # the single collective of the sharded path, every step, inside the timed region: device-side pack of the
                    # packed records + one NCCL all-gather on the gather's side stream (overlaps the next step's kernels)
                    fields, count = model.record_fields()
                    h = gather.submit(fields, count, rank * B, rows_hint=B * 10)
                    stream.wait_event(h["packed"])
                    return h
            return None

        for _ in range(warm):
            h = step()
            model.collect(to_numpy=False)
            if h is not None:
                gather.counts(h)
        barrier()
        e0, e1 = _events()
        e0.record(stream)
        h = None
        for _ in range(k_steps):
            h = step()
        if h is not None:
            gather.wait(h, stream)                  # the last all-gather (and, in stream order, all before it) is done
        e1.record(stream)
        barrier()
        t_dev = e0.elapsed_time(e1) / 1e3
        n0, n1 = _events()
        n0.record(stream)
        for _ in range(k_steps):
            with torch.cuda.stream(stream):
                model.run_maps(frames_dev)
        n1.record(stream)
        barrier()
        return t_dev, n0.elapsed_time(n1) / 1e3

    model = build(args.precision)
    gather = shard.ShardGather(world, model.record_layout(), capacity=model.cap, rows_hint=B * 10) if world > 1 else None
    # warm the streaming path (pinned read-back mirrors of both slots, per-slot frame buffers, CUDA graphs, NCCL buffers)
    for r in model.forward_batches((frames_host for _ in range(3)), center_override=planted, gather=gather, frame_offset=rank * B):
        if gather is not None:
            gather.counts(r[1])
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # ---------------- device-resident timing (value) + net-only timing (roofline) --------------------------
    t_dev, t_net = device_legs(model, gather, steps)
    # ---------------- end to end through the public API with host buffers --------------------------------
    # public streaming API: per step H2D of that step's pinned frames, the whole path, D2H of THIS rank's result dict; sharded:
    # plus pack + all-gather of every step's records, whose gathered headers are read by every rank (device-resident records)
    out, gathered_persons = None, 0
    barrier()
    w0 = time.perf_counter()
    for r in model.forward_batches((frames_host for _ in range(steps)), center_override=planted, to_numpy=True, gather=gather,
                                   frame_offset=rank * B):
        if gather is not None:
            out, h = r
            gathered_persons = sum(gather.counts(h)[0])      # every rank reads the gathered headers; the records stay on the device
        else:
            out = r
    barrier()
    t_e2e = time.perf_counter() - w0
    d2h = 0 if out is None else int(sum(v.nbytes for v in out.values()))
    times = torch.tensor([t_dev, t_net, t_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    t_dev, t_net, t_e2e = times.tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)     # rank 0's shard of the last end-to-end step
    fps = world * B * steps / t_dev
    net_tflops = B * steps * FLOP_PER_FRAME / t_net / 1e12          # per GPU
    nb, _ = model._net(2)
    desc = nb.describe()
    n_launch = nb.lib.b200romp_net_num_launches(nb.net)
    peak_key = "bf16_burst" if args.precision == "bf16" else "bf16_burst"
    peak = peaks[peak_key] * (1.0 if args.precision == "bf16" else 0.5)
    traffic = committed_traffic(args.precision)
    line = {
        "metric": "frames/sec 512x512 ROMP-HRNet32 (whole hot path)", "value": fps, "unit": "frames/s",
        "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": t_dev / steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"bf16": "bf16", "tf32": "tf32", "fp32": "f32"}[args.precision], "data": "synthetic",
        "config": {"workload": "cfg2 ROMP HRNet-32, batch 64 x 512x512 uint8 frames per GPU, planted 1..10 persons/frame",
                   "batch_per_gpu": B, "persons_per_gpu_step": persons, "parallelism": f"frames sharded x{world}",
                   "collective": None if world == 1 else "one NCCL all_gather_into_tensor of packed per-person records per step, inside "
                                 "the timed region of `value` and of `e2e` (%d rows x %d B per rank)" % (1 + B * 10, model.record_layout().row_bytes),
                   "l2": "working set per step (activations > 1 GB) exceeds the 126 MB L2; no explicit flush"},
        "persons_per_sec": world * persons * steps / t_dev,
        "e2e": {"value": world * B * steps / t_e2e, "unit": "frames/s",
                "h2d_bytes_per_step": int(frames_host.numel()), "d2h_bytes_per_step": d2h,
                "note": "per rank: H2D of its frames, D2H of its own shard's result dict" +
                        ("; all ranks' records all-gathered on the device every step (%d persons seen by rank 0)" % gathered_persons if world > 1 else "")},
        "gpu_launches": (n_launch + 2 + 4 + 2 + (1 if world > 1 else 0)) * steps,   # per timed device pass: conv graph, parse 2, SMPL 4 (pose, blend GEMM, skinning GEMM, joints), projection 2, pack
        "roofline": {"bound": "tensor", "achieved": net_tflops, "peak": peak, "unit": "TFLOP/s",
                     "frac": net_tflops / peak, "frac_of_sustained_peak": net_tflops / (peaks["bf16"] * (1.0 if args.precision == "bf16" else 0.5)),
                     "traffic": traffic,
                     "algorithmic_flop_per_launch": B * FLOP_PER_FRAME,
                     "peak_source": peaks["src"] + (" bf16 burst (cuBLAS 8192^3)" if args.precision == "bf16" else " bf16 burst / 2 (TF32 issues at half the bf16 rate)"),
                     "kernel": "conv graph (backbone+heads), one CUDA-graph replay = %d tcgen05 / %d simt ops; traffic = ncu dram bytes per replay"
                               % (desc.count("tcgen05"), desc.count("simt   "))},
    }
    extra = {}
    if world == 1 and not args.no_extra:
        # ---- a >= 2 s sustained window of the same device loop (the K-step window above is short)
        n_sus = max(steps, int(2.2 / (t_dev / steps)) + 1)
        ts, _ = device_legs(model, None, n_sus)
        extra["sustained"] = {"frames_per_s": B * n_sus / ts, "steps": n_sus, "seconds": ts}
        # ---- the other precisions of the conv engine on the same workload (TF32 = the reference's own GPU arithmetic)
        del model
        torch.cuda.empty_cache()
        for prec in [p for p in ("tf32",) if p != args.precision]:
            m2 = build(prec)
            k2 = max(3, min(steps, 10))
            td, tn = device_legs(m2, None, k2)
            tfl = B * k2 * FLOP_PER_FRAME / tn / 1e12
            nb2, _ = m2._net(2)
            d2 = nb2.describe()
            extra[prec] = {"frames_per_s": B * k2 / td, "ms_per_step": td / k2 * 1e3, "conv_graph_tflops": tfl,
                           "frac_of_tf32_peak": tfl / (peaks["bf16_burst"] * 0.5), "steps": k2,
                           "ops": "%d tcgen05-tf32 / %d simt" % (d2.count("tc-tf32"), d2.count("simt   ")),
                           "traffic": committed_traffic(prec)}
            del m2
            torch.cuda.empty_cache()
        try:
            extra["cfg5_smpl"] = run_smpl(args, emit_line=False)
            extra["cfg3_bev"] = run_bev(args, emit_line=False)
        except Exception as e:                       # an extra must never cost the main line
            extra["error"] = repr(e)
        try:
            cmp_ = pytorch_cuda_comparator(B)
            if cmp_:
                line["pytorch_cuda_baseline"] = cmp_
                line["vs_pytorch_cuda"] = fps / cmp_["value"]
                if "tf32" in extra:
                    extra["tf32"]["vs_pytorch_cuda"] = extra["tf32"]["frames_per_s"] / cmp_["value"]
        except Exception as e:
            extra["comparator_error"] = repr(e)
    line["clocks"] = sampler.finish()
    if extra:
        line["extra"] = extra
    if world == 1 and not args.no_cpu_baseline:
        cores = best_thread_count()
        v, _ = oracle_fps(4, cores)
        line["cpu_baseline"] = {"value": v, "unit": "frames/s", "cores": cores, "kind": "port",
                                "sample": "4 frames of the cfg2 workload through oracle/romp_oracle.py (torch CPU fp32), after 1 warm-up frame"}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_smpl(args, emit_line=True):
    """BASELINE.json configs[4]: SMPL-only, 65,536 persons, GB/s against the HBM roofline (83,860 B/person)."""
    import torch
    from romp_b200 import synth
    from romp_b200.main import SMPLParser
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    n = args.persons
    sm = SMPLParser(synth.smpl_pack(0), torch.cuda.current_device())
    g = torch.Generator(device="cpu").manual_seed(0)
    betas = torch.randn(n, 10, generator=g).cuda()
    thetas = (torch.randn(n, 72, generator=g) * 0.3).cuda()
    verts = torch.empty(n, 6890, 3, device="cuda"); joints = torch.empty(n, 71, 3, device="cuda")
    ws = torch.empty(n, sm.ws_floats, device="cuda")
    st = torch.cuda.Stream()
    run = lambda: sm.forward(betas, thetas, n, None, False, ws, verts, joints, st.cuda_stream)
    steps = args.steps if emit_line else max(3, min(args.steps, 10))
    for _ in range(max(args.warmup, 3)):
        run()
    st.synchronize()
    e0, e1 = _events()
    e0.record(st)
    for _ in range(steps):
        run()
    e1.record(st)
    st.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if emit_line and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"verts": verts, "joints": joints})
    peaks = measured_peaks()
    gbs = n * SMPL_BYTES_PER_PERSON / ms / 1e6
    res = {
        "metric": "persons/sec SMPL forward (verts + 71 joints)", "value": n / ms * 1e3, "unit": "persons/s", "n_gpus": 1,
        "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg5 SMPL-only, %d persons, betas~N(0,1), thetas~N(0,0.3), synthetic SMPL pack" % n},
        "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs / peaks["hbm"],
                     "traffic": None, "peak_source": peaks["src"], "kernel": "smpl_pose + smpl_blend_tc (tcgen05 GEMM) + smpl_skin_tc (tcgen05 GEMM) + smpl_joints",
                     "algorithmic_bytes_per_launch": n * SMPL_BYTES_PER_PERSON},
        "gpu_launches": 4 * steps}
    del verts, joints, ws
    torch.cuda.empty_cache()
    if emit_line:
        emit(res)
    return res


def run_bev(args, emit_line=True):
    """BASELINE.json configs[2]: BEV HRNet-32 (+ bird's-eye-view head), batch 32 x 512x512, planted 3-D detections."""
    import torch
    from romp_b200 import synth
    from romp_b200.bev import BEV, bev_settings
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    B = args.batch if args.batch != BATCH else 32
    s = bev_settings(["--precision", args.precision, "--max_batch", str(B)])
    m = BEV(s, state_dict=synth.bev_damp_cam_offsets(synth.bev_state_dict(0)), smpla_pack=synth.smpl_pack(0, num_betas=11), smil_pack=synth.smpl_pack(1))
    frames_host = torch.from_numpy(synth.synthetic_frames(B, seed=0)).pin_memory()
    frames_dev = frames_host.cuda()
    vol_np, persons = synth.plant_centers_3d(B, seed=0)
    vol = torch.from_numpy(vol_np).cuda()
    off = [0, 512, 0, 512, 512, 512]
    steps = args.steps if emit_line else max(3, min(args.steps, 10))

    def step():
        with torch.cuda.stream(m.stream):
            m.run_model(frames_dev, vol)
            m.run_post(B, off)
    for _ in range(max(args.warmup, 3)):
        step()
        m.collect(False)
    e0, e1 = _events()
    torch.cuda.synchronize()
    e0.record(m.stream)
    for _ in range(steps):
        step()
    e1.record(m.stream)
    torch.cuda.synchronize()
    t_dev = e0.elapsed_time(e1) / 1e3
    w0 = time.perf_counter()
    out = None
    for _ in range(steps):
        out = m.forward_batch(frames_host, center3d_override=vol)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - w0
    if emit_line and args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    peaks = measured_peaks()
    fps = B * steps / t_dev
    res = {
        "metric": "frames/sec 512x512 BEV-HRNet32 (whole hot path)", "value": fps, "unit": "frames/s", "n_gpus": 1,
        "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": t_dev / steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": "cfg3 BEV HRNet-32 + BEV head, batch %d x 512x512 uint8, planted 1..10 persons/frame "
                               "(synthetic weights with damped cam offsets so that planted people survive BEV's post-filters)" % B,
                   "persons_planted": persons, "persons_out": 0 if out is None else int(len(out["cam"]))},
        "e2e": {"value": B * steps / t_e2e, "unit": "frames/s", "h2d_bytes_per_step": int(frames_host.numel()),
                "d2h_bytes_per_step": 0 if out is None else int(sum(v.nbytes for v in out.values()))},
        "roofline": {"bound": "tensor", "achieved": fps * 96_851_656_704 / 1e12, "peak": peaks["bf16_burst"], "unit": "TFLOP/s",
                     "frac": fps * 96_851_656_704 / 1e12 / peaks["bf16_burst"], "traffic": None, "peak_source": peaks["src"] + " bf16 burst",
                     "kernel": "whole BEV step (conv graphs + BEV stages); 96.85 GFLOP/frame (SURVEY 8d)"}}
    del m, vol, frames_dev
    torch.cuda.empty_cache()
    if emit_line:
        emit(res)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", type=str, default="romp", choices=["romp", "bev", "smpl"],
                    help="romp = the contract's default (cfg2); bev = cfg3; smpl = cfg5 microbenchmark")
    ap.add_argument("--persons", type=int, default=65536)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", type=str, default="bf16", choices=["bf16", "tf32", "fp32"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--no-extra", dest="no_extra", action="store_true",
                    help="skip the extra legs of the N=1 line (sustained window, TF32 engine, cfg3/cfg5, PyTorch-CUDA comparator)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write the results of the last one as DIR/<name>.npy (float32 / float64, "
                         "at most 64 MB: a seeded sample of the persons when the whole is larger)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours")
    # stdout carries exactly ONE line (the JSON): library chatter written to file descriptor 1 while we run (NCCL prints
    # its version banner there on the first communicator) is diverted to stderr; emit() restores the real stdout.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "smpl":
        run_smpl(args)
    elif args.workload == "bev":
        run_bev(args)
    else:
        run_ours(args)


_REAL_STDOUT = None


def emit(line):
    """print the result line on the process's original stdout"""
    text = json.dumps(line) + "\n"
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        sys.stdout.write(text)
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, text.encode())


if __name__ == "__main__":
    main()
