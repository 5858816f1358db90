"""ctypes binding of libb200romp.so (C ABI declared in include/b200romp.h).

The library is the product: if it is missing or fails to load this module raises - there is no
PyTorch/CPU fallback path anywhere in ``romp_b200``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LIB_PATH = os.path.join(HERE, "lib", "libb200romp.so")
CSRC = os.path.join(HERE, "csrc")
SOURCES = ["net.cu", "conv_simt.cu", "conv_tc.cu", "conv_tc_s2.cu", "conv_stem_tc.cu", "conv_tc_2cta.cu", "conv1d_tc.cu", "parse.cu", "smpl.cu", "smpl_blend_tc.cu", "project.cu", "bev.cu", "pack.cu", "preproc.cu", "temporal.cu", "resnet_ops.cu"]

F32, BF16, U8 = 0, 1, 2
ENGINE_AUTO, ENGINE_SIMT, ENGINE_TCGEN05, ENGINE_TF32 = 0, 1, 2, 3


class ConvDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "in_", "in_c_off", "out", "out_c_off", "res", "res_c_off", "res_broadcast", "cin", "cout",
        "ksize", "stride", "relu", "upsample", "input_norm", "pow_channel", "engine")]


class SumDesc(C.Structure):
    _fields_ = [("out", C.c_int), ("base", C.c_int), ("n_terms", C.c_int), ("term", C.c_int * 4), ("up", C.c_int * 4),
                ("relu", C.c_int), ("term_c_off", C.c_int * 4)]


class BevWeights(C.Structure):
    _fields_ = [(n, C.POINTER(C.c_float)) for n in (
        "center_ref", "cam_ref", "coordmap", "anchors", "embed", "w0", "b0", "w1", "b1", "w2", "b2")]


NVCC_FLAGS = ["-Xcompiler", "-fPIC", "-std=c++17", "-O3", "-lineinfo", "-gencode", "arch=compute_100a,code=sm_100a"]
OBJ_DIR = os.path.join(HERE, "lib", "obj")


def _nvcc():
    return os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def nvcc_command(out_path=LIB_PATH):
    """The one-shot equivalent of build(): every source -> one sm_100a shared library."""
    return [_nvcc(), "-shared"] + NVCC_FLAGS + ["-o", out_path] + [os.path.join(CSRC, s) for s in SOURCES]


def _headers_mtime():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hs.append(os.path.join(ROOT, "include", "b200romp.h"))
    return max(os.path.getmtime(h) for h in hs)


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", "b200romp.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=True):
    """Compile every CUDA source for sm_100a (nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo) into
    romp_b200/lib/libb200romp.so (in-tree).  One object per source, compiled in parallel and reused while the
    source and the headers are unchanged."""
    if not force and not needs_build():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(OBJ_DIR, exist_ok=True)
    hdr_t = _headers_mtime()
    jobs = []
    for s in SOURCES:
        src, obj = os.path.join(CSRC, s), os.path.join(OBJ_DIR, s.replace(".cu", ".o"))
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_t):
            jobs.append([_nvcc(), "-c"] + NVCC_FLAGS + ["-o", obj, src])
    if verbose:
        for j in jobs:
            print("[romp_b200] " + " ".join(j), file=sys.stderr)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if verbose and r.stderr.strip():
            print(r.stderr, file=sys.stderr)

    with ThreadPoolExecutor(max_workers=min(len(jobs) or 1, os.cpu_count() or 4)) as ex:
        list(ex.map(run, jobs))
    link = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH] + [os.path.join(OBJ_DIR, s.replace(".cu", ".o")) for s in SOURCES]
    if verbose:
        print("[romp_b200] " + " ".join(link), file=sys.stderr)
    subprocess.run(link, check=True)
    return LIB_PATH


_lib = None


def _sig(fn, restype, *argtypes):
    fn.restype = restype
    fn.argtypes = list(argtypes)


def load():
    """dlopen the library and declare every prototype of include/b200romp.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(romp_b200 has no fallback path without its CUDA library)")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    vp, i32, f32, i64 = C.c_void_p, C.c_int, C.c_float, C.c_longlong
    fp, ip, lp = C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_longlong)
    _sig(lib.b200romp_version, i32)
    _sig(lib.b200romp_last_error, C.c_char_p)
    _sig(lib.b200romp_device_info, i32, ip, ip, ip)
    _sig(lib.b200romp_net_create, vp, i32)
    _sig(lib.b200romp_net_destroy, None, vp)
    _sig(lib.b200romp_net_add_tensor, i32, vp, i32, i32, i32, i32, i32, i32)
    _sig(lib.b200romp_net_add_const_tensor, i32, vp, i32, i32, i32, i32, vp)
    _sig(lib.b200romp_net_add_conv, i32, vp, C.POINTER(ConvDesc), fp, fp)
    _sig(lib.b200romp_net_add_sum, i32, vp, C.POINTER(SumDesc))
    _sig(lib.b200romp_net_set_lane, i32, vp, i32, i32)
    _sig(lib.b200romp_net_add_maxpool, i32, vp, i32, i32)
    _sig(lib.b200romp_net_finalize, i32, vp, i32)
    _sig(lib.b200romp_net_bind, i32, vp, i32, vp)
    _sig(lib.b200romp_net_run, i32, vp, i32, vp)
    _sig(lib.b200romp_net_read_tensor, i32, vp, i32, i32, vp, vp)
    _sig(lib.b200romp_net_describe, i32, vp, C.c_char_p, i32)
    _sig(lib.b200romp_net_num_launches, i32, vp)
    _sig(lib.b200romp_net_workspace_bytes, i64, vp)
    _sig(lib.b200romp_net_profile, i32, vp, i32, i32, fp, vp)
    _sig(lib.b200romp_net_read_stamps, i32, vp, vp, i32)
    _sig(lib.b200romp_conv2d, i32, C.POINTER(ConvDesc), fp, fp, vp, i32, i32, i32, i32, vp, i32, i32, i32, vp, i32, i32, vp)
    _sig(lib.b200romp_parse, i32, vp, vp, i32, i32, i32, f32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp)
    _sig(lib.b200romp_parse_workspace_bytes, i64, i32)
    _sig(lib.b200romp_smpl_create, vp, i32, i32, fp, fp, fp, fp, fp, lp, lp, fp, fp)
    _sig(lib.b200romp_smpl_destroy, None, vp)
    _sig(lib.b200romp_smpl_workspace_floats, i32)
    _sig(lib.b200romp_smpl_forward, i32, vp, vp, i32, vp, i32, vp, i32, vp, vp, vp, vp)
    _sig(lib.b200romp_project, i32, vp, vp, vp, i32, vp, fp, vp, vp, vp, vp, vp)
    _sig(lib.b200romp_bev_create, vp, i32, C.POINTER(BevWeights))
    _sig(lib.b200romp_bev_destroy, None, vp)
    _sig(lib.b200romp_bev_bv_input, i32, vp, vp, i32, i32, i32, vp, i32, vp)
    _sig(lib.b200romp_bev_center3d, i32, vp, vp, vp, i32, i32, vp, vp, vp)
    _sig(lib.b200romp_bev_parse_workspace_bytes, i64, i32)
    _sig(lib.b200romp_bev_parse3d, i32, vp, i32, f32, i32, vp, vp, vp, vp, vp, vp)
    _sig(lib.b200romp_bev_regress, i32, vp, vp, vp, i32, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp)
    _sig(lib.b200romp_bev_post, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, fp, f32, f32, f32, vp, vp, vp, vp, vp)
    _sig(lib.b200romp_gather_rows, i32, vp, i32, vp, vp, i32, vp, vp)
    _sig(lib.b200romp_gather_rows_at, i32, vp, i32, vp, vp, vp, i32, vp, vp)
    _sig(lib.b200romp_bev_long_crops, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, vp, i32, i32, i32, i32, i32, f32, f32,
         vp, vp, vp, vp, vp, vp, vp, i32, vp)
    _sig(lib.b200romp_bev_long_merge, i32, vp, vp, vp, i32, vp, i32, i32, f32, f32, vp, vp, vp, vp, vp, vp)
    _sig(lib.b200romp_tracks_create, vp, i32, i32)
    _sig(lib.b200romp_tracks_destroy, None, vp)
    _sig(lib.b200romp_tracks_reset, i32, vp, i32, vp)
    _sig(lib.b200romp_one_euro_smooth, i32, vp, vp, i32, vp, vp, vp, i32, i32, vp, f32, f32, vp)
    _sig(lib.b200romp_preprocess_bgr, i32, vp, i32, i32, i32, i32, vp, fp, vp)
    _sig(lib.b200romp_preprocess_crops_bgr, i32, vp, i32, i32, i32, i32, vp, i32, i32, i32, vp, vp)
    _sig(lib.b200romp_pack_rows, i32, C.POINTER(vp), ip, i32, vp, i32, i32, i32, i32, vp, i32, vp)
    if lib.b200romp_version() != 200:
        raise RuntimeError("libb200romp.so version mismatch - rebuild")
    _lib = lib
    return lib


def check(rc, what=""):
    if rc is None or (isinstance(rc, int) and rc < 0):
        msg = load().b200romp_last_error().decode()
        raise RuntimeError(f"libb200romp {what} failed ({rc}): {msg}")
    return rc


EXPORTS = [
    "b200romp_version", "b200romp_last_error", "b200romp_device_info", "b200romp_net_create",
    "b200romp_net_destroy", "b200romp_net_add_tensor", "b200romp_net_add_const_tensor", "b200romp_net_add_conv",
    "b200romp_net_add_sum", "b200romp_net_set_lane", "b200romp_net_add_maxpool",
    "b200romp_net_finalize", "b200romp_net_bind", "b200romp_net_run", "b200romp_net_read_tensor",
    "b200romp_net_describe", "b200romp_net_num_launches", "b200romp_net_workspace_bytes", "b200romp_net_profile", "b200romp_net_read_stamps",
    "b200romp_conv2d",
    "b200romp_parse", "b200romp_parse_workspace_bytes", "b200romp_smpl_create", "b200romp_smpl_destroy",
    "b200romp_smpl_workspace_floats", "b200romp_smpl_forward", "b200romp_project",
    "b200romp_bev_create", "b200romp_bev_destroy", "b200romp_bev_bv_input", "b200romp_bev_center3d",
    "b200romp_bev_parse_workspace_bytes", "b200romp_bev_parse3d", "b200romp_bev_regress", "b200romp_bev_post",
    "b200romp_gather_rows", "b200romp_pack_rows", "b200romp_preprocess_bgr", "b200romp_tracks_create", "b200romp_tracks_destroy",
    "b200romp_tracks_reset", "b200romp_one_euro_smooth", "b200romp_gather_rows_at", "b200romp_bev_long_crops",
    "b200romp_bev_long_merge", "b200romp_preprocess_crops_bgr",
]
