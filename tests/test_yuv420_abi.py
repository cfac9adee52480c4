"""The FD_YUV420_* layouts and the *_yuv420 entry points of include/fd_b200.h, and their Rust and ctypes mirrors."""
import importlib.util
import os
import re

from conftest import ROOT

BASES = ("fd_preprocess_batch", "fd_align_batch", "fd_align_detections", "fd_select_detections", "fd_align_selected")
LAYOUTS = {"FD_YUV420_NV12": 0, "FD_YUV420_NV21": 1, "FD_YUV420_I420": 2, "FD_YUV420_YV12": 3}


def _gen():
    spec = importlib.util.spec_from_file_location("gen_rust_ffi", os.path.join(ROOT, "scripts", "gen_rust_ffi.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    return gen, open(os.path.join(ROOT, "include", "fd_b200.h")).read()


def _rust():
    return open(os.path.join(ROOT, "rust", "src", "ffi.rs")).read()


def test_entry_points_take_the_nv12_parameters_and_a_layout():
    gen, src = _gen()
    _, _, _, _, funcs = gen.parse_header(src)
    params = {name: plist for name, _, plist in funcs}
    rets = {name: ret for name, ret, _ in funcs}
    rs = _rust()
    for base in BASES:
        nv, yuv = params[base + "_nv12"], params[base + "_yuv420"]
        assert yuv == nv[:1] + [("frames", nv[1][1]), ("layout", "i32")] + nv[2:], base
        assert nv[1][0] == "frames" and rets[base + "_yuv420"] == rets[base + "_nv12"] == "int"
        m = re.search(r"pub fn %s_yuv420\((.*?)\) -> c_int;" % base, rs)
        assert m and "frames: *const fd_frame_nv12, layout: i32, " in m.group(1), base


def test_layout_constants_agree_across_header_rust_and_python():
    from rs_face_detection_b200 import ffi
    gen, src = _gen()
    _, enums, _, _, _ = gen.parse_header(src)
    anon = {k: v for name, vals in enums if name is None for k, v in vals}
    rs = _rust()
    for k, v in LAYOUTS.items():
        assert anon[k] == v, k
        assert "pub const %s: c_int = %d;" % (k, v) in rs, k
        assert getattr(ffi, k) == v, k


def test_python_mirrors_every_entry_point():
    from rs_face_detection_b200 import Context, ffi
    for base in BASES:
        assert base + "_yuv420" in ffi.SYMBOLS
        assert callable(getattr(Context, base[len("fd_"):] + "_yuv420"))
