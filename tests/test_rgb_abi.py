"""The FD_RGB_* layouts and the *_rgb entry points of include/fd_b200.h, and their Rust and ctypes mirrors."""
import importlib.util
import os
import re

from conftest import ROOT

BASES = ("fd_preprocess_batch", "fd_align_batch", "fd_align_detections", "fd_select_detections", "fd_align_selected")
LAYOUTS = {"FD_RGB_RGB24": 0, "FD_RGB_RGBA": 1, "FD_RGB_BGRA": 2, "FD_RGB_GRAY8": 3}


def _gen():
    spec = importlib.util.spec_from_file_location("gen_rust_ffi", os.path.join(ROOT, "scripts", "gen_rust_ffi.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    return gen, open(os.path.join(ROOT, "include", "fd_b200.h")).read()


def _rust():
    return open(os.path.join(ROOT, "rust", "src", "ffi.rs")).read()


def test_entry_points_take_the_bgr_parameters_and_a_layout():
    gen, src = _gen()
    _, _, _, _, funcs = gen.parse_header(src)
    params = {name: plist for name, _, plist in funcs}
    rets = {name: ret for name, ret, _ in funcs}
    rs = _rust()
    for base in BASES:
        bgr, rgb = params[base], params[base + "_rgb"]
        assert bgr[1][0] == "frames" and "fd_frame" in bgr[1][1] and "nv12" not in bgr[1][1], base
        assert rgb == bgr[:2] + [("layout", "i32")] + bgr[2:], base
        assert rets[base + "_rgb"] == rets[base] == "int"
        m = re.search(r"pub fn %s_rgb\((.*?)\) -> c_int;" % base, rs)
        b = re.search(r"pub fn %s\((.*?)\) -> c_int;" % base, rs)
        assert m and b and m.group(1) == b.group(1).replace("frames: *const fd_frame, ", "frames: *const fd_frame, layout: i32, "), base


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
        assert base + "_rgb" in ffi.SYMBOLS
        assert callable(getattr(Context, base[len("fd_"):] + "_rgb"))
