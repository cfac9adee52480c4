"""fd_pipeline_host_yuv420 / _yuv422 / _rgb of include/fd_b200.h, and their Rust and ctypes mirrors."""
import importlib.util
import os
import re

from conftest import ROOT

CALLS = {"fd_pipeline_host_yuv420": "fd_frame_nv12", "fd_pipeline_host_yuv422": "fd_frame", "fd_pipeline_host_rgb": "fd_frame"}


def _gen():
    spec = importlib.util.spec_from_file_location("gen_rust_ffi", os.path.join(ROOT, "scripts", "gen_rust_ffi.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    return gen, open(os.path.join(ROOT, "include", "fd_b200.h")).read()


def test_entry_points_take_the_bgr_parameters_with_the_frame_type_and_a_layout():
    gen, src = _gen()
    _, _, _, _, funcs = gen.parse_header(src)
    params = {name: plist for name, _, plist in funcs}
    rets = {name: ret for name, ret, _ in funcs}
    rs = open(os.path.join(ROOT, "rust", "src", "ffi.rs")).read()
    bgr = params["fd_pipeline_host"]
    assert bgr[1][0] == "frames" and "fd_frame" in bgr[1][1]
    b = re.search(r"pub fn fd_pipeline_host\((.*?)\) -> c_int;", rs)
    for name, frame in CALLS.items():
        got = params[name]
        assert got[0] == bgr[0] and got[1][0] == "frames" and frame in got[1][1] and (frame != "fd_frame" or "nv12" not in got[1][1]), name
        assert got[2] == ("layout", "i32") and got[3:] == bgr[2:], name
        assert rets[name] == rets["fd_pipeline_host"] == "int"
        m = re.search(r"pub fn %s\((.*?)\) -> c_int;" % name, rs)
        assert m and b and m.group(1) == b.group(1).replace("frames: *const fd_frame, ", "frames: *const %s, layout: i32, " % frame), name


def test_python_mirrors_every_entry_point():
    from rs_face_detection_b200 import Context, ffi
    for name in CALLS:
        assert name in ffi.SYMBOLS
        assert callable(getattr(Context, name[len("fd_"):]))
