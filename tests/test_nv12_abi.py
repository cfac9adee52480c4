"""The NV12 frame descriptor of include/fd_b200.h: its ctypes and Rust mirrors, its layout, and the *_nv12 entry points."""
import ctypes as C
import importlib.util
import os
import re

from conftest import ROOT


def _gen():
    spec = importlib.util.spec_from_file_location("gen_rust_ffi", os.path.join(ROOT, "scripts", "gen_rust_ffi.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    return gen, open(os.path.join(ROOT, "include", "fd_b200.h")).read()


def test_ctypes_mirror_matches_the_header():
    from rs_face_detection_b200 import ffi
    gen, src = _gen()
    plain = dict(gen.parse_plain_structs(src))
    assert set(plain) == {"fd_frame_nv12"}
    assert [n for n, _ in ffi.FdFrameNV12._fields_] == [n for n, _ in plain["fd_frame_nv12"]]
    assert C.sizeof(ffi.FdFrameNV12) == 32
    assert ffi.FdFrameNV12.height.offset == 16 and ffi.FdFrameNV12.pitch_uv.offset == 28


def test_generated_rust_declares_the_struct_not_an_opaque_type():
    gen, src = _gen()
    _, _, _, opaque, funcs = gen.parse_header(src)
    assert "fd_frame_nv12" not in opaque
    rs = open(os.path.join(ROOT, "rust", "src", "ffi.rs")).read()
    m = re.search(r"pub struct fd_frame_nv12 \{(.*?)\}", rs, flags=re.S)
    assert m and "pub y: *const u8" in m.group(1) and "pub pitch_uv: i32" in m.group(1)
    names = {name for name, _, _ in funcs}
    for base in ("fd_preprocess_batch", "fd_align_batch", "fd_align_detections", "fd_select_detections", "fd_align_selected"):
        assert base + "_nv12" in names
        bgr = next(p for n, _, p in funcs if n == base)
        nv = next(p for n, _, p in funcs if n == base + "_nv12")
        assert [t for _, t in nv] == [t.replace("fd_frame", "fd_frame_nv12") for _, t in bgr], base
