"""The C-ABI library loads without a GPU, exports every symbol include/fd_b200.h declares, and the product path fails
loudly (no CPU fallback) when no device is present."""
import os
import re
import subprocess

import pytest

from conftest import HAS_GPU, ROOT


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "fd_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = set(re.findall(r"\b(fd_[a-z0-9_]+|_nms|_set_device)\s*\(", src))
    return names


def test_library_builds_and_exports_header():
    from rs_face_detection_b200 import build as B, ffi
    lib_path = B.build()
    out = subprocess.check_output(["nm", "-D", "--defined-only", lib_path], text=True)
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    header = _header_symbols()
    assert header, "no symbols parsed from the header"
    assert header <= exported, "declared but not exported: %s" % sorted(header - exported)
    assert set(ffi.SYMBOLS) == header, "ffi.SYMBOLS out of sync with the header: %s" % sorted(set(ffi.SYMBOLS) ^ header)
    lib = ffi.load()
    assert lib.fd_abi_version() == 2


def test_struct_layout_matches_c():
    from rs_face_detection_b200 import ffi
    import ctypes as C
    assert C.sizeof(ffi.FdConfig) == 4 * (2 + 2 + 1 + 8 + 1 + 8 * 4 * 4 + 3 + 3 + 1 + 4 + 1 + 2 + 10)
    assert C.sizeof(ffi.FdFrame) == 24
    cfg = ffi.default_config()
    assert (cfg.image_w, cfg.image_h, cfg.n_strides, cfg.num_anchors) == (640, 640, 3, 2)
    assert abs(cfg.conf_thr - 0.7) < 1e-7 and abs(cfg.iou_thr - 0.45) < 1e-7
    assert list(cfg.strides)[:3] == [32, 16, 8]
    assert (cfg.crop_w, cfg.crop_h) == (112, 112)


@pytest.mark.skipif(HAS_GPU, reason="only meaningful without a GPU")
def test_no_cpu_fallback_without_gpu():
    from rs_face_detection_b200 import Context, FdError, ffi
    with pytest.raises(FdError) as e:
        Context(0)
    assert e.value.code == ffi.FD_ERR_NO_DEVICE
    assert "no CPU fallback" in str(e.value)


def test_product_never_touches_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's baseline legs may use oracle/."""
    pkg = os.path.join(ROOT, "rs_face_detection_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                txt = open(os.path.join(dirpath, f), errors="replace").read()
                assert "fd_oracle" not in txt and "import oracle" not in txt and "from oracle" not in txt and "libfd_oracle" not in txt, f


# ---- the three declarations of the boundary (header / ctypes / Rust) and the two build recipes cannot drift -------------
def _split_args(argstr):
    out, depth, cur = [], 0, ""
    for ch in argstr:
        if ch in "([{":
            depth += 1
        elif ch in ")]}":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur)
            cur = ""
        else:
            cur += ch
    if cur.strip():
        out.append(cur)
    return out


def _call_sites(text, prefix_re):
    """[(name, n_args)] for every `<prefix>name(...)` call in text (balanced parentheses, top-level commas)."""
    sites = []
    for m in re.finditer(prefix_re + r"(fd_[a-z0-9_]+|_nms|_set_device)\s*\(", text):
        i, depth = m.end(), 1
        while depth and i < len(text):
            depth += text[i] in "([{"
            depth -= text[i] in ")]}"
            i += 1
        sites.append((m.group(1), len(_split_args(text[m.end():i - 1]))))
    return sites


def _header_arity():
    import importlib.util
    spec = importlib.util.spec_from_file_location("gen_rust_ffi", os.path.join(ROOT, "scripts", "gen_rust_ffi.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    _, _, structs, _, funcs = gen.parse_header(open(os.path.join(ROOT, "include", "fd_b200.h")).read())
    return gen, {name: len(params) for name, _, params in funcs}, dict(structs)


def test_rust_ffi_is_generated_from_the_header():
    gen, arity, _ = _header_arity()
    assert set(arity) == _header_symbols()
    committed = open(os.path.join(ROOT, "rust", "src", "ffi.rs")).read()
    assert committed == gen.generate(), "rust/src/ffi.rs is stale: run python scripts/gen_rust_ffi.py"
    for name in arity:                                   # every header symbol is declared on the Rust side
        assert re.search(r"pub fn %s\(" % re.escape(name), committed), name


def test_rust_and_python_call_sites_match_the_header_arity():
    _, arity, structs = _header_arity()
    rust_dir = os.path.join(ROOT, "rust", "src")
    n_sites = 0
    for dirpath, _, files in os.walk(rust_dir):
        for f in files:
            if not f.endswith(".rs") or f == "ffi.rs":
                continue
            txt = re.sub(r"//[^\n]*", "", open(os.path.join(dirpath, f)).read())
            for name, n in _call_sites(txt, r"ffi::"):
                assert name in arity, "%s calls unknown symbol %s" % (f, name)
                assert n == arity[name], "%s: %s called with %d args, header declares %d" % (f, name, n, arity[name])
                n_sites += 1
    assert n_sites >= 20
    py = open(os.path.join(ROOT, "rs_face_detection_b200", "ffi.py")).read()
    py = re.sub(r"#[^\n]*", "", py)
    n_py = 0
    for name, n in _call_sites(py, r"(?:self\.lib|load\(\)|lib|_lib)\."):
        if name in ("fd_last_error", "fd_ctx_stream") and n == 0:
            continue                                     # attribute access for restype, not a call
        assert n == arity[name], "ffi.py: %s called with %d args, header declares %d" % (name, n, arity[name])
        n_py += 1
    assert n_py >= 40
    # ctypes struct mirrors: same field names in the same order as the header
    from rs_face_detection_b200 import ffi
    mirrors = {"fd_config": ffi.FdConfig, "fd_frame": ffi.FdFrame, "fd_anchor_cfg": ffi.FdAnchorCfg, "fd_det_view": ffi.FdDetView,
               "fd_host_batch_out": ffi.FdHostBatchOut, "fd_select_params": ffi.FdSelectParams, "fd_pipeline_opts": ffi.FdPipelineOpts}
    assert set(mirrors) == set(structs)
    for cname, cls in mirrors.items():
        assert [n for n, _ in cls._fields_] == [n for n, _ in structs[cname]], cname


def test_build_recipes_compile_every_translation_unit():
    from rs_face_detection_b200 import build as B
    cu = sorted(f for f in os.listdir(B.CSRC) if f.endswith(".cu"))
    assert sorted(B.SOURCES) == cu, "build.py SOURCES != csrc/*.cu"
    rs = open(os.path.join(ROOT, "rust", "build.rs")).read()
    assert "read_dir(&csrc)" in rs and '"cu"' in rs, "rust/build.rs must compile every csrc/*.cu"
    assert "defs" in rs, "rust/build.rs must link with -z defs so a missing translation unit fails the build"
    for flag in ("arch=compute_100a,code=sm_100a", "-fmad=false", "-lineinfo"):
        assert flag in rs and flag in " ".join(B.FLAGS), flag
    # the library itself has no undefined symbol outside libc / libstdc++ / libcudart
    out = subprocess.check_output(["nm", "-D", "--undefined-only", B.build()], text=True)
    for line in out.splitlines():
        sym = line.split()[-1]
        assert not sym.startswith(("fd_", "_ZN2fd")), "undefined in libfd_b200.so: " + sym


REFERENCE_SIGNATURES = {   # file under rust/src -> signatures copied verbatim from the reference (file:line), whitespace-normalised
    "processing/nms.rs": ["pub fn nms(dets: &Array2<f32>, thresh: f32) -> Vec<usize>"],                                   # nms.rs:3
    "processing/bbox_transform.rs": [
        "pub fn bbox_overlaps_py(boxes: &Array2<f32>, query_boxes: &Array2<f32>) -> Array2<f32>",                          # :2
        "pub fn clip_boxes(boxes: &mut Array2<f32>, im_shape: (usize, usize))",                                            # :27
        "pub fn clip_points(points: &mut Array2<f32>, im_shape: (usize, usize))",                                          # :47
        "pub fn nonlinear_transform(ex_rois: &Array2<f32>, gt_rois: &Array2<f32>) -> Array2<f32>",                         # :67
        "pub fn nonlinear_pred(boxes: &Array2<f32>, box_deltas: &Array2<f32>) -> Array2<f32>",                             # :90
        "pub fn landmark_pred(boxes: &Array2<f32>, point_deltas: &Array2<f32>) -> Array2<f32>",                            # :123
        "pub fn iou_pred(boxes: &Array2<f32>, box_deltas: &Array2<f32>, num_classes: usize) -> Array2<f32>"],              # :162
    "processing/generate_anchors.rs": [
        "pub fn generate_anchors(base_size: usize, ratios: Array1<f32>, scales: Array1<f32>) -> Array2<f32>",              # :41
        "pub fn generate_anchors2(base_size: usize, ratios: Array1<f32>, scales: Array1<f32>, stride: usize, dense_anchor: bool) -> Array2<f32>",
        "pub fn generate_anchors_fpn(base_size: Vec<i32>, ratios: Vec<f32>, scales: Vec<f32>) -> Vec<Array2<f32>>",        # :95
        "pub fn generate_anchors_fpn2(dense_anchor: bool, cfg: Option<&Config>) -> Vec<Array2<f32>>"],                     # :116
    "rcnn/anchors.rs": ["pub fn anchors(height: usize, width: usize, stride: usize, base_anchors: &Array2<f32>) -> Array4<f32>"],   # :3
    "rcnn/bbox.rs": ["pub(crate) fn bbox_overlaps(boxes: &Array2<f32>, query_boxes: &Array2<f32>) -> Array2<f32>"],        # :4
    "rcnn/cpu_nms.rs": ["fn cpu_nms(dets: ArrayView2<f32>, thresh: f32) -> Vec<usize>"],                                   # :10
    "rcnn/gpu_nms.rs": ["pub fn gpu_nms(dets: Array2<f32>, thresh: f32, device_id: i32) -> Vec<usize>"],                   # gpu_nms.rs:21
    "pipeline/module/face_alignment.rs": [
        "pub fn new(image_size: (i32, i32), standard_landmarks: Array2<f32>) -> Self",                                     # :20
        "pub fn call(&self, img: &Mat, bbox: Option<Array1<f32>>, landmarks: Option<Array2<f32>>, _is_debug: Option<bool>) -> Result<Mat, Error>"],
    "pipeline/module/face_selection.rs": [
        "pub fn call(&self, img: &Mat, face_boxes: Array2<f32>, key_points: Option<Array3<f32>>, is_enroll: Option<bool>, _is_debug: Option<bool>) "
        "-> Result<(Option<Array1<f32>>, Option<Array2<f32>>), Error>"],                                                   # :72
    "pipeline/module/face_detection.rs": ["-> Result<(Array2<f32>, Option<Array3<f32>>), Error>"],                         # :496
    "utils/utils.rs": ["pub fn byte_data_to_opencv(im_bytes: &[u8]) -> Result<Mat, Error>"],                              # utils.rs:8
}


def test_rust_wrappers_keep_the_reference_signatures():
    norm = lambda t: " ".join(t.split())
    for rel, sigs in REFERENCE_SIGNATURES.items():
        txt = norm(open(os.path.join(ROOT, "rust", "src", rel)).read())
        for sig in sigs:
            assert norm(sig) in txt, "%s: missing `%s`" % (rel, sig)
