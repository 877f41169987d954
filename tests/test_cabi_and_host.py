"""CPU: the C-ABI library builds for sm_100a, loads, exports every symbol include/ffr.h declares, reports errors
without a GPU (no compute), and the host-side helpers mirror the reference's (tests/base/test_similar_faces_filter.py)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest


def test_library_exports_every_header_symbol(ffr_lib):
    from face_detection_and_recognition_b200 import _lib
    names = _lib.header_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(ffr_lib, n), f"{n} declared in include/ffr.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature"
    assert ffr_lib.ffr_abi_version() == 1
    assert b"sm_100a" in ffr_lib.ffr_build_info()


def test_library_contains_blackwell_sass(ffr_lib):
    """The .so carries sm_100a SASS with tcgen05 (UTC*MMA), TMEM loads (LDTM) and TMA (UTMALDG)."""
    from face_detection_and_recognition_b200._build import LIB_PATH
    cuobjdump = "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG"):
        assert mnemonic in sass, f"{mnemonic} missing from SASS"


def test_padded_dim_and_workspace_queries(ffr_lib):
    assert [ffr_lib.ffr_padded_dim(d) for d in (1, 64, 65, 128, 200, 512)] == [64, 64, 128, 128, 256, 512]
    assert ffr_lib.ffr_filter_workspace_bytes(0, 10, 128, 0, 0) == 0
    small = ffr_lib.ffr_filter_workspace_bytes(1, 1000, 128, 0, 1)          # euclid -> fp32 path, header only
    big = ffr_lib.ffr_filter_workspace_bytes(1000, 100000, 256, 0, 0)       # cosine -> fp16 copies + recheck list
    assert small == 256
    assert big >= 1000 * 256 * 2 + 100000 * 256 * 2 + 100000 * 16
    # 128-d rows at this size take the stage32 schedule: the fp16 A tiles only exist in shared memory, no fp16 copy of the
    # candidates in the workspace (references + re-check lists only)
    st32 = ffr_lib.ffr_filter_workspace_bytes(1000, 100000, 128, 0, 0)
    assert 1000 * 128 * 2 + 100000 * 28 <= st32 < 1000 * 128 * 2 + 100000 * 28 + 100000 * 128 * 2
    assert ffr_lib.ffr_allgather_workspace_bytes(8, 1000) >= 9 * 1008 * 5


def test_errors_without_gpu_are_reported_not_swallowed(ffr_lib):
    """No CPU fallback: invalid arguments give FFR_ERR_INVALID, and on a GPU-less host compute calls give FFR_ERR_CUDA."""
    from face_detection_and_recognition_b200 import _lib
    rc = ffr_lib.ffr_filter(None, 0, None, 0, 128, 0, None, None, 0, 0.5, 0, None, None, None, None, 0, None)
    assert rc == -1 and b"n_ref" in ffr_lib.ffr_last_error()
    rc = ffr_lib.ffr_l2norm_rows_f32(None, 4, 128, None, 128, None, None, None)
    assert rc == -1
    if ffr_lib.ffr_device_count() == 0:
        buf = (C.c_float * 128)()
        rc = ffr_lib.ffr_l2norm_rows_f32(C.addressof(buf), 1, 128, None, 128, None, None, None)
        assert rc == -2 and b"no CUDA device" in ffr_lib.ffr_last_error()
        h = C.c_void_p()
        assert ffr_lib.ffr_ctx_create(0, 10, 10, 128, C.byref(h)) == -2
        with pytest.raises(_lib.FfrError):
            _lib.check(rc)


def test_ops_refuse_cpu_tensors(ffr_lib):
    import torch
    from face_detection_and_recognition_b200 import ops
    with pytest.raises(TypeError):
        ops.face_filter(torch.zeros(2, 128), torch.zeros(4, 128), 0.5)
    with pytest.raises(TypeError):
        ops.l2norm_rows(torch.zeros(2, 128))


def test_product_never_imports_oracle():
    """The shipped package must not reference oracle/ (test infrastructure only)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, "face_detection_and_recognition_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, os.path.join(dirpath, f)


# ---- host helpers: same tests as the reference's tests/base/test_similar_faces_filter.py:8-27 -------------
def test_fix_path_for_globbing():
    from face_detection_and_recognition_b200.filter_faces_using_reference import _fix_path_for_globbing
    assert _fix_path_for_globbing("data/") == "data/*"
    assert _fix_path_for_globbing("data") == "data/*"
    assert _fix_path_for_globbing("data/*") == "data/*"


def test_get_class_name_list(tmp_path):
    from face_detection_and_recognition_b200.filter_faces_using_reference import get_class_name_list
    root = tmp_path / "data"
    root.mkdir()
    for i in range(10):
        (root / f"class_{i}").mkdir()
    assert get_class_name_list(str(root)) == [f"class_{i}" for i in range(10)]


def test_read_and_preprocess_img(tmp_path):
    from PIL import Image
    from face_detection_and_recognition_b200.filter_faces_using_reference import read_and_preprocess_img
    np.random.seed(42)
    img_np = (np.random.randn(160, 160, 3) * 255).astype(np.uint8)
    p = str(tmp_path / "numpy_random_img.jpg")
    Image.fromarray(img_np).save(p)
    img_np = np.array(Image.open(p))
    out = read_and_preprocess_img(p, in_size=(160, 160), dct_method="INTEGER_ACCURATE").numpy()
    n = img_np.size
    want = (img_np - np.mean(img_np)) / max(np.std(img_np), 1 / (n ** 0.5))
    assert out.shape == (160, 160, 3)
    assert np.allclose(out, want, atol=1e-4)
    assert read_and_preprocess_img(p, in_size=(112, 96)).shape == (112, 96, 3)


def test_cli_flags_match_reference():
    from face_detection_and_recognition_b200.filter_faces_using_reference import get_parsed_args
    a = get_parsed_args(["--ud", "u", "--rd", "r"])
    assert (a.unfiltered_data_path, a.reference_data_path, a.target_data_path) == ("u", "r", "data/faces_filtered")
    assert (a.savedmodel_path, a.batch_size, a.ref_img_per_class) == ("models/facenet/facenet_keras_p38", 32, 32)
    a = get_parsed_args(["--unfiltered_data_path", "u", "--reference_data_path", "r", "--target_data_path", "t",
                         "-m", "w", "-b", "8", "-r", "4"])
    assert (a.target_data_path, a.savedmodel_path, a.batch_size, a.ref_img_per_class) == ("t", "w", 8, 4)
    with pytest.raises(SystemExit):
        get_parsed_args(["--ud", "u"])


def test_class_mismatch_raises(tmp_path):
    from face_detection_and_recognition_b200.filter_faces_using_reference import main
    (tmp_path / "u" / "a").mkdir(parents=True)
    (tmp_path / "r" / "a").mkdir(parents=True)
    (tmp_path / "r" / "b").mkdir(parents=True)
    with pytest.raises(Exception, match="Class number Error"):
        main(["--ud", str(tmp_path / "u"), "--rd", str(tmp_path / "r"), "--td", str(tmp_path / "t")], model=object())
    (tmp_path / "u" / "c").mkdir()
    with pytest.raises(Exception, match="did not match"):
        main(["--ud", str(tmp_path / "u"), "--rd", str(tmp_path / "r"), "--td", str(tmp_path / "t")], model=object())


# Stands in for the reference's face_detection_and_extraction/modules/mobile_facenet/mobile_facenet.py, which is not part
# of this repository: same module name, same MobileFaceNet(embedding_size) constructor, [b, 3, 112, 112] in, and the
# output goes through the reference's l2_norm (:30-33, :154).
MOBILE_FACENET_PY = '''
import torch


def l2_norm(input, axis=1):
    norm = torch.norm(input, 2, axis, True)
    return torch.div(input, norm)


class MobileFaceNet(torch.nn.Module):
    def __init__(self, embedding_size):
        super().__init__()
        self.conv = torch.nn.Conv2d(3, 16, 3, stride=2, padding=1, bias=False)
        self.bn = torch.nn.BatchNorm2d(16)
        self.pool = torch.nn.AdaptiveAvgPool2d(7)
        self.linear = torch.nn.Linear(16 * 7 * 7, embedding_size)

    def forward(self, x):
        x = self.pool(torch.relu(self.bn(self.conv(x))))
        return l2_norm(self.linear(x.flatten(1)))
'''


def test_mobilefacenet_adapter_wraps_the_reference_model(tmp_path):
    """north_star: embedding extraction stays in the reference's own PyTorch MobileFaceNet.  The adapter imports that
    class from the given directory (never a copy), honours the predict() contract of filter_faces_using_reference.py:84,184
    and returns exactly what the wrapped network computes."""
    import sys
    import torch
    from face_detection_and_recognition_b200.filter_faces_using_reference import MobileFaceNetModel
    REFERENCE_MFN = str(tmp_path / "mobile_facenet")
    os.makedirs(REFERENCE_MFN)
    with open(os.path.join(REFERENCE_MFN, "mobile_facenet.py"), "w") as f:
        f.write(MOBILE_FACENET_PY)
    sys.modules.pop("mobile_facenet", None)
    with pytest.raises(FileNotFoundError):
        MobileFaceNetModel(str(tmp_path / "missing.pth"), str(tmp_path), device="cpu", allow_random_init=True)
    with pytest.raises(FileNotFoundError):
        MobileFaceNetModel(str(tmp_path / "missing.pth"), REFERENCE_MFN, device="cpu")
    torch.manual_seed(0)
    model = MobileFaceNetModel(str(tmp_path / "missing.pth"), REFERENCE_MFN, device="cpu", allow_random_init=True)
    assert type(model.net).__module__ == "mobile_facenet" and type(model.net).__name__ == "MobileFaceNet"
    assert "face_detection_and_recognition_b200" not in sys.modules["mobile_facenet"].__file__
    batch = np.random.default_rng(0).standard_normal((3, 160, 160, 3)).astype(np.float32)
    out = model.predict(batch, verbose=0)
    assert out.shape == (3, 512) and out.dtype == np.float32
    np.testing.assert_allclose(np.linalg.norm(out, axis=1), 1.0, atol=1e-5)       # the net ends in l2_norm (:30-33,154)
    x = torch.nn.functional.interpolate(torch.from_numpy(batch).permute(0, 3, 1, 2), size=(112, 112), mode="bilinear",
                                        align_corners=False)
    with torch.no_grad():
        want = model.net(x).numpy()
    np.testing.assert_allclose(out, want, atol=1e-6)
    # a state dict saved from the reference class loads through -m
    torch.save(model.net.state_dict(), str(tmp_path / "w.pth"))
    m2 = MobileFaceNetModel(str(tmp_path / "w.pth"), REFERENCE_MFN, device="cpu")
    np.testing.assert_allclose(m2.predict(batch), out, atol=1e-6)
