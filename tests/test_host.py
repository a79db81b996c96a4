"""CPU: host-side logic - C ABI exports, constants, Zernike basis, module construction, no-fallback rule."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest
import torch

import b200cam
from b200cam import _lib, zernike
import b200cam.constants as K
from b200cam.optics import Camera
from oracle import camera_oracle as co
from oracle import ref_shim

REPO = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def library():
    _lib.build_library()
    return _lib.load_library()


def test_abi_exports_every_declared_symbol(library):
    header = (REPO / "include" / "b200cam.h").read_text()
    declared = set(re.findall(r"\b(b200cam_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTED_SYMBOLS)
    for name in declared:
        assert getattr(library, name) is not None


def test_column_kernel_batch_split(library):
    """col_chunks (b200cam.cu): one wave of CTAs where that fills the SMs, a finer split where the wave model predicts >= 10 %."""
    f = library.b200cam_col_chunks
    assert f(256, 64, 592) == 12 and f(256, 64, 444) == 9          # config 2: convolve (4 CTAs/SM), accumulate (3 CTAs/SM)
    assert f(256, 512, 592) == 12
    assert f(512, 32, 296) == 3 and f(512, 32, 148) == 3           # N = 512: 97 column groups; accumulate runs one CTA per SM
    assert f(1024, 8, 148) == 2                                    # 193 column groups cannot be one wave
    assert f(100, 8, 148) == 0 and f(256, 0, 148) == 0
    for N in (64, 128, 256, 512, 1024):
        for B in (1, 2, 3, 7, 16, 37, 64, 150):
            for slots in (148, 296, 444, 592):
                n = f(N, B, slots)
                assert 1 <= n <= min(B, 16)


def test_abi_size_queries_without_gpu(library):
    assert library.b200cam_version() == 100
    assert [library.b200cam_supported(n) for n in (64, 100, 256, 1024, 2048)] == [1, 0, 1, 1, 0]
    N = 256
    assert library.b200cam_otf_bytes(N) == 3 * (N // 2 + 1) * N * 8
    assert library.b200cam_otf_bytes(100) == 0
    per_plane = (N // 2 + 1) * N * 8
    assert library.b200cam_sensor_workspace_bytes(N, 64, 0) >= 2 * 64 * 3 * per_plane
    assert library.b200cam_psf_workspace_bytes(N) >= 3 * N * N * 8
    assert b"workspace" in library.b200cam_error_string(-3)


def test_abi_rejects_bad_arguments_before_touching_the_gpu(library):
    null = ctypes.c_void_p(0)
    kappa = (ctypes.c_float * 3)(1, 2, 3)
    assert library.b200cam_psf_fwd(null, null, null, null, kappa, null, null, null, null, 0, 100, null) == -1
    assert library.b200cam_psf_fwd(null, null, null, null, kappa, null, null, null, null, 0, 256, null) == -2
    assert library.b200cam_sensor_fwd(null, null, null, null, null, null, null, null, null, 0, 0, 256, null) == -1
    # the split PSF entry points and the Zernike projection validate the same way
    assert library.b200cam_psf_field(null, null, null, kappa, null, null, 0, 100, null, null, 0) == -1
    assert library.b200cam_psf_field(null, null, null, kappa, null, null, 0, 256, null, null, 0) == -2
    assert library.b200cam_psf_otf_early(null, null, 0, 256, null) == -2
    assert library.b200cam_psf_finish(null, null, null, null, 0, 256, null) == -2
    assert library.b200cam_zernike_workspace_bytes(300, 256 * 256) >= 256 * 256 * 4
    assert library.b200cam_zernike_workspace_bytes(300, 6) == 0                 # N*N must be a multiple of 4
    assert library.b200cam_zernike_fwd(null, null, null, null, 0, 300, 6, null) == -1
    assert library.b200cam_zernike_fwd(null, null, null, null, 0, 300, 65536, null) == -2
    assert library.b200cam_zernike_bwd(null, null, null, 0, 65536, null) == -1


def test_lens_abi_geometry_and_argument_checks_without_gpu(library):
    """The Image_Caption entry points (round 2): geometry predicates, workspace sizes and argument validation run on the host
    before anything is enqueued."""
    null = ctypes.c_void_p(0)
    d3 = (ctypes.c_double * 3)(1.0, 2.0, 3.0)
    # padded size 3R/2 must factor into radices <= 31; R a multiple of 4; P <= R
    assert [library.b200cam_lens_psf_supported(r, 64) for r in (896, 736, 128, 160, 130, 4 * 37 * 2)] == [1, 1, 1, 1, 0, 0]
    assert library.b200cam_lens_psf_padded(896) == 1344 and library.b200cam_lens_psf_padded(736) == 1104
    assert library.b200cam_lens_psf_workspace_bytes(896, 256) >= 3 * 896 * 1344 * 8
    assert library.b200cam_lens_psf_workspace_bytes(130, 64) == 0
    assert library.b200cam_lens_psf_fwd(null, null, null, d3, null, null, null, null, null, null, null, null, 0, null, null, null, 0,
                                        130, 64, null) == -1
    assert library.b200cam_lens_psf_fwd(null, null, null, d3, null, null, null, null, null, null, null, null, 0, null, null, null, 0,
                                        896, 256, null) == -2
    assert library.b200cam_lens_psf_bwd(null, null, null, null, null, null, null, d3, null, null, null, null, 0, null, null, 0,
                                        896, 256, null) == -2
    # sensor path: patch sizes 64 ... 512 (transform size 2P)
    assert library.b200cam_lens_sensor_workspace_bytes(256, 128) >= 128 * 3 * 257 * 512 * 8
    assert library.b200cam_lens_sensor_workspace_bytes(368, 8) == 0
    assert library.b200cam_lens_sensor_fwd(null, null, null, null, null, null, null, 0, 4, 368, null) == -1
    assert library.b200cam_lens_sensor_fwd(null, null, null, null, null, null, null, 0, 4, 256, null) == -2
    assert library.b200cam_lens_sensor_bwd(null, null, null, null, null, null, null, null, null, 0, 4, 256, null) == -2
    assert library.b200cam_lens_sensor_dot(null, null, null, null, null, 0, 4, 256, null) == -2
    assert library.b200cam_lens_normalise(null, null, null, 16, null) == -2
    # Zernike support-list variants
    assert library.b200cam_zernike_fwd_ex(null, null, null, null, 0, 300, 65536, null, null, 0) == -2
    assert library.b200cam_zernike_bwd_ex(null, null, null, 300, 6, null, null, 0) == -1


def test_no_cpu_fallback():
    cam = Camera(N=64, zernike_terms=6)
    with pytest.raises(RuntimeError, match="CUDA"):
        cam(torch.rand(1, 3, 64, 64))
    with pytest.raises(RuntimeError, match="CUDA"):
        cam.get_psf()


def test_product_does_not_import_oracle():
    for py in (REPO / "privacy-preserving-vision_b200").glob("*.py"):
        text = py.read_text()
        assert "import oracle" not in text and "from oracle" not in text, py


def test_constants_match_oracle():
    for N in (64, 256):
        T, C = K.build(N), co.build_constants(N)
        A = co.pupil_field(torch.zeros(1, N, N), C)
        assert (T.table_A - A).abs().max() <= 2e-6
        assert torch.equal(T.table_Ht, co.transfer_function(C).transpose(-1, -2))
        assert np.allclose(T.kappa, (C.k * C.flmb).flatten().numpy())
        assert torch.equal(T.rho, C.rho)


def test_noll_indices_and_orthonormality():
    assert [zernike.noll_to_nm(j) for j in range(1, 12)] == [
        (0, 0), (1, 1), (1, -1), (2, 0), (2, -2), (2, 2), (3, -1), (3, 1), (3, -3), (3, 3), (4, 0)]
    Z = zernike.zernike_basis(15, 256, outside=0.0)
    mask = Z[0] > 0
    gram = np.einsum("iyx,jyx->ij", Z, Z) / mask.sum()
    assert np.allclose(gram, np.eye(15), atol=3e-2)        # Noll-normalised: unit variance over the disk
    assert zernike.zernike_volume(64, 5).max() <= 4e-6


@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference sources not present (B200CAM_REFERENCE_ROOT)")
def test_module_constructs_like_the_reference():
    torch.manual_seed(3)
    ours = Camera(N=64, zernike_terms=10)
    torch.manual_seed(3)
    ref = ref_shim.load_face_deid_camera()(N=64, zernike_terms=10)
    so, sr = ours.state_dict(), ref.state_dict()
    assert list(so.keys()) == list(sr.keys())
    assert all(torch.equal(so[k], sr[k]) for k in sr)
    assert [n for n, p in ours.named_parameters() if p.requires_grad] == ["Zer_train"]
    for name in ("XY", "FF", "XY2", "rho", "rad", "k", "flmb", "lamb", "u", "x2", "fx1", "r", "r2"):
        assert torch.equal(getattr(ours, name), getattr(ref, name)), name
    assert torch.equal(ours.get_Heith_Map(), ref.get_Heith_Map())
    assert torch.equal(ours.get_phase_shift(), ref.get_phase_shift())
    ours.load_state_dict(ref.state_dict(), strict=True)


def test_module_constructs_like_the_stored_state():
    """The checks of test_module_constructs_like_the_reference against tests/golden/camera_init_n64_t10.npz, without the
    live reference.  The file's ``source`` names the Camera class that wrote it (oracle/make_golden.py writes it from the
    reference); written from this package, it guards the constructor against change rather than pinning it to the
    reference."""
    z = np.load(REPO / "tests" / "golden" / "camera_init_n64_t10.npz")
    torch.manual_seed(3)
    ours = Camera(N=64, zernike_terms=10)
    so = ours.state_dict()
    assert list(so) == z["state_keys"].tolist()
    assert all(torch.equal(so[k], torch.from_numpy(z[f"sd.{k}"])) for k in so)
    assert [n for n, p in ours.named_parameters() if p.requires_grad] == z["trainable"].tolist()
    attrs = [k for k in z.files if k.startswith("attr.")]
    assert len(attrs) == 13
    for key in attrs:
        assert torch.equal(getattr(ours, key[len("attr."):]), torch.from_numpy(z[key])), key
    with torch.no_grad():
        assert torch.equal(ours.get_Heith_Map(), torch.from_numpy(z["heith_map"]))
        assert torch.equal(ours.get_phase_shift(), torch.from_numpy(z["phase_shift"]))


def test_state_dict_roundtrip(tmp_path):
    a = Camera(N=64, zernike_terms=8)
    torch.save({"Camera": a.state_dict()}, tmp_path / "cam.pth")   # solver.py:90 layout
    b = Camera(N=64, zernike_terms=8)
    b.load_state_dict(torch.load(tmp_path / "cam.pth")["Camera"])  # solver.py:46-48
    assert torch.equal(a.Zer_train, b.Zer_train) and torch.equal(a.ca, b.ca)


def test_caption_camera_loads_both_reference_checkpoint_layouts():
    """SURVEY 8 f3: the shipped 3+1+(T-4) layout (Lens.py:92-96) and Model.pth's 3+(T-3) layout with `optics.` keys
    (train.py:71-78, Lens.py:99-101) load into the same module."""
    from b200cam.lens import OpticsZernike
    T = 12
    cam = OpticsZernike(input_shape=[None, 16, 16, 3], device="cpu", zernike_terms=T, patch_size=16,
                        wave_resolution=[32, 32], sample_interval=3e-6, height_tolerance=None)
    g = torch.Generator().manual_seed(1)
    full = torch.randn(T, 1, 1, generator=g)
    legacy = {"model": {"optics.zernike_coeffs_no_train": full[:3].clone(), "optics.zernike_coeffs_train": full[3:].clone()}}
    cam.load_reference_state_dict(legacy)
    got = torch.cat((cam.zernike_coeffs_no_train, cam.zernike_coeffs_train.unsqueeze(0), cam.zernike_coeffs_no_train2), 0)
    assert torch.equal(got.detach(), full)
    assert cam.zernike_coeffs_train.shape == (1, 1) and cam.zernike_coeffs_train.requires_grad
    shipped = {k: v.detach().clone() + 1.0 for k, v in cam.state_dict().items()}
    cam.load_reference_state_dict(shipped)
    assert torch.equal(cam.zernike_coeffs_no_train2.detach(), full[4:] + 1.0)


@pytest.mark.skipif(not (ref_shim.reference_available()
                         and (ref_shim.REFERENCE_ROOT / "Image_Caption" / "Camera" / "Model.pth").is_file()),
                    reason="reference sources not present (B200CAM_REFERENCE_ROOT)")
def test_caption_camera_loads_the_real_reference_checkpoint():
    """SURVEY 8 f3 with the checkpoint the reference ships: Image_Caption/Camera/Model.pth holds {'model': {optics.
    zernike_coeffs_no_train (3,1,1), optics.zernike_coeffs_train (347,1,1)}} - the 3 + (T-3) layout of train.py:71-78 at
    T = 350, which the shipped module's own load_state_dict rejects.  Loaded here into a T = 350 camera (small wave grid:
    the coefficient vector, not the basis, is what the checkpoint defines)."""
    from b200cam.lens import OpticsZernike
    ck = torch.load(ref_shim.REFERENCE_ROOT / "Image_Caption" / "Camera" / "Model.pth", map_location="cpu", weights_only=False)
    ref = ck["model"]
    cam = OpticsZernike(input_shape=[None, 16, 16, 3], device="cpu", zernike_terms=350, patch_size=16,
                        wave_resolution=[32, 32], sample_interval=3e-6, height_tolerance=None)
    cam.load_reference_state_dict(ck)
    got = torch.cat((cam.zernike_coeffs_no_train, cam.zernike_coeffs_train.unsqueeze(0), cam.zernike_coeffs_no_train2), 0)
    want = torch.cat((ref["optics.zernike_coeffs_no_train"], ref["optics.zernike_coeffs_train"]), 0)
    assert got.shape == (350, 1, 1) and torch.equal(got.detach(), want)
    assert float(cam.zernike_coeffs_train) == float(ref["optics.zernike_coeffs_train"][0])


def test_bench_dump_outputs_stays_in_budget_and_samples_reproducibly(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 .npy files, at most DUMP_BYTES in all; an output too large for that is cut to the
    same seeded sample of its batch dimension on every run."""
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 100_000)
    g = torch.Generator().manual_seed(0)
    outs = {"sensor": torch.rand(40, 3, 16, 16, generator=g), "grad_h": torch.rand(1, 16, 16, generator=g),
            "loss_rad": torch.tensor(0.5)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outs)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["grad_h.npy", "loss_rad.npy", "sensor.npy", "sensor_index.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 100_000
    idx = np.load(tmp_path / "a" / "sensor_index.npy")
    sensor = np.load(tmp_path / "a" / "sensor.npy")
    assert sensor.dtype == np.float32 and 1 <= len(idx) < 40 and np.all(np.diff(idx) > 0)
    assert np.array_equal(sensor, outs["sensor"].numpy()[idx.astype(int)])
    assert np.array_equal(idx, np.load(tmp_path / "b" / "sensor_index.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "grad_h.npy"), outs["grad_h"].numpy())
