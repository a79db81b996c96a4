"""GPU (-m gpu): uint8 images on the Face-DeId camera are read by the sensor kernels as they are.

The contract: ``cam(u8)`` equals ``cam(u8.to(torch.float32).div_(255.0))`` bit for bit - sensor image (fp32 and bf16), PSF, both
regularisers and dL/dZer_train - while no fp32 copy of the batch is made or kept for the backward."""
import ctypes
import os
import subprocess
import sys

import pytest
import torch

import b200cam.synthetic as synth
from b200cam import _lib
from b200cam import functional as F
from conftest import REPO, rel_l2
from u8_switch_runner import BF16, DEV, bits_equal, camera, face_step, u8_equals_converted, u8_images

pytestmark = pytest.mark.gpu

CASES = [(64, 3, overlap, dtype, epi) for overlap in (True, False) for dtype in (torch.float32, BF16) for epi in (False, True)] + [
    (128, 4, True, torch.float32, False), (128, 4, False, BF16, True),
    (256, 64, True, torch.float32, False), (256, 64, False, torch.float32, True), (256, 16, True, BF16, True),
    (512, 3, True, torch.float32, True), (512, 3, False, BF16, False),
    (1024, 2, True, torch.float32, False), (1024, 2, False, BF16, True)]


@pytest.mark.parametrize("N,B,overlap,dtype,epi", CASES)
def test_camera_u8_is_the_camera_on_the_converted_batch(N, B, overlap, dtype, epi):
    names = ("sensor", "psf", "loss_rad", "centering_loss", "Zer_train.grad")
    same = u8_equals_converted(N, B, overlap, dtype, epi)
    assert all(same), [n for n, ok in zip(names, same) if not ok]


def test_u8_step_repeats_itself():
    N, B = 64, 3
    cam = camera(N)
    u = u8_images(B, N, seed=1)
    g = (synth.upstream_grad(B, N, seed=2) * 1e-2).to(DEV)
    a = face_step(cam, u, g)
    b = face_step(cam, u, g)
    for x, y in zip(a, b):
        assert bits_equal(x, y)


# ------------------------------------------------------------------------------------------------------------ C ABI
def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _same_ties(a, b):
    """tie_pos is written only up to tie_count (its other slots are never read).  With more than 8 ties (the saturated image 0)
    which 8 are recorded depends on the order of the recording atomics: only the count is compared there (the arg-max term of
    a constant plane is the same for any 8 of its positions)."""
    assert torch.equal(a["tc"], b["tc"])
    for i, n in enumerate(a["tc"].tolist()):
        if n <= 8:
            assert sorted(a["tp"][i, :n].tolist()) == sorted(b["tp"][i, :n].tolist())


@pytest.mark.parametrize("N,B", [(64, 3), (256, 5), (1024, 2)])
def test_abi_u8_entry_points_equal_the_fp32_calls(N, B):
    """every uint8 entry point against its fp32 counterpart on the converted batch; b200cam_sensor_bwd_u8 with spectrum = NULL
    (the uint8 K1 row pass rebuilds the spectra) against the same call with the saved spectrum and against the fp32 call"""
    plan = F.DevicePlan(N, DEV)
    lib = plan.lib
    P = _lib.ptr
    u = u8_images(B, N, seed=N)
    x = u.to(torch.float32).div_(255.0)
    psf = torch.rand(3, N, N, generator=torch.Generator().manual_seed(1)).to(DEV)
    psf /= psf.sum()
    ws = torch.empty(lib.b200cam_sensor_workspace_bytes(N, B, 1), dtype=torch.uint8, device=DEV)
    sfloats = lib.b200cam_spectrum_bytes(N, B) // 4

    def bufs():
        return dict(img_max=torch.empty(B, device=DEV), tc=torch.empty(B, dtype=torch.int32, device=DEV),
                    tp=torch.empty(B, 8, dtype=torch.int32, device=DEV), otf=torch.empty(plan.otf_floats, device=DEV),
                    spec=torch.empty(sfloats, device=DEV), y=torch.empty(B, 3, N, N, device=DEV))

    def fwd(fn, img, d):
        _lib.check(fn(P(img), P(psf), P(d["y"]), P(d["img_max"]), P(d["tc"]), P(d["tp"]), P(d["otf"]), P(d["spec"]),
                      P(ws), ws.numel(), B, N, _stream(), 0, None, 0.0, 0))

    a, b = bufs(), bufs()
    fwd(lib.b200cam_sensor_fwd_ex, x, a)
    fwd(lib.b200cam_sensor_fwd_u8, u, b)
    for k in ("y", "img_max", "tc", "otf", "spec"):
        assert bits_equal(a[k], b[k]), k
    _same_ties(a, b)
    # split forward: uint8 rows, then the unchanged finish
    c = bufs()
    _lib.check(lib.b200cam_sensor_rows_u8(P(u), P(c["spec"]), P(c["img_max"]), P(c["tc"]), B, N, _stream()))
    assert bits_equal(c["spec"], a["spec"])
    _lib.check(lib.b200cam_sensor_finish_ex(P(psf), P(c["y"]), P(c["img_max"]), P(c["tc"]), P(c["tp"]), P(c["otf"]), P(c["spec"]),
                                            0, P(ws), ws.numel(), B, N, _stream(), 0, None, 0.0, 0))
    assert bits_equal(c["y"], a["y"])
    _same_ties(a, c)
    # bf16 sensor image
    conv = torch.empty(B, 3, N, N, device=DEV)
    y16 = [torch.empty(B, 3, N, N, device=DEV, dtype=BF16) for _ in range(2)]
    for img, fn, out in ((x, lib.b200cam_sensor_fwd_bf16, y16[0]), (u, lib.b200cam_sensor_fwd_u8_bf16, y16[1])):
        d = bufs()
        _lib.check(fn(P(img), P(psf), P(conv), P(out), P(d["img_max"]), P(d["tc"]), P(d["tp"]), P(d["otf"]), P(d["spec"]),
                      P(ws), ws.numel(), B, N, _stream(), 0, None, 0.0, 0))
    assert bits_equal(y16[0], y16[1]) and bits_equal(y16[1], a["y"].to(BF16))
    # backward: fp32 call, uint8 call with the saved spectrum, uint8 call without (uint8 K1), bf16 gradient variants
    g32 = (synth.upstream_grad(B, N, seed=2) * 1e-2).to(DEV)
    g16 = g32.to(BF16)
    res = {}
    for name, fn, g, img, spec in (("fp32", lib.b200cam_sensor_bwd, g32, x, a["spec"]),
                                   ("u8", lib.b200cam_sensor_bwd_u8, g32, u, a["spec"]),
                                   ("u8_nospec", lib.b200cam_sensor_bwd_u8, g32, u, None),
                                   ("fp32_nospec", lib.b200cam_sensor_bwd, g32, x, None)):
        gp = torch.empty(3, N, N, device=DEV)
        _lib.check(fn(P(g), P(img), P(a["y"]), P(a["img_max"]), P(a["tc"]), P(a["tp"]), P(psf), P(a["otf"]), P(spec), P(gp), None,
                      P(ws), ws.numel(), B, N, _stream()))
        res[name] = gp
    for name, fn, img in (("bf16", lib.b200cam_sensor_bwd_bf16, x), ("u8_bf16", lib.b200cam_sensor_bwd_u8_bf16, u)):
        gp = torch.empty(3, N, N, device=DEV)
        _lib.check(fn(P(g16), P(img), P(a["img_max"]), P(a["tc"]), P(a["tp"]), P(psf), P(a["otf"]), None, P(gp), None,
                      P(ws), ws.numel(), B, N, _stream()))
        res[name] = gp
    assert bits_equal(res["u8"], res["fp32"])
    assert bits_equal(res["u8_nospec"], res["u8"])
    assert bits_equal(res["u8_nospec"], res["fp32_nospec"])
    assert bits_equal(res["u8_bf16"], res["bf16"])
    # dL/dimg (w.r.t. the converted image) is available from the uint8 call as well
    gi = [torch.empty(B, 3, N, N, device=DEV) for _ in range(2)]
    for img, fn, out in ((x, lib.b200cam_sensor_bwd, gi[0]), (u, lib.b200cam_sensor_bwd_u8, gi[1])):
        gp = torch.empty(3, N, N, device=DEV)
        _lib.check(fn(P(g32), P(img), P(a["y"]), P(a["img_max"]), P(a["tc"]), P(a["tp"]), P(psf), P(a["otf"]), P(a["spec"]), P(gp),
                      P(out), P(ws), ws.numel(), B, N, _stream()))
    assert bits_equal(gi[0], gi[1])


# ------------------------------------------------------------------------------------------------------------ module level
def test_graphed_u8_step():
    """graphed() from uint8: the replay repeats itself, equals the graphed step on the converted batch bit for bit, and agrees
    with the eager step to the rounding of the eager (cooperative) PSF chain (bit for bit under B200CAM_COOP=0: see
    test_u8_under_switches)"""
    N, B = 128, 4
    u = u8_images(B, N, seed=11)
    g = (synth.upstream_grad(B, N, seed=4) * 1e-2).to(DEV)
    res = []
    for img in (u, u.to(torch.float32).div_(255.0)):
        cam = camera(N, seed=3)
        step = cam.graphed(img)
        outs = []
        for _ in range(2):
            cam.Zer_train.grad = None
            y, rad, cen = step(img)
            torch.autograd.backward([y, rad, cen], [g, torch.tensor(0.3, device=DEV), torch.tensor(1.7, device=DEV)])
            outs.append((y.detach().clone(), rad.detach().clone(), cen.detach().clone(), cam.Zer_train.grad.clone()))
        for p, q in zip(outs[0], outs[1]):
            assert bits_equal(p, q)
        res.append((outs[0], cam))
    for p, q in zip(res[0][0], res[1][0]):
        assert bits_equal(p, q)
    e = face_step(res[0][1], u, g)
    assert rel_l2(e[0], res[0][0][0]) <= 1e-4
    assert rel_l2(e[4], res[0][0][3]) <= 1e-3


@pytest.mark.parametrize("dtype", [torch.float32, BF16])
@pytest.mark.parametrize("overlap", [True, False])
def test_u8_node_keeps_the_uint8_image_and_no_fp32_copy(overlap, dtype):
    N, B = 64, 3
    u = u8_images(B, N, seed=5)
    cam = camera(N)
    cam.overlap_psf = overlap
    cam.sensor_dtype = dtype
    packed = []

    def pack(t):
        packed.append(t)
        return t

    with torch.autograd.graph.saved_tensors_hooks(pack, lambda t: t):
        y = cam(u)
    img_sized = [t for t in packed if tuple(t.shape) == (B, 3, N, N)]
    assert any(t.dtype == torch.uint8 and t.data_ptr() == u.data_ptr() for t in img_sized)
    fp32 = [t for t in img_sized if t.dtype == torch.float32]
    if dtype == torch.float32:
        assert len(fp32) == 1 and fp32[0].data_ptr() == y.data_ptr()     # the fp32 node keeps its own sensor image, no more
    else:
        assert fp32 == []
    y.float().sum().backward()


def test_u8_step_peak_memory_drops_by_the_fp32_batch():
    N, B = 256, 64
    u = u8_images(B, N, seed=7)
    g = (synth.upstream_grad(B, N, seed=8) * 1e-2).to(DEV)
    cam = camera(N)

    def peak(convert):
        face_step(cam, u.to(torch.float32).div_(255.0) if convert else u, g)      # warm: plan, workspace, tables
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        start = torch.cuda.memory_allocated()
        out = face_step(cam, u.to(torch.float32).div_(255.0) if convert else u, g)
        torch.cuda.synchronize()
        del out
        return torch.cuda.max_memory_allocated() - start

    old, new = peak(True), peak(False)
    assert old - new >= B * 3 * N * N * 4, (old, new)


def test_rows_u8_refuses_the_plane_layout_only_when_selected():
    """without B200CAM_PLANE=1 the uint8 split forward runs at N = 256 (with it: E_BAD_SIZE, checked in the switch runs)"""
    N, B = 256, 2
    plan = F.DevicePlan(N, DEV)
    u = u8_images(B, N, seed=2)
    spec = torch.empty(plan.lib.b200cam_spectrum_bytes(N, B) // 4, device=DEV)
    mx, tc = torch.empty(B, device=DEV), torch.empty(B, dtype=torch.int32, device=DEV)
    rc = plan.lib.b200cam_sensor_rows_u8(_lib.ptr(u), _lib.ptr(spec), _lib.ptr(mx), _lib.ptr(tc), B, N, _stream())
    assert rc == (-1 if F.PLANE_KERNELS else 0)


@pytest.mark.parametrize("switch", ["B200CAM_TIE_SPECTRAL=1", "B200CAM_ONE_PASS=1", "B200CAM_PLANE=1", "B200CAM_COOP=0"])
def test_u8_under_switches(switch):
    """the same equality under the opt-in switches (read once per process: a subprocess per switch, tests/u8_switch_runner.py).
    B200CAM_PLANE=1 at N = 256 converts with torch for the fp32 image (the plane kernels read fp32 only) and runs the uint8
    kernels for bf16; B200CAM_COOP=0 also checks graphed() from uint8 against the eager step, bit for bit."""
    k, v = switch.split("=")
    res = subprocess.run([sys.executable, str(REPO / "tests" / "u8_switch_runner.py")], capture_output=True, text=True,
                         timeout=900, env=dict(os.environ, **{k: v}))
    assert res.returncode == 0 and "ok=True" in res.stdout, (res.stdout + res.stderr)[-3000:]
