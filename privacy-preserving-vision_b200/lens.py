"""``OpticsZernike`` - drop-in for the Image_Caption optical encoder (``Image_Caption/Camera/Lens.py:11``).

Same constructor signature, parameters / ``state_dict`` keys (``zernike_coeffs_no_train`` (3,1,1),
``zernike_coeffs_no_train2`` (T-4,1,1), ``zernike_coeffs_train`` (1,1)), ``forward`` signature and
4-tuple result ``(sensor_img, psf, zernike_coeffs_concat, loss)``.

What runs where (everything below the Zernike coefficients is b200cam kernels, ``include/b200cam.h``)
* height map: ``b200cam_zernike_fwd_ex / _bwd_ex`` over the support of the basis; the partial sum of the frozen terms (349 of 350 as
  shipped) is cached, so a step reads one basis plane each way (``_height_map``);
* PSF synthesis (``Lens.py:176-274``: phase plate with the reference's ``torch.rand`` tolerance noise, spherical wavefront,
  aperture, Fresnel propagation on a (3/2 * wave_res)^2 grid - 1344^2 = 2^6*3*7 for the shipped config - intensity, area
  down-sampling, per-channel normalisation, disc masks and energy loss) and its adjoint into the height map:
  ``b200cam_lens_psf_fwd / _bwd`` (``csrc/lens_psf.cu``: pruned mixed-radix transforms, complex64), class ``LensPsf``;
* sensor image (``img_psf_conv``, ``Utils.py:251-297`` + the batch-global max of ``Lens.py:312``): ``b200cam_lens_sensor_*``
  (``csrc/lens_conv.cu``: zero padding, abs, crop, nearest resize and the maximum inside the transform kernels), class
  ``LensSensor``; with ``data_parallel(group)`` the maximum, sum(g*y) and the tie count are all-reduced, so N ranks reproduce
  the 1-GPU result;
* geometries the kernels do not cover (padded size with a prime factor above 31; patch sizes whose doubled size is not a power of
  two, e.g. the constructor default 368) use the reference's own torch expression on the GPU (``_psf``, ``_sensor_torch``,
  ``CircConv`` / ``CropAbsResize`` / ``GlobalMaxNormalise``).

Read-out (no reference counterpart, same meaning as on the Face-DeId ``Camera``)
* uint8 images (B,3,P,P) are accepted as they are: the row kernel reads them (``b200cam_lens_sensor_fwd_u8``) as
  ``img.float() / 255.0``, bit for bit, so the host-to-device copy is a quarter of the fp32 one; the other geometries convert
  with that torch expression;
* ``sensor_noise_sigma`` / ``sensor_quant_bits`` (default 0 / 0 = the reference): y += sigma * noise, then
  y = round(clamp(y, 0, 1) * L) / L, L = 2^bits - 1, applied after the batch-global max by the normalise kernel
  (``b200cam_lens_normalise_ex``; the torch expression elsewhere), straight through in backward.  ``forward(..., noise=)``
  takes the standard-normal tensor; otherwise it is drawn with ``torch.randn`` after the lens tolerance field.  With
  ``data_parallel`` each rank draws the noise of its own shard.  ``sensor_noise_rng = "philox"``: a key is drawn there instead
  and the normalise kernel draws the noise (``b200cam_lens_normalise_ex`` with ``B200CAM_SENSOR_NOISE_PHILOX``; the other
  geometries use its materialised values, ``F.philox_normal``); sharded batches then get the one-GPU noise;
* ``sensor_dtype`` (default torch.float32): torch.bfloat16 returns the sensor image in bf16 for a bf16 encoder - the normalise
  kernel rounds the fp32 result to nearest-even (``b200cam_lens_normalise_bf16``) and the backward reads the bf16 gradient as it
  is (``_dot_bf16`` / ``_bwd_bf16``); the other geometries cast with torch.  Bit for bit the fp32 module followed by
  ``.to(torch.bfloat16)``.

Not reproduced: comet.ml summaries (``attach_summaries``), the ``psf_lab`` image file path, ``upsample=True``
(1792^2 convolution, not a power of two) - they raise ``NotImplementedError`` - and the side effect of caching the
Zernike volume as ``zernike_volumes/*.npy`` in the working directory (``Lens.py:66-75``).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch
from torch import nn
from torch.nn import functional as TF

from . import _lib
from . import functional as F
from .zernike import zernike_volume as _zernike_volume


def get_zernike_volume(resolution, n_terms, scale_factor=1e-6):
    """Noll Zernike stack in metres (reference: ``Image_Caption/Camera/Utils.py:75-77``, via poppy)."""
    return _zernike_volume(resolution, n_terms, scale_factor)


def _disc_masks(size: int = 256, radius: int = 32):
    """mask_1 (1 outside the disc) and mask_2 (1 inside), (size,size,3) fp64, as drawn by ``cv2.circle`` with
    ``thickness=-1`` at ``Lens.py:113-129``."""
    try:
        import cv2
        m1 = np.ones((size, size, 3))
        cv2.circle(img=m1, center=[size // 2, size // 2], radius=radius, color=0, thickness=-1, lineType=cv2.FILLED)
        m2 = np.zeros((size, size, 3))
        cv2.circle(img=m2, center=[size // 2, size // 2], radius=radius, color=(255, 255, 255), thickness=-1,
                   lineType=cv2.FILLED)
        m2 = m2 / m2.max()
    except ImportError:       # same disc from its definition when OpenCV is not installed
        yy, xx = np.mgrid[0:size, 0:size]
        inside = ((xx - size // 2) ** 2 + (yy - size // 2) ** 2 <= radius ** 2).astype(np.float64)
        m2 = np.repeat(inside[:, :, None], 3, axis=2)
        m1 = 1.0 - m2
    return torch.from_numpy(m1), torch.from_numpy(m2)


class CircConv(torch.autograd.Function):
    """out = irfft2(rfft2(img) * rfft2(roll(kernel, -N/2))) per channel, N a power of two (b200cam_conv_fwd/bwd)."""

    @staticmethod
    @F.nvtx("b200cam.CircConv.forward")
    def forward(ctx, img: torch.Tensor, kernel: torch.Tensor, plan: F.DevicePlan):
        N = plan.N
        x = F._as_f32(img.detach(), plan.device)
        k = F._as_f32(kernel.detach(), plan.device).reshape(3, N, N)
        B = x.shape[0]
        out = torch.empty_like(x)
        otf = torch.empty(plan.otf_floats, dtype=torch.float32, device=plan.device)
        spectrum = None
        if any(ctx.needs_input_grad[:2]):
            spectrum = torch.empty(plan.lib.b200cam_spectrum_bytes(N, B) // 4, dtype=torch.float32, device=plan.device)
        ws = plan.sensor_workspace(B)
        with torch.cuda.device(plan.index):
            _lib.check(plan.lib.b200cam_conv_fwd(_lib.ptr(x), _lib.ptr(k), _lib.ptr(out), _lib.ptr(otf), _lib.ptr(spectrum),
                                                 _lib.ptr(ws), ws.numel(), B, N, F._stream()))
        ctx.plan, ctx.spectrum, ctx.kshape = plan, spectrum, kernel.shape
        ctx.save_for_backward(x, otf)
        return out

    @staticmethod
    @F.nvtx("b200cam.CircConv.backward")
    def backward(ctx, g):
        plan: F.DevicePlan = ctx.plan
        N = plan.N
        x, otf = ctx.saved_tensors
        B = x.shape[0]
        gc = F._as_f32(g, plan.device)
        grad_k = torch.empty(3, N, N, dtype=torch.float32, device=plan.device)
        grad_img = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        ws = plan.sensor_workspace(B)
        with torch.cuda.device(plan.index):
            _lib.check(plan.lib.b200cam_conv_bwd(_lib.ptr(gc), _lib.ptr(x), _lib.ptr(otf), _lib.ptr(ctx.spectrum),
                                                 _lib.ptr(grad_k), _lib.ptr(grad_img), _lib.ptr(ws), ws.numel(), B, N,
                                                 F._stream()))
        return grad_img, grad_k.reshape(ctx.kshape), None


class CropAbsResize(torch.autograd.Function):
    """``abs`` -> ``[off : off+P-1]`` crop -> nearest resize back to P (``out[i] = crop[max(i-1, 0)]``) of the padded
    convolution output, ``Image_Caption/Camera/Utils.py:289-295``, in one kernel each way (b200cam_crop_abs_resize_*)."""

    @staticmethod
    @F.nvtx("b200cam.CropAbsResize.forward")
    def forward(ctx, conv: torch.Tensor, P: int, off: int, plan: F.DevicePlan):
        c = F._as_f32(conv.detach(), plan.device)
        B, C, n, _ = c.shape
        out = torch.empty(B, C, P, P, dtype=torch.float32, device=plan.device)
        if B * C > 0:
            with torch.cuda.device(plan.index):
                _lib.check(plan.lib.b200cam_crop_abs_resize_fwd(_lib.ptr(c), _lib.ptr(out), B * C, n, P, off, F._stream()))
        ctx.plan, ctx.geom = plan, (P, off)
        ctx.save_for_backward(c)
        return out

    @staticmethod
    @F.nvtx("b200cam.CropAbsResize.backward")
    def backward(ctx, g):
        plan: F.DevicePlan = ctx.plan
        (c,) = ctx.saved_tensors
        P, off = ctx.geom
        B, C, n, _ = c.shape
        gc = torch.empty_like(c)
        if B * C > 0:
            go = F._as_f32(g, plan.device)
            with torch.cuda.device(plan.index):
                _lib.check(plan.lib.b200cam_crop_abs_resize_bwd(_lib.ptr(go), _lib.ptr(c), _lib.ptr(gc), B * C, n, P, off,
                                                                F._stream()))
        return gc, None, None, None


class GlobalMaxNormalise(torch.autograd.Function):
    """y = x / max(x) over the whole batch (``Lens.py:312``); with a process group the max is taken over all ranks
    and the backward's arg-max term (-sum(g*y)/m at the arg-max) is routed to the rank that owns it."""

    @staticmethod
    @F.nvtx("b200cam.GlobalMaxNormalise.forward")
    def forward(ctx, x: torch.Tensor, group):
        import torch.distributed as dist
        m_local = x.max()
        m = m_local.clone()
        if group is not None and dist.is_initialized():
            dist.all_reduce(m, op=dist.ReduceOp.MAX, group=group)
        y = x / m
        ctx.group = group
        ctx.save_for_backward(y, m, m_local)
        return y

    @staticmethod
    @F.nvtx("b200cam.GlobalMaxNormalise.backward")
    def backward(ctx, g):
        import torch.distributed as dist
        y, m, m_local = ctx.saved_tensors
        s = (g * y).sum()
        if ctx.group is not None and dist.is_initialized():
            dist.all_reduce(s, op=dist.ReduceOp.SUM, group=ctx.group)
        # only the rank that holds the maximum carries the arg-max term (no host sync: a 0/1 factor);
        # exact ties are split evenly like torch's max() backward (cross-rank exact ties: measure zero, not split)
        owner = (m_local == m).to(g.dtype)
        ties = (y == 1).to(g.dtype)
        n = ties.sum().clamp(min=1)
        return g / m - ties * (owner * s / (m * n)), None


class LensSensor(torch.autograd.Function):
    """sensor = |img_psf_conv(img, psf)| / max over the whole batch (Utils.py:251-297 + Lens.py:312) on the pruned kernels of
    ``csrc/lens_conv.cu``: the zero-padded image and the padded convolution output are never materialised.  With a process
    group the maximum is all-reduced (MAX) and, in the backward, sum(g*y) and the tie count (SUM): N ranks reproduce the
    one-GPU result, the arg-max term landing on the rank(s) that hold the maximum.
    ``img`` may be fp32 or uint8 (read by the row kernel as img / 255.0).  ``epilogue``: None or (noise, noise_scale,
    quant_bits) of ``F.read_out``, applied by the normalise kernel after the maximum; straight through in backward.
    ``out_dtype`` torch.bfloat16: the normalise kernel writes y in bf16 (its fp32 value rounded to nearest-even) and the bf16
    gradient is read by the dot and row kernels as it is - the fp32 backward on g.float(), bit for bit."""

    @staticmethod
    @F.nvtx("b200cam.LensSensor.forward")
    def forward(ctx, img: torch.Tensor, kpad: torch.Tensor, plan: F.DevicePlan, group, epilogue=None,
                out_dtype: torch.dtype = torch.float32):
        import torch.distributed as dist
        dev, n = plan.device, plan.N
        P = n // 2
        lib = plan.lib
        if img.dtype == torch.uint8:
            if img.device != dev:
                raise RuntimeError(f"b200cam: tensor on {img.device}, camera tables on {dev}")
            x, fwd = img.detach().contiguous(), lib.b200cam_lens_sensor_fwd_u8
        else:
            x, fwd = F._as_f32(img.detach(), dev), lib.b200cam_lens_sensor_fwd
        k = F._as_f32(kpad.detach(), dev).reshape(3, n, n)
        B = x.shape[0]
        flags, noise, noise_scale, quant_bits = F.epilogue_flags(epilogue, x.shape, dev)
        raw = torch.empty(x.shape, dtype=torch.float32, device=dev)
        bf16 = out_dtype == torch.bfloat16
        y = torch.empty(x.shape, dtype=out_dtype, device=dev)
        gmax = torch.zeros(1, dtype=torch.float32, device=dev)
        otf = torch.empty(plan.otf_floats, dtype=torch.float32, device=dev)
        spectrum = torch.empty(lib.b200cam_spectrum_bytes(n, B) // 4, dtype=torch.float32, device=dev)
        ws = torch.empty(lib.b200cam_lens_sensor_workspace_bytes(P, B), dtype=torch.uint8, device=dev)
        with torch.cuda.device(plan.index):
            _lib.check(fwd(_lib.ptr(x), _lib.ptr(k), _lib.ptr(raw), _lib.ptr(gmax), _lib.ptr(otf), _lib.ptr(spectrum), _lib.ptr(ws),
                           ws.numel(), B, P, F._stream()))
            if group is not None and dist.is_initialized():
                dist.all_reduce(gmax, op=dist.ReduceOp.MAX, group=group)
            normalise = lib.b200cam_lens_normalise_bf16 if bf16 else lib.b200cam_lens_normalise_ex
            _lib.check(normalise(_lib.ptr(raw), _lib.ptr(gmax), _lib.ptr(y), raw.numel(), F._stream(), flags,
                                 _lib.ptr(noise), float(noise_scale), int(quant_bits)))
        ctx.plan, ctx.group, ctx.kshape = plan, group, kpad.shape
        ctx.spectrum = spectrum if any(ctx.needs_input_grad[:2]) else None
        ctx.save_for_backward(raw, gmax, otf)
        return y

    @staticmethod
    @F.nvtx("b200cam.LensSensor.backward")
    def backward(ctx, g):
        import torch.distributed as dist
        plan: F.DevicePlan = ctx.plan
        raw, gmax, otf = ctx.saved_tensors
        dev, n = plan.device, plan.N
        P, B = n // 2, raw.shape[0]
        lib = plan.lib
        if g.dtype == torch.bfloat16:         # bf16 sensor image: the kernels widen the gradient themselves
            if g.device != dev:
                raise RuntimeError(f"b200cam: tensor on {g.device}, camera tables on {dev}")
            gy, sdot, sbwd = g.contiguous(), lib.b200cam_lens_sensor_dot_bf16, lib.b200cam_lens_sensor_bwd_bf16
        else:
            gy, sdot, sbwd = F._as_f32(g, dev), lib.b200cam_lens_sensor_dot, lib.b200cam_lens_sensor_bwd
        dot = torch.empty(2, dtype=torch.float32, device=dev)
        grad_k = torch.empty(3, n, n, dtype=torch.float32, device=dev)
        grad_img = torch.empty_like(raw) if ctx.needs_input_grad[0] else None
        ws = torch.empty(lib.b200cam_lens_sensor_workspace_bytes(P, B), dtype=torch.uint8, device=dev)
        with torch.cuda.device(plan.index):
            _lib.check(sdot(_lib.ptr(gy), _lib.ptr(raw), _lib.ptr(gmax), _lib.ptr(dot), _lib.ptr(ws), ws.numel(),
                                                   B, P, F._stream()))
            if ctx.group is not None and dist.is_initialized():
                dist.all_reduce(dot, op=dist.ReduceOp.SUM, group=ctx.group)
            coef = (dot[0] / (gmax[0] * dot[1].clamp(min=1.0))).reshape(1)      # s / (m n); torch.max splits exact ties evenly
            _lib.check(sbwd(_lib.ptr(gy), _lib.ptr(raw), _lib.ptr(gmax), _lib.ptr(coef), _lib.ptr(otf),
                                                   _lib.ptr(ctx.spectrum), _lib.ptr(grad_k), _lib.ptr(grad_img), _lib.ptr(ws),
                                                   ws.numel(), B, P, F._stream()))
        return grad_img, grad_k.reshape(ctx.kshape), None, None, None, None


class LensPsf(torch.autograd.Function):
    """height map (R,R) [+ tolerance noise] -> normalised PSF (1,P,P,3) and the energy loss, Lens.py:176-274, on the
    b200cam kernels of ``csrc/lens_psf.cu`` (phase plate, pruned mixed-radix Fresnel propagation, intensity, area
    down-sampling, per-channel normalisation, masks / loss) with the closed-form adjoint chain as backward.
    ``flags``: 1 = energy loss against mask_1 (prueba "1"/"3"), 2 = multiply by mask_2 (prueba "2"/"3")."""

    @staticmethod
    @F.nvtx("b200cam.LensPsf.forward")
    def forward(ctx, h: torch.Tensor, noise, c: dict, flags: int, R: int, P: int, lib):
        dev = h.device
        hh = F._as_f32(h.detach(), dev).reshape(R, R)
        nz = F._as_f32(noise.detach(), dev).reshape(R, R) if noise is not None else None
        field = torch.empty(3, R, R, 2, dtype=torch.float32, device=dev)
        U = torch.empty(3, R, R, 2, dtype=torch.float32, device=dev)
        psf = torch.empty(1, P, P, 3, dtype=torch.float32, device=dev)
        psf_out = torch.empty(1, P, P, 3, dtype=torch.float64, device=dev)
        chan_sum = torch.empty(3, dtype=torch.float32, device=dev)
        loss = torch.zeros((), dtype=torch.float64, device=dev)
        ws = torch.empty(lib.b200cam_lens_psf_workspace_bytes(R, P), dtype=torch.uint8, device=dev)
        m1, m2 = (c["mask1"] if flags & 1 else None), (c["mask2"] if flags & 2 else None)
        with torch.cuda.device(dev):
            _lib.check(lib.b200cam_lens_psf_fwd(_lib.ptr(hh), _lib.ptr(nz), _lib.ptr(c["A"]), c["delta_c"], _lib.ptr(c["Hx"]),
                                                _lib.ptr(c["tw"]), _lib.ptr(field), _lib.ptr(U), _lib.ptr(psf), _lib.ptr(chan_sum),
                                                _lib.ptr(m1), _lib.ptr(m2), flags, _lib.ptr(psf_out), _lib.ptr(loss),
                                                _lib.ptr(ws), ws.numel(), R, P, F._stream()))
        ctx.c, ctx.flags, ctx.geom, ctx.lib, ctx.hshape = c, flags, (R, P), lib, h.shape
        ctx.save_for_backward(psf, chan_sum, field, U, loss)
        # the reference's PSF is fp32 until an fp64 mask promotes it (Lens.py:239 vs :274)
        return (psf_out if flags & 2 else psf), (loss if flags & 1 else None)

    @staticmethod
    @F.nvtx("b200cam.LensPsf.backward")
    def backward(ctx, g_psf, g_loss):
        psf, chan_sum, field, U, loss = ctx.saved_tensors
        c, flags, (R, P), lib = ctx.c, ctx.flags, ctx.geom, ctx.lib
        dev = psf.device
        gp = g_psf.detach().to(device=dev, dtype=torch.float64).contiguous() if g_psf is not None else None
        gl = g_loss.detach().to(device=dev, dtype=torch.float64).reshape(()).contiguous() if g_loss is not None else None
        grad_h = torch.empty(R, R, dtype=torch.float32, device=dev)
        ws = torch.empty(lib.b200cam_lens_psf_workspace_bytes(R, P), dtype=torch.uint8, device=dev)
        m1, m2 = (c["mask1"] if flags & 1 else None), (c["mask2"] if flags & 2 else None)
        with torch.cuda.device(dev):
            _lib.check(lib.b200cam_lens_psf_bwd(_lib.ptr(gp), _lib.ptr(gl), _lib.ptr(loss), _lib.ptr(psf), _lib.ptr(chan_sum),
                                                _lib.ptr(field), _lib.ptr(U), c["delta_c"], _lib.ptr(c["Hx"]), _lib.ptr(c["tw"]),
                                                _lib.ptr(m1), _lib.ptr(m2), flags, _lib.ptr(grad_h), _lib.ptr(ws), ws.numel(),
                                                R, P, F._stream()))
        return grad_h.reshape(ctx.hshape), None, None, None, None, None, None


class OpticsZernike(nn.Module):
    def __init__(self,
                 input_shape,
                 device,
                 experiment=None,
                 sensor_distance=25e-3,
                 refractive_idcs=np.array([1.499, 1.493, 1.488]),
                 wave_lengths=np.array([460, 550, 640]) * 1e-9,
                 height_tolerance=20e-9,
                 wave_resolution=(736, 736),
                 patch_size=368,
                 sample_interval=2e-6,
                 upsample=False,
                 frames=8,
                 optics_cfg=1,
                 zernike_terms=350,
                 mask_1=None,
                 mask_2=None):
        super().__init__()
        self.device = device
        self.sensor_distance = sensor_distance
        self.height_tolerance = height_tolerance
        self.upsample = upsample
        self.patch_size = patch_size
        self.wave_lengths = np.asarray(wave_lengths, dtype=np.float64)
        self.sample_interval = sample_interval
        self.refractive_idcs = np.asarray(refractive_idcs, dtype=np.float64)
        self.frames = frames
        self.optics_cfg = optics_cfg
        self.zernike_terms = zernike_terms
        self.wave_res = [patch_size * 4, patch_size * 4] if wave_resolution is None else list(wave_resolution)
        self.physical_size = float(self.wave_res[0] * self.sample_interval)
        self.channels = input_shape[-1]
        if self.channels != 3 or len(self.wave_lengths) != 3:
            raise ValueError("the camera models three wavelengths / colour channels")

        vol = get_zernike_volume(resolution=self.wave_res[0], n_terms=self.zernike_terms).astype(np.float32)
        self.zernike_volume = torch.tensor(vol, dtype=torch.float32, device=self.device)
        num = self.zernike_volume.shape[0]
        inits = np.zeros((num, 1, 1))
        inits[3] = -22                                           # defocus (Lens.py:88)
        self.zernike_coeffs_no_train = nn.Parameter(torch.tensor(inits[:3, ...], dtype=torch.float32),
                                                    requires_grad=False)
        self.zernike_coeffs_no_train2 = nn.Parameter(torch.tensor(inits[4:, ...], dtype=torch.float32),
                                                     requires_grad=False)
        self.zernike_coeffs_train = nn.Parameter(torch.tensor(inits[3, ...], dtype=torch.float32))

        self.training_info = None
        self.gpu_rank = None
        self.experiment = experiment
        m1, m2 = _disc_masks()
        self.mask_1 = m1.to(self.device)
        self.mask_2 = m2.to(self.device)

        # opt-in sensor read-out, as on the Face-DeId Camera (the reference's gaussian_noise call is commented out, Lens.py:295-301):
        # additive Gaussian noise of this standard deviation on the normalised sensor image, then quantisation to this many
        # bits; 0 / 0 = the reference
        self.sensor_noise_sigma = 0.0
        self.sensor_quant_bits = 0
        # dtype of the returned sensor image, as on Camera: torch.float32 (the reference) or torch.bfloat16 for a downstream
        # encoder that runs in bf16 - exactly the fp32 image .to(torch.bfloat16), written by the normalise kernel; backward =
        # the fp32 one on g.float().  PSF, coefficients, loss and dL/dimg keep their dtypes.  Set by the caller.
        self.sensor_dtype = torch.float32
        # generator of the opt-in sensor noise, as on Camera: "torch" (torch.randn tensor) or "philox" (drawn in the normalise
        # kernel from a key drawn with torch.randint; the key of the last forward is `sensor_noise_seed`)
        self.sensor_noise_rng = "torch"
        self.sensor_noise_seed = None
        self._const: dict = {}           # per-device constant tables (wavefront, aperture, transfer function)
        self._plans: dict = {}
        self._process_group = None

    # ------------------------------------------------------------------ helpers
    def data_parallel(self, process_group=None, enabled: bool = True):
        """Batch sharded over ranks: the batch-global max of ``Lens.py:312`` is all-reduced (one float) in forward
        and its arg-max term routed to the owning rank in backward."""
        import torch.distributed as dist
        self._process_group = (process_group or dist.group.WORLD) if enabled else None
        return self

    def _project(self, coeffs: torch.Tensor) -> torch.Tensor:
        """sum_j coef_j Z_j (Lens.py:176).  The basis volume is 1.12 GB at the shipped 896^2 x 350: on CUDA it is read
        once by b200cam_zernike_fwd (and once by its adjoint) instead of materialising coef * volume."""
        vol = self.zernike_volume
        if coeffs.is_cuda and vol.is_cuda and vol.dtype == torch.float32 and vol.is_contiguous() and vol[0].numel() % 4 == 0:
            return F.zernike_project(coeffs, vol, self._plan(vol.device, 256))      # any plan of that device will do
        return torch.sum(coeffs * vol, dim=0)

    def _height_map(self, coeffs: torch.Tensor) -> torch.Tensor:
        """h = sum_j coef_j Z_j for the module's own coefficient vector.  As shipped only the defocus term (#3) is trainable
        (Lens.py:90-96): the partial sum of the T-1 frozen terms is cached - keyed on the frozen parameters' version counters,
        so an in-place update or load_state_dict refreshes it - and a step reads one basis plane each way instead of the
        whole T x R x R volume (1.12 GB at 350 x 896^2)."""
        vol = self.zernike_volume
        frozen_ok = (not self.zernike_coeffs_no_train.requires_grad and not self.zernike_coeffs_no_train2.requires_grad
                     and coeffs.is_cuda and vol.is_cuda and vol.shape[0] > 4)
        if not frozen_ok:
            return self._project(coeffs)
        key = (self.zernike_coeffs_no_train._version, self.zernike_coeffs_no_train2._version,
               self.zernike_coeffs_no_train.data_ptr(), self.zernike_coeffs_no_train2.data_ptr(), vol.data_ptr())
        if getattr(self, "_frozen_key", None) != key:
            with torch.no_grad():
                c = coeffs.detach().clone()
                c[3] = 0
                self._frozen_sum = self._project(c)
            self._frozen_key = key
        return self._frozen_sum + self._project_one(self.zernike_coeffs_train.reshape(1, 1, 1), vol[3:4])

    def invalidate_cache(self) -> None:
        """Drop the cached partial sum of the frozen Zernike terms.  In-place updates of the frozen parameters and
        ``load_state_dict`` are detected through the tensors' version counters; writes through ``param.data`` are not -
        call this after such a write."""
        self._frozen_key = None
        self._frozen_sum = None

    def _project_one(self, coef: torch.Tensor, plane: torch.Tensor) -> torch.Tensor:
        if plane.dtype == torch.float32 and plane.is_contiguous() and plane[0].numel() % 4 == 0:
            return F.zernike_project(coef, plane, self._plan(plane.device, 256))
        return torch.sum(coef * plane, dim=0)

    def get_Heith_Map(self):
        coeffs = torch.cat((self.zernike_coeffs_no_train, self.zernike_coeffs_train.unsqueeze(0),
                            self.zernike_coeffs_no_train2), 0)
        return self._project(coeffs).unsqueeze(0)

    def _constants(self, dev: torch.device):
        """Spherical wavefront (Lens.py:191-210), aperture (Utils.py:88-97) and Fresnel transfer function
        (Utils.py:329-373): built in fp64 with numpy exactly like the reference, once per device."""
        key = (dev, self.optics_cfg)
        c = self._const.get(key)
        if c is not None:
            return c
        N, M = self.wave_res
        x, y = np.mgrid[-N // 2:N // 2, -M // 2:M // 2].astype(np.float64)
        x = x / N * self.physical_size
        y = y / M * self.physical_size
        squared_sum = x ** 2 + y ** 2
        wave_nos = torch.tensor((2. * np.pi / self.wave_lengths).reshape([1, 1, 1, -1]))
        depth = 1 / 2 if self.optics_cfg == 1 else 1
        curvature = torch.sqrt(torch.tensor(squared_sum) + torch.tensor(depth, dtype=torch.float64) ** 2)
        phase = (wave_nos * curvature.unsqueeze(0).unsqueeze(-1)).to(torch.float64)
        wavefront = torch.cos(phase).to(torch.complex64) + 1.j * torch.sin(phase).to(torch.complex64)

        ax, ay = np.mgrid[-N // 2: N // 2, -M // 2: M // 2].astype(np.float64)
        r = np.sqrt(ax ** 2 + ay ** 2)[None, :, :, None]
        aperture = torch.tensor((r < np.amax(ax)).astype(np.float64))

        Mpad, Npad = N // 4, M // 4
        Mp, Np = N + 2 * Mpad, M + 2 * Npad
        fx, fy = np.mgrid[-Np // 2:Np // 2, -Mp // 2:Mp // 2]
        fx = np.fft.ifftshift(fx / (self.sample_interval * Np))
        fy = np.fft.ifftshift(fy / (self.sample_interval * Mp))
        sq = (np.square(fx) + np.square(fy))[None, :, :, None]
        expo = torch.tensor(np.float64(self.wave_lengths * np.pi * -1. * sq * self.sensor_distance), dtype=torch.float64)
        H = torch.cos(expo).to(torch.complex64) + 1.j * torch.sin(expo).to(torch.complex64)
        delta = torch.tensor((2. * np.pi / self.wave_lengths).reshape([1, 1, 1, -1])
                             * (self.refractive_idcs.reshape([1, 1, 1, -1]) - 1.))
        c = {"wavefront": wavefront.to(dev), "aperture": aperture.to(dev), "H": H.to(dev), "delta": delta.to(dev),
             "pad": (Mpad, Npad)}
        lib = _lib.load_library() if dev.type == "cuda" else None
        c["kernels"] = bool(lib is not None and N == M and lib.b200cam_lens_psf_supported(N, self.patch_size))
        if c["kernels"]:
            # tables of csrc/lens_psf.cu: A = aperture * wavefront, planar (3,R,R) complex64 (the aperture is 0/1: exact);
            # the transfer function as two 1-D fp64 factors H(fx,fy) = E(fx) E(fy), E = exp(-i pi lambda z f^2) in FFT order;
            # twiddles exp(-2 pi i k / n) rounded from fp64
            n = Np
            A = (aperture.to(torch.complex64) * wavefront)[0].permute(2, 0, 1).contiguous()
            f1 = np.fft.ifftshift(np.arange(-n // 2, n // 2) / (self.sample_interval * n))
            e1 = self.wave_lengths[:, None] * np.pi * -1. * np.square(f1)[None, :] * self.sensor_distance      # (3, n) fp64
            ang = -2.0 * np.pi * np.arange(n) / n
            c["A"] = torch.view_as_real(A).contiguous().to(dev)
            c["Hx"] = torch.tensor(np.stack([np.cos(e1), np.sin(e1)], axis=-1), dtype=torch.float64, device=dev).contiguous()
            c["tw"] = torch.tensor(np.stack([np.cos(ang), np.sin(ang)], axis=-1).astype(np.float32), device=dev).contiguous()
            c["delta_c"] = (ctypes.c_double * 3)(*[float(v) for v in delta.reshape(-1)])
            c["lib"] = lib
        self._const[key] = c
        return c

    def _plan(self, device: torch.device, n: int) -> F.DevicePlan:
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        plan = self._plans.get((device, n))
        if plan is None:
            plan = F.DevicePlan(n, device, tables=False)
            self._plans[(device, n)] = plan
        return plan

    def _psf_kernels(self, height_map: torch.Tensor, flags: int):
        """(psf, loss) through csrc/lens_psf.cu, or None when the geometry is outside what the kernels cover (padded
        size with a prime factor above 31, masks of another size): the caller then uses the torch expression."""
        c = self._constants(height_map.device)
        if not c["kernels"]:
            return None
        if flags:      # the disc masks are module attributes a caller may replace: follow them (fp64, on the device, contiguous)
            mkey = (self.mask_1.data_ptr(), self.mask_1._version, self.mask_2.data_ptr(), self.mask_2._version)
            if c.get("mask_key") != mkey:
                ok = tuple(self.mask_1.shape) == tuple(self.mask_2.shape) == (self.patch_size, self.patch_size, 3)
                dev = height_map.device
                c["mask1"] = self.mask_1.to(device=dev, dtype=torch.float64).contiguous() if ok else None
                c["mask2"] = self.mask_2.to(device=dev, dtype=torch.float64).contiguous() if ok else None
                c["mask_key"] = mkey
            if c["mask1"] is None:
                return None
        else:
            c.setdefault("mask1", None)
            c.setdefault("mask2", None)
        noise = None
        if self.height_tolerance is not None:                      # PhasePlate._build, Utils.py:396-406: same torch.rand call
            noise = ((-self.height_tolerance - self.height_tolerance)
                     * torch.rand(list(height_map.shape), dtype=height_map.dtype, device=height_map.device)
                     + self.height_tolerance)
        R = self.wave_res[0]
        return LensPsf.apply(height_map.reshape(R, R), noise, c, flags, R, self.patch_size, c["lib"])

    def _psf(self, height_map: torch.Tensor) -> torch.Tensor:
        """height map (1,R,R,1) -> normalised PSF (1,P,P,3)  (Lens.py:180-239), torch expression (geometries the kernels
        do not cover)."""
        c = self._constants(height_map.device)
        if self.height_tolerance is not None:                      # PhasePlate._build, Utils.py:396-406
            height_map = height_map + ((-self.height_tolerance - self.height_tolerance)
                                       * torch.rand(list(height_map.shape), dtype=height_map.dtype,
                                                    device=height_map.device) + self.height_tolerance)
        phi = (c["delta"] * height_map).to(torch.float64)          # Utils.py:192-205
        shifts = torch.cos(phi).to(torch.complex64) + 1.j * torch.sin(phi).to(torch.complex64)
        field = c["aperture"] * (shifts * c["wavefront"])          # Lens.py:212-213 (fp64 mask: complex128 from here)
        Mpad, Npad = c["pad"]
        padded = TF.pad(field, [0, 0, Npad, Npad, Mpad, Mpad])
        obj = torch.fft.fftn(padded.permute(0, 3, 1, 2), dim=[-1, -2]).permute(0, 2, 3, 1)
        out = torch.fft.ifftn((obj * c["H"]).permute(0, 3, 1, 2), dim=[-1, -2]).permute(0, 2, 3, 1)
        out = out[:, Mpad:-Mpad, Npad:-Npad, :]
        psf = torch.square(torch.abs(out))                         # get_intensities, Utils.py:208
        psf = self._area_downsample(psf, self.patch_size)
        return psf / torch.sum(psf, dim=[1, 2], keepdim=True)      # per channel (Lens.py:239)

    @staticmethod
    def _area_downsample(img: torch.Tensor, target: int) -> torch.Tensor:
        """area_downsampling_tf, Utils.py:216-248."""
        img = img.to(torch.float32)
        side = img.shape[1]
        x = img.permute(0, 3, 1, 2)
        if side % target == 0:
            f = side // target
            return TF.avg_pool2d(x, f, stride=f).permute(0, 2, 3, 1)
        lcm = abs(target * side) // np.gcd(target, side) / target
        up = 10 if lcm > 10 else int(lcm)
        x = TF.interpolate(x, size=2 * [up * target], mode="nearest")     # torchvision Resize(interpolation=0)
        return TF.avg_pool2d(x, up, stride=up).permute(0, 2, 3, 1)

    def _sensor(self, img: torch.Tensor, psf: torch.Tensor, epilogue=None, out_dtype: torch.dtype = torch.float32) -> torch.Tensor:
        """img_psf_conv (Utils.py:251-297): zero-pad to 2P, circular FFT convolution, abs, crop, nearest resize; then the batch-global
        max of Lens.py:312 and the opt-in read-out ``epilogue`` (``F.read_out``).  ``img``: fp32, or uint8 read as img / 255.0.
        ``out_dtype``: the fused kernels write bf16 themselves; the other geometries cast the fp32 result with torch."""
        P = img.shape[2]
        if img.dim() != 4 or img.shape[1] != 3 or img.shape[3] != P or psf.shape[1] != P:
            raise ValueError(f"expected images (B,3,{psf.shape[1]},{psf.shape[1]}), got {tuple(img.shape)}")
        if img.device.type != "cuda":
            raise RuntimeError("b200cam runs on CUDA (sm_100a) only; there is no CPU path")
        n = 2 * P
        pad = (n - P) / 2
        pt, pb = int(np.ceil(pad)), int(np.floor(pad))
        fused = P in (64, 128, 256, 512)
        if not fused and img.dtype == torch.uint8:       # the fused row kernel reads uint8 itself; elsewhere: torch's expression
            img = img.to(torch.float32) / 255.0
        if not fused and not _lib.load_library().b200cam_supported(n):
            # patch sizes whose padded transform is not a power of two (the constructor default 368 -> 736): the reference's
            # own expression on the GPU (torch.fft), so that every constructor-valid geometry runs
            y = GlobalMaxNormalise.apply(self._sensor_torch(img.to(torch.float32), psf, n, pt, pb), self._process_group)
            return self._read_out_torch(y, epilogue).to(out_dtype)
        x = None if fused else TF.pad(img.to(torch.float32), [pt, pb, pt, pb])
        # psf2otf (Utils.py:127-158): pad so that the PSF centre lands on n/2, the kernel's "centred frame"
        if (n - P) % 2 != 0:
            kt, kb = int(np.ceil(pad)), int(np.floor(pad))
        else:
            kt, kb = int(pad) + 1, int(pad) - 1
        k = TF.pad(psf[0].permute(2, 0, 1).to(torch.float32), [kt, kb, kt, kb])          # (3, n, n)
        plan = self._plan(img.device, n)
        if fused:      # padding, |.|, crop, resize, the batch-global max and the read-out inside the kernels (csrc/lens_conv.cu)
            return LensSensor.apply(img, k, plan, self._process_group, epilogue, out_dtype)
        # |.|, the [pt+1 : n-pb] crop to (P-1)^2 and the nearest resize back to P (out[i] = crop[max(i-1,0)]) in one pass
        out = CropAbsResize.apply(CircConv.apply(x, k, plan), P, pt + 1, plan)
        return self._read_out_torch(GlobalMaxNormalise.apply(out, self._process_group), epilogue).to(out_dtype)

    @staticmethod
    def _read_out_torch(y: torch.Tensor, epilogue) -> torch.Tensor:
        """The read-out epilogue of the kernels (kernels.cuh apply_epilogue) as torch ops, straight through in backward - for
        the geometries the fused kernels do not cover.  A Philox seed block is materialised with ``F.philox_normal``: the values the
        fused normalise kernel would draw for it."""
        if epilogue is None:
            return y
        noise, sigma, bits = epilogue
        z = y
        if noise is not None and noise.dtype == torch.int64:
            noise = F.philox_normal(noise, y.shape)
        if noise is not None:
            if noise.shape != y.shape:
                raise ValueError(f"sensor noise must have the shape of the images {tuple(y.shape)}, got {tuple(noise.shape)}")
            z = z + sigma * noise.to(y.dtype)
        if bits:
            L = float(2 ** bits - 1)
            z = torch.round(torch.clamp(z, 0.0, 1.0) * L) / L
        return y + (z - y).detach()

    @staticmethod
    def _sensor_torch(img: torch.Tensor, psf: torch.Tensor, n: int, pt: int, pb: int) -> torch.Tensor:
        """img_psf_conv (Utils.py:251-297) as torch ops on the image's device - only for patch sizes the kernels do not cover."""
        P = img.shape[2]
        pad = (n - P) / 2
        lo, hi = (int(np.ceil(pad)), int(np.floor(pad))) if (n - P) % 2 != 0 else (int(pad) + 1, int(pad) - 1)
        kern = TF.pad(psf[0].permute(2, 0, 1).to(torch.float32), [lo, hi, lo, hi])
        split = n - (n + 1) // 2
        order = torch.cat((torch.arange(split, n), torch.arange(split))).to(img.device)
        otf = torch.fft.fftn(kern[:, order][:, :, order].to(torch.complex64), dim=[-1, -2])
        x = TF.pad(img, [pt, pb, pt, pb])
        res = torch.abs(torch.fft.ifftn(torch.fft.fftn(x, dim=[-1, -2]) * otf[None], dim=[-1, -2]))
        res = res[:, :, pt + 1:n - pb, pt + 1:n - pb]
        return TF.interpolate(res, size=[P, P], mode="nearest")

    # ------------------------------------------------------------------ reference API
    def forward(self, input_img, new_zernike=None, prueba=None, psf_lab=None, enfoco=None, noise=None):
        """The reference's forward (Lens.py:157-316).  ``input_img``: (B,3,P,P) fp32, or uint8 (what a decoder or the caption
        HDF5 store yields; read as input_img / 255.0 on the GPU, a quarter of the host-to-device bytes).  ``noise``: optional
        standard-normal tensor shaped like the batch for the opt-in sensor noise (``sensor_noise_sigma``); with sigma > 0 and
        none given it is drawn with torch.randn AFTER the lens tolerance field, so a seeded run draws both in the same order.
        The sensor image is returned in ``sensor_dtype``.  With ``sensor_noise_rng = "philox"`` a key is drawn at that point
        instead and the normalise kernel draws the noise (``sensor_noise_seed``)."""
        out_dtype = F.check_sensor_dtype(self.sensor_dtype)
        rng = F.check_noise_rng(self.sensor_noise_rng)
        if psf_lab is True:
            raise NotImplementedError("psf_lab loads '../dataset_paula_real/psf_lab.jpg' in the reference (Lens.py:222-236)")
        if self.upsample:
            raise NotImplementedError("upsample=True convolves at the wave resolution (not a power of two)")
        coeffs = torch.cat((self.zernike_coeffs_no_train, self.zernike_coeffs_train.unsqueeze(0),
                            self.zernike_coeffs_no_train2), 0)
        if enfoco is True:                                          # Lens.py:160-162
            coeffs = coeffs.clone()
            coeffs[:] = 0
            coeffs[3] = -22
            height_map = self._project(coeffs).unsqueeze(0).unsqueeze(-1)
        else:
            height_map = self._height_map(coeffs).unsqueeze(0).unsqueeze(-1)
        flags = (1 if prueba in ("1", "3") else 0) | (2 if prueba in ("2", "3") else 0)
        fused = self._psf_kernels(height_map, flags) if height_map.is_cuda else None
        if fused is not None:
            psf, loss = fused
        else:
            psf = self._psf(height_map)
            loss = None
            if prueba == "1" or prueba == "3":
                loss = torch.norm((psf * self.mask_1) - psf)
            if prueba == "2" or prueba == "3":
                psf = psf * self.mask_2

        epilogue = (F.read_out(input_img, self.sensor_noise_sigma, self.sensor_quant_bits, noise, rng,
                               F.shard_first4(input_img, self._process_group))
                    if torch.is_tensor(input_img) else None)
        self.sensor_noise_seed = F.noise_seed(epilogue)
        sensor = self._sensor(input_img, psf, epilogue, out_dtype)
        np.random.uniform(low=0.001, high=0.02)                     # noise_sigma is drawn and discarded (Lens.py:295)
        return sensor, psf, coeffs, loss                            # (the batch-global max of Lens.py:312 is inside _sensor)

    def load_pretrained_from_numpy(self, path):
        weights = np.load(path)['optics_trained_weights']
        self.state_dict()['zernike_coeffs_train'].copy_(torch.tensor(weights))

    def load_pretrained_from_warmup(self, path):
        import os
        ckpt = torch.load(os.path.expanduser(path), map_location=self.device)
        self.state_dict()['zernike_coeffs_train'].copy_(ckpt['model_state_dict']['optics.zernike_coeffs_train'])

    def load_reference_state_dict(self, state: dict, strict: bool = True):
        """Load a camera checkpoint in EITHER of the reference's two parameterisations (SURVEY 8 f3):

        * shipped module (``Lens.py:92-96``): ``zernike_coeffs_no_train`` (3,1,1), ``zernike_coeffs_train`` (1,1) - the
          defocus term only - and ``zernike_coeffs_no_train2`` (T-4,1,1);
        * ``Camera/Model.pth`` as ``train.py:71-78`` reads it (the commented-out layout of ``Lens.py:99-101``):
          ``[optics.]zernike_coeffs_no_train`` (3,1,1) and ``[optics.]zernike_coeffs_train`` (T-3,1,1), i.e. every term
          from the defocus on in one tensor.  The reference's own ``load_state_dict`` rejects this one; here its first
          entry becomes the trainable defocus and the rest ``zernike_coeffs_no_train2``.

        A leading ``optics.`` on the keys and a wrapping ``{'model': ...}`` / ``{'model_state_dict': ...}`` are accepted."""
        for wrap in ("model", "model_state_dict"):
            if isinstance(state, dict) and wrap in state and isinstance(state[wrap], dict):
                state = state[wrap]
        sd = {(k[len("optics."):] if k.startswith("optics.") else k): v for k, v in state.items()}
        if "zernike_coeffs_no_train2" not in sd and "zernike_coeffs_train" in sd:
            tr = torch.as_tensor(sd["zernike_coeffs_train"])
            T = self.zernike_coeffs_no_train2.shape[0] + 4
            if tr.dim() == 3 and tr.shape[0] == T - 3:                  # legacy 3 + (T-3) layout
                sd = dict(sd)
                sd["zernike_coeffs_train"] = tr[0].reshape(self.zernike_coeffs_train.shape)
                sd["zernike_coeffs_no_train2"] = tr[1:]
        keys = ("zernike_coeffs_no_train", "zernike_coeffs_train", "zernike_coeffs_no_train2")
        return self.load_state_dict({k: sd[k] for k in keys if k in sd}, strict=strict)

