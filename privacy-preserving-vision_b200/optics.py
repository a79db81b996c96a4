"""``Camera`` - drop-in for the reference Face-DeId optical encoder (``Face-DeId/Camera/Optics.py:9``).

Same constructor, parameters / ``state_dict`` keys (``Zer_no_train``, ``Zer_train``, ``ca``),
public attributes and methods; ``forward`` / ``get_psf`` run in the b200cam CUDA kernels.

Differences a caller can observe (all documented in DESIGN.md):
* forward needs a CUDA device - there is no CPU path;
* the constant tensors (``XY``, ``FF``, ``rho`` ...) are built once; the kernel tables follow the
  input's device lazily, so ``Camera(...).cuda()`` works even though the reference keeps such
  tensors on the constructor device;
* optional ``data_parallel(group)`` all-reduces dL/dh across ranks inside backward.
"""
from __future__ import annotations

import numpy as np
import torch
from torch import nn

from . import constants as K
from . import functional as F
from .zernike import zernike_volume as _zernike_volume


def get_zernike_volume(resolution, n_terms, scale_factor=1e-6, height_tolerance=2e-8):
    """Noll Zernike stack in metres (reference: ``Face-DeId/Camera/Utils.py:60-63``, via poppy)."""
    return _zernike_volume(resolution, n_terms, scale_factor)


class Camera(nn.Module):
    def __init__(self, device="cpu", N=256, lamdas=3, zernike_terms=50, height_tolerance=2e-8):
        super().__init__()
        if lamdas != 3:
            raise ValueError("the optical model has three fixed wavelengths (640/550/440 nm)")
        self.lamdas = lamdas
        self.device = device
        self.height_tolerance = height_tolerance

        tables = K.build(N)
        self._tables = tables
        for name in ("zi", "z0", "f", "radii", "N", "c", "L_len", "px", "L_sen", "du", "dx2"):
            setattr(self, name, getattr(tables, name))
        self.R = tables.R.to(device) if torch.is_tensor(tables.R) else tables.R
        for name in K.TENSOR_ATTRS:
            setattr(self, name, getattr(tables, name).to(device))
        self.z = tables.z                      # the reference keeps this one on the CPU (Optics.py:36)

        # Zernike parameters: same RNG calls, in the same order, as Optics.py:59-70
        self.zernike_inits = torch.rand((zernike_terms, 1, 1), device=self.device) / 100
        self.zernike_inits[:3] = 0
        self.Zer_no_train = nn.Parameter(self.zernike_inits[:3, ...], requires_grad=False)
        self.Zer_train = nn.Parameter(self.zernike_inits[3:, ...], requires_grad=True)
        self.zernike_volume = torch.tensor(get_zernike_volume(resolution=self.N, n_terms=zernike_terms),
                                           dtype=torch.float32, device=self.device)
        size = (1, 1, 32, 32)
        self.ca = torch.where(torch.rand(size=size) > 0.5, torch.ones(size), torch.zeros(size))
        self.ca = nn.Parameter(self.ca, requires_grad=False)

        self.loss_psf = 0.0
        self.loss_rad = 0.0
        self.psfs = None
        self.centering_loss = None
        self.psf_rad = None

        # opt-in sensor read-out (north_star step 5; the reference has neither, SURVEY trap T6): additive Gaussian noise of this
        # standard deviation on the normalised sensor image, then quantisation to this many bits; 0 / 0 = the reference
        self.sensor_noise_sigma = 0.0
        self.sensor_quant_bits = 0
        # dtype of the returned sensor image: torch.float32 (the reference) or torch.bfloat16 for a downstream net that runs in
        # bf16 (torch.autocast).  bf16 = the fp32 image rounded to nearest-even, written by the kernels; its bf16 gradient is read
        # by them as it is (backward = the fp32 one on g.float()).  Set by the caller, never inferred from autocast.
        self.sensor_dtype = torch.float32
        # generator of the opt-in sensor noise: "torch" (the default: a torch.randn tensor shaped like the batch) or "philox" (the
        # normalise kernel draws it from a key drawn with torch.randint - no noise tensor; include/b200cam.h
        # B200CAM_SENSOR_NOISE_PHILOX).  The seed block {key, first4} of the last forward is `sensor_noise_seed` (None when the
        # kernels drew nothing): F.philox_normal(seed, shape) re-creates that step's noise.
        self.sensor_noise_rng = "torch"
        self.sensor_noise_seed = None
        self.overlap_psf = True         # run the PSF-independent half of forward() beside the PSF synthesis
        self._plans: dict[torch.device, F.DevicePlan] = {}
        self._pending_centering = None
        self._process_group = None
        self._average_grads = True

    # ------------------------------------------------------------------ kernels' per-device state
    def _plan(self, device: torch.device) -> F.DevicePlan:
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        plan = self._plans.get(device)
        if plan is None:
            plan = F.DevicePlan(self.N, device, self._tables)
            plan.process_group = self._process_group
            plan.average_grads = self._average_grads
            comm = getattr(self, "_peer_comm", None)
            plan.peer_comm = comm if comm is not None and comm.buf.device == device else None
            self._plans[device] = plan
        return plan

    def data_parallel(self, process_group=None, average: bool = True, enabled: bool = True, peer_memory: bool = True,
                      device=None):
        """All-reduce dL/dh (N*N floats) over ``process_group`` inside backward (one rank per GPU).

        With ``peer_memory`` (default, NCCL groups on CUDA) the all-reduce is fused into the last PSF-backward kernel
        over NVLink peer memory (``parallel.PeerComm``; a collective set-up happens here, so call it on every rank);
        otherwise, or if symmetric memory is unavailable, ``dist.all_reduce`` is used."""
        import torch.distributed as dist
        from .parallel import PeerComm
        self._process_group = (process_group or dist.group.WORLD) if enabled else None
        self._average_grads = average
        self._peer_comm = None
        if (enabled and peer_memory and torch.cuda.is_available() and dist.get_backend(self._process_group) == "nccl"
                and dist.get_world_size(self._process_group) > 1):
            dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
            try:
                F._lib.ensure_init(self.N, dev.index if dev.index is not None else torch.cuda.current_device())
                self._peer_comm = PeerComm(self.N, dev, self._process_group)
            except Exception as exc:      # no symmetric memory on this system: NCCL path
                import warnings
                warnings.warn(f"b200cam: peer-memory all-reduce unavailable ({exc}); using dist.all_reduce")
                self._peer_comm = None
        for plan in self._plans.values():
            plan.process_group = self._process_group
            plan.average_grads = average
            plan.peer_comm = self._peer_comm if plan.device == getattr(self._peer_comm, "buf", torch.empty(0)).device else None
        return self

    def check_device_errors(self, synchronize: bool = True) -> None:
        """Raise if a kernel of this camera gave up waiting for other CTAs / ranks (a peer all-reduce whose peers never
        arrived, an image-max exchange or grid barrier that timed out).  Such a step's outputs are invalid (dL/dh is NaN
        after an all-reduce time-out).  Called automatically at the start of every PSF synthesis; call it yourself
        after the last step of a run."""
        from . import _lib
        for dev in self._plans:
            if synchronize:
                torch.cuda.synchronize(dev)
            _lib.raise_on_device_error(dev.index if dev.index is not None else torch.cuda.current_device())

    # ------------------------------------------------------------------ reference API
    def get_Heith_Map(self):
        zernike_coeffs_concat = torch.cat((self.Zer_no_train, self.Zer_train), 0)
        volume = self.zernike_volume
        if volume.device != zernike_coeffs_concat.device:
            volume = self.zernike_volume = volume.to(zernike_coeffs_concat.device)
        if zernike_coeffs_concat.is_cuda and volume.dtype == torch.float32 and volume.is_contiguous() and (self.N * self.N) % 4 == 0:
            # one pass over the basis volume (b200cam_zernike_fwd / _bwd) instead of materialising coef * volume
            return F.zernike_project(zernike_coeffs_concat, volume, self._plan(volume.device)).unsqueeze(0)
        height_map = torch.sum(zernike_coeffs_concat * volume, dim=0)     # CPU tensors: the reference's expression
        return height_map.unsqueeze(0)

    def load_ckpt(self):
        ckpt = torch.load('./Camera/Cam_focus.pth', map_location=self.device)
        self.load_state_dict(ckpt['camera'])

    def get_phase_shift(self):
        h = self.get_Heith_Map()
        return self.k.to(h.device) * self.flmb.to(h.device) * h

    def get_psf(self, _stream=None):
        h = self.get_Heith_Map()
        plan = self._plan(h.device)
        psf, loss_rad, centering = F.psf_synth(h, plan, _stream)
        self.psfs = psf
        self.loss_rad = loss_rad
        self._pending_centering = centering
        return self.psfs

    def forward(self, img, noise=None):
        """`noise`: optional standard-normal tensor shaped like `img` for the opt-in sensor noise (drawn here with
        torch.randn when `sensor_noise_sigma > 0` and none is given, or in the kernels with `sensor_noise_rng = "philox"`).  The
        sensor image is returned in `sensor_dtype`."""
        out_dtype = F.check_sensor_dtype(self.sensor_dtype)
        rng = F.check_noise_rng(self.sensor_noise_rng)
        # uint8 images (what a decoder produces; the reference's loader turns them into fp32 in [0,1] with ToTensor on the
        # host, Face-DeId/core/data_loader.py:118-124) may be passed as they are: the sensor kernels read the bytes and convert
        # them in registers as x * fp32(1/255), bit for bit torch's x.float() / 255.0 on the GPU - no fp32 copy of the batch is
        # made or kept for the backward, and the host->device copy is a quarter of the fp32 one.  Only the opt-in plane kernels
        # (B200CAM_PLANE=1 at N = 256) read fp32 images alone: there the batch is converted with that torch expression.
        if (torch.is_tensor(img) and img.dtype == torch.uint8 and img.is_cuda and self.N == 256 and F.PLANE_KERNELS
                and out_dtype == torch.float32):
            img = img.to(torch.float32).div_(255.0)
        # The PSF synthesis is a chain of small latency-bound kernels and the row transforms of the images do not
        # depend on it: put the chain on a high-priority side stream, run the row pass on the current stream meanwhile
        # and join before the spectral product.
        h_dev = self.Zer_train.device
        overlap = (self.overlap_psf and torch.is_tensor(img) and img.is_cuda and img.dim() == 4 and img.shape[0] > 0
                   and h_dev.type == "cuda")
        epi = (F.read_out(img, self.sensor_noise_sigma, self.sensor_quant_bits, noise, rng, F.shard_first4(img, self._process_group))
               if torch.is_tensor(img) else None)
        self.sensor_noise_seed = F.noise_seed(epi)
        if not overlap:
            psf = self.get_psf()
            self.centering_loss = self._pending_centering
            return F.sensor_conv(img, psf, self._plan(psf.device), None, epi, out_dtype)
        plan = self._plan(img.device)
        side = plan.side_stream()
        psf = self.get_psf(_stream=side)                       # enqueued on `side`, not joined yet
        # (the bf16 and Philox read-outs run the default pipeline only: not the plane layout that sensor_rows writes with
        # B200CAM_PLANE=1; a uint8 batch reaches this point at N = 256 with B200CAM_PLANE=1 only with bf16, see above)
        default_only = out_dtype == torch.bfloat16 or self.sensor_noise_seed is not None
        split = psf.device == img.device and not (default_only and self.N == 256 and F.PLANE_KERNELS)
        rows = F.sensor_rows(img, plan) if split else None
        cur = torch.cuda.current_stream(psf.device)
        if rows is not None and plan.otf_event is not None:
            # the spectral product only needs the OTF: the PSF itself and the two regularisers are written on a
            # normal-priority stream while the sensor kernels run, and joined at the end
            ev, plan.otf_event = plan.otf_event, None
            # psf / regularisers: beside the OTF kernels (both only read |U|^2), i.e. before the spectral product fills
            # every SM - a finalise that straggles into the one-pass inverse-row kernel keeps part of that kernel's
            # persistent grid from becoming resident and its per-image max exchange then waits (measured 50 vs 35 us)
            aux = plan.aux_stream()
            fev, plan.field_event = plan.field_event, None
            aux.wait_event(fev if fev is not None else ev)
            plan.finish_psf(aux)
            cur.wait_event(ev)
            self.centering_loss = self._pending_centering
            y = F.sensor_conv(img, psf, self._plan(psf.device), rows, epi, out_dtype)
            cur.wait_stream(aux)
            cur.wait_stream(side)
            return y
        plan.finish_psf(side)
        cur.wait_stream(side)
        self.centering_loss = self._pending_centering
        return F.sensor_conv(img, psf, self._plan(psf.device), rows, epi, out_dtype)

    # ------------------------------------------------------------------ CUDA-graph helper (no reference counterpart)
    def graphed(self, sample_img: torch.Tensor, num_warmup_iters: int = 3):
        """CUDA-graphed ``camera(img) -> (sensor, loss_rad, centering_loss)`` for a FIXED input shape.

        An eager forward + backward of this module costs ~400 us of host time (16 kernel launches through ctypes, autograd,
        stream bookkeeping) for ~175 us of device time at B = 64: training loops that run the camera in front of a
        downstream net should not pay that every step.  The returned callable replays one captured graph for the forward
        and one for the backward (``torch.cuda.make_graphed_callables``: static input / output / gradient buffers, inputs are
        copied in, autograd sees an ordinary differentiable op), so the downstream net and the optimiser stay eager:

            step = camera.graphed(images[:B])              # once; images: (B,3,N,N) fp32 or uint8 on the GPU
            sensor, loss_rad, centering = step(images_b)   # every iteration
            (task_loss(net(sensor)) + a * loss_rad + b * centering).backward()

        The two regularisers are RETURNED (the module attributes ``loss_rad`` / ``centering_loss`` set during capture are not
        connected to the replayed graph).  Capture before the module's first eager backward (PyTorch's rule for
        ``make_graphed_callables``: gradient-accumulation nodes created on the default stream cannot join a capture).  Re-capture after changing N, the batch size, ``data_parallel``, the epilogue
        switches or ``sensor_dtype`` (the graph keeps the dtype it was captured with).  Parameter updates in place (optimiser steps, ``load_state_dict``) are picked up by the replays."""
        if not (torch.is_tensor(sample_img) and sample_img.is_cuda):
            raise RuntimeError("b200cam runs on CUDA (sm_100a) only; capture needs a sample batch on the GPU")

        class _WithLosses(nn.Module):
            def __init__(self, cam):
                super().__init__()
                self.cam = cam

            def forward(self, img):
                y = self.cam(img)
                return y, self.cam.loss_rad, self.cam.centering_loss

        wrapped = _WithLosses(self)
        sample = sample_img.detach().clone()
        return torch.cuda.make_graphed_callables(wrapped, (sample,), num_warmup_iters=num_warmup_iters)
