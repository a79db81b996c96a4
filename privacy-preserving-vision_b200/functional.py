"""torch.autograd glue between the nn.Module boundary and the C ABI.

Two differentiable ops, both thin ctypes calls into ``libb200cam.so`` on the current CUDA stream:

* ``psf_synth(h, plan)        -> psf (1,3,N,N), loss_rad (), centering_loss ()``
  (``Face-DeId/Camera/Optics.py:89-120,124-125``)
* ``sensor_conv(img, psf, plan) -> sensor (B,3,N,N)``
  (``Optics.py:126-128`` + ``Face-DeId/Camera/Utils.py:7-12``)

PyTorch owns every buffer (outputs, saved tensors, scratch); the library only enqueues kernels.
"""
from __future__ import annotations

import ctypes
import os

import torch

from . import _lib
from . import constants as K


class DevicePlan:
    """Per-(device, N) constant tables and scratch buffers for the kernels."""

    def __init__(self, N: int, device: torch.device, tables=None):
        if device.type != "cuda":
            raise RuntimeError("b200cam runs on CUDA (sm_100a) only; there is no CPU path "
                               f"(got device={device})")
        self.N = N
        self.device = device
        self.index = device.index if device.index is not None else torch.cuda.current_device()
        self.lib = _lib.load_library()
        if not self.lib.b200cam_supported(N):
            raise ValueError(f"b200cam supports N in (64,128,256,512,1024), got {N}")
        _lib.ensure_init(N, self.index)
        if tables is not False:           # tables=False: convolution-only plan (Image_Caption camera), no PSF chain
            t = tables if tables is not None else K.build(N)
            self.A = torch.view_as_real(t.table_A).contiguous().to(device)
            self.Ht = torch.view_as_real(t.table_Ht).contiguous().to(device)
            self.rho = t.rho.to(torch.float32).contiguous().to(device)
            self.kappa = (ctypes.c_float * 3)(*t.kappa)
            self.kappa_list = list(t.kappa)
            # zero-filled ONCE: the grid-barrier words of the cooperative PSF kernels live in it (the library leaves them zero)
            self._psf_ws = torch.zeros(self.lib.b200cam_psf_workspace_bytes(N), dtype=torch.uint8, device=device)
        self._sensor_ws: dict[int, torch.Tensor] = {}
        self._zernike_ws: dict[tuple[int, int], torch.Tensor] = {}
        self.otf_floats = self.lib.b200cam_otf_bytes(N) // 4
        self.process_group = None      # set by Camera.data_parallel(): all-reduce dL/dh over ranks
        self.average_grads = True
        self.peer_comm = None          # parallel.PeerComm: fused NVLink all-reduce instead of the NCCL call
        self.otf_cache = None          # (psf tensor, its OTF) left by the last asynchronous psf_synth
        self.otf_event = None          # recorded on the side stream once that OTF is complete
        self.field_event = None        # recorded on the side stream once |U|^2 is complete (what finish_psf needs)
        self._side_stream = None       # runs the PSF-independent half of the sensor forward beside the PSF chain
        self._aux_stream = None
        self.pending_finish = None     # (psf, stats) still to be written by finish_psf()

    def side_stream(self) -> torch.cuda.Stream:
        """High-priority stream for the PSF chain: its small kernels must be dispatched ahead of the thousands of
        CTAs of the image row pass that runs beside it on the caller's stream."""
        if self._side_stream is None:
            self._side_stream = torch.cuda.Stream(device=self.device, priority=-1)
        return self._side_stream

    def aux_stream(self) -> torch.cuda.Stream:
        """Normal-priority stream for work that only has to be finished by the end of forward()."""
        if self._aux_stream is None:
            self._aux_stream = torch.cuda.Stream(device=self.device)
        return self._aux_stream

    def finish_psf(self, stream: torch.cuda.Stream) -> None:
        """Second half of an asynchronous psf_synth (b200cam_psf_finish) on `stream`, ordered after the OTF."""
        if self.pending_finish is None:
            return
        psf, stats = self.pending_finish
        self.pending_finish = None
        ws = self._psf_ws
        with torch.cuda.device(self.index):
            _lib.check(self.lib.b200cam_psf_finish(
                _lib.ptr(self.rho), _lib.ptr(psf), _lib.ptr(stats), _lib.ptr(ws), ws.numel(), self.N,
                ctypes.c_void_p(stream.cuda_stream)))

    def psf_workspace(self) -> torch.Tensor:
        return self._psf_ws

    def zernike_workspace(self, T: int, NN: int) -> torch.Tensor:
        """Zero-filled once (arrival counters live in it); the kernel leaves it reusable."""
        key = (T, NN)
        ws = self._zernike_ws.get(key)
        if ws is None:
            ws = torch.zeros(self.lib.b200cam_zernike_workspace_bytes(T, NN), dtype=torch.uint8, device=self.device)
            self._zernike_ws = {key: ws}
        return ws

    def zernike_support(self, Z: torch.Tensor):
        """int32 list of the float4 positions at which some basis plane is non-zero (the Zernike basis vanishes outside the
        unit disc), or None when (almost) every position is.  Computed once per volume (keyed on storage and version)."""
        key = (Z.data_ptr(), Z._version, tuple(Z.shape))
        cache = self.__dict__.setdefault("_zsupport", {})
        if key not in cache:
            if len(cache) >= 4:
                cache.clear()
            with torch.no_grad():
                nz = (Z.reshape(Z.shape[0], -1, 4) != 0).any(dim=2).any(dim=0)
                idx = torch.nonzero(nz).reshape(-1).to(torch.int32)
            cache[key] = idx.contiguous() if 0 < idx.numel() < 0.95 * nz.numel() else None
        return cache[key]

    def sensor_workspace(self, B: int) -> torch.Tensor:
        ws = self._sensor_ws.get(B)
        if ws is None:
            nbytes = self.lib.b200cam_sensor_workspace_bytes(self.N, B, 1)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            self._sensor_ws = {B: ws}          # keep one: batch size rarely changes
        return ws


# B200CAM_NVTX=1: NVTX ranges around every autograd entry point of the camera (SURVEY 5: tracing) - they show up as named
# spans in nsys / ncu timelines; off by default (a push / pop pair costs ~1 us of host time each)
_NVTX = os.environ.get("B200CAM_NVTX", "0") == "1"


def nvtx(name):
    """Decorator: wrap a static forward / backward in an NVTX range when B200CAM_NVTX=1."""
    def deco(fn):
        if not _NVTX:
            return fn

        def wrapped(*args, **kwargs):
            torch.cuda.nvtx.range_push(name)
            try:
                return fn(*args, **kwargs)
            finally:
                torch.cuda.nvtx.range_pop()
        return wrapped
    return deco


# 1: the caller's image row pass is ordered behind the first PSF kernel (see b200cam_psf_field); B200CAM_HOLD_ROWS=0 lets
# both start together (A/B switch)
_HOLD_ROWS = 0 if os.environ.get("B200CAM_HOLD_ROWS", "1") == "0" else 1
# B200CAM_PLANE=1 (opt-in N = 256 plane kernels, read once per process by the library): b200cam_sensor_rows then writes the
# plane layout, which the bf16 sensor path and the uint8 image path (default two-pass pipeline only) cannot read
PLANE_KERNELS = os.environ.get("B200CAM_PLANE", "0")[:1] == "1"


def _stream() -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _as_f32(t: torch.Tensor, device: torch.device) -> torch.Tensor:
    if t.device != device:
        raise RuntimeError(f"b200cam: tensor on {t.device}, camera tables on {device}")
    if t.dtype != torch.float32:
        raise TypeError(f"b200cam computes in fp32, got {t.dtype}")
    return t.contiguous()


def _as_img(t: torch.Tensor, device: torch.device) -> torch.Tensor:
    """An image batch for the sensor kernels: fp32, or uint8 as it is (converted in the kernels as x * fp32(1/255), bit for
    bit torch's ``x.float() / 255.0`` on the GPU)."""
    if t.dtype == torch.uint8:
        if t.device != device:
            raise RuntimeError(f"b200cam: tensor on {t.device}, camera tables on {device}")
        return t.contiguous()
    return _as_f32(t, device)


class PsfSynth(torch.autograd.Function):
    @staticmethod
    @nvtx("b200cam.PsfSynth.forward")
    def forward(ctx, h: torch.Tensor, plan: DevicePlan, stream: torch.cuda.Stream | None = None):
        """`stream`: enqueue the kernels there (after everything already on the current stream) and return WITHOUT
        joining - the caller must `current_stream().wait_stream(stream)` before using the outputs."""
        N = plan.N
        _lib.raise_on_device_error(plan.index)          # a wait that timed out in an earlier step is reported here
        hc = _as_f32(h.detach(), plan.device).reshape(N, N)
        psf = torch.empty(1, 3, N, N, dtype=torch.float32, device=plan.device)
        field = torch.empty(3, N, N, 2, dtype=torch.float32, device=plan.device)
        stats = torch.empty(4, dtype=torch.float32, device=plan.device)
        ws = plan.psf_workspace()
        if stream is not None:
            stream.wait_stream(torch.cuda.current_stream(plan.device))
        launch = ctypes.c_void_p(stream.cuda_stream) if stream is not None else _stream()
        with torch.cuda.device(plan.index):
            if stream is None:
                _lib.check(plan.lib.b200cam_psf_fwd(
                    _lib.ptr(hc), _lib.ptr(plan.A), _lib.ptr(plan.Ht), _lib.ptr(plan.rho), plan.kappa,
                    _lib.ptr(psf), _lib.ptr(field), _lib.ptr(stats), _lib.ptr(ws), ws.numel(), N, launch))
            else:
                # field -> OTF -> (event) -> psf + regularisers: the OTF only needs |U|^2 and its sum, so the sensor
                # pipeline that waits for `plan.otf_event` does not wait for the PSF to be written out
                _lib.check(plan.lib.b200cam_psf_field(
                    _lib.ptr(hc), _lib.ptr(plan.A), _lib.ptr(plan.Ht), plan.kappa, _lib.ptr(field),
                    _lib.ptr(ws), ws.numel(), N, launch, _stream(), _HOLD_ROWS))
                plan.field_event = torch.cuda.Event()          # |U|^2 and its partial sums are in the workspace
                plan.field_event.record(stream)
                otf = torch.empty(plan.otf_floats, dtype=torch.float32, device=plan.device)
                _lib.check(plan.lib.b200cam_psf_otf_early(_lib.ptr(otf), _lib.ptr(ws), ws.numel(), N, launch))
                plan.otf_event = torch.cuda.Event()
                plan.otf_event.record(stream)
                plan.otf_cache = (psf.data_ptr(), otf)
                # psf and the regularisers are written by `plan.finish_psf(stream)`, which the caller enqueues where it
                # does not delay the sensor pipeline (Camera.forward: low-priority stream, after the spectral product)
                plan.pending_finish = (psf, stats)
        ctx.plan = plan
        ctx.h_shape = h.shape
        ctx.save_for_backward(hc, psf, field, stats)
        # the two regularisers are returned as separate 0-dim outputs (views of `stats`): their upstream gradients then
        # arrive as two scalars instead of going through select-backward (zeros + index_put + add per loss)
        return psf, stats[1], stats[2]

    @staticmethod
    @nvtx("b200cam.PsfSynth.backward")
    def backward(ctx, g_psf, g_rad, g_cen):
        plan: DevicePlan = ctx.plan
        N = plan.N
        hc, psf, field, stats = ctx.saved_tensors
        gp = _as_f32(g_psf, plan.device).reshape(3, N, N) if g_psf is not None else None
        # the two regulariser gradients are passed as two device scalars (no stack / zeros kernels in between)
        gr = _as_f32(g_rad, plan.device).reshape(1) if g_rad is not None else None
        gc = _as_f32(g_cen, plan.device).reshape(1) if g_cen is not None else None
        grad_h = torch.empty(N, N, dtype=torch.float32, device=plan.device)
        ws = plan.psf_workspace()
        comm = plan.peer_comm
        if comm is not None:
            # all-reduce fused into the last kernel: peer-memory pushes over NVLink, no NCCL call
            with torch.cuda.device(plan.index):
                _lib.check(plan.lib.b200cam_psf_bwd_allreduce(
                    _lib.ptr(gp), _lib.ptr(gr), _lib.ptr(gc), _lib.ptr(hc), _lib.ptr(plan.A), _lib.ptr(plan.Ht),
                    _lib.ptr(plan.rho), plan.kappa, _lib.ptr(psf), _lib.ptr(field), _lib.ptr(stats), _lib.ptr(grad_h),
                    _lib.ptr(ws), ws.numel(), N, _stream(), comm.ptr_array, comm.rank, comm.world,
                    1.0 / comm.world if plan.average_grads else 1.0))
            return grad_h.reshape(ctx.h_shape), None, None
        with torch.cuda.device(plan.index):
            _lib.check(plan.lib.b200cam_psf_bwd(
                _lib.ptr(gp), _lib.ptr(gr), _lib.ptr(gc), _lib.ptr(hc), _lib.ptr(plan.A), _lib.ptr(plan.Ht),
                _lib.ptr(plan.rho), plan.kappa, _lib.ptr(psf), _lib.ptr(field), _lib.ptr(stats), _lib.ptr(grad_h),
                _lib.ptr(ws), ws.numel(), N, _stream()))
        if plan.process_group is not None:
            from .parallel import allreduce_height_grad
            allreduce_height_grad(grad_h, plan.process_group, plan.average_grads)
        return grad_h.reshape(ctx.h_shape), None, None


class ZernikeProject(torch.autograd.Function):
    """h = sum_j coef_j * Z_j (``get_Heith_Map``, ``Face-DeId/Camera/Optics.py:79-83``; ``Image_Caption/Camera/Lens.py:176``)
    and its adjoint, one pass over the basis volume each way (SURVEY 8 f1)."""

    @staticmethod
    @nvtx("b200cam.ZernikeProject.forward")
    def forward(ctx, coef: torch.Tensor, volume: torch.Tensor, plan: DevicePlan):
        T = volume.shape[0]
        NN = volume[0].numel()
        c = _as_f32(coef.detach(), plan.device).reshape(T)
        Z = _as_f32(volume.detach(), plan.device)
        h = torch.empty(volume.shape[1:], dtype=torch.float32, device=plan.device)
        ws = plan.zernike_workspace(T, NN)
        active = plan.zernike_support(Z)
        with torch.cuda.device(plan.index):
            _lib.check(plan.lib.b200cam_zernike_fwd_ex(_lib.ptr(c), _lib.ptr(Z), _lib.ptr(h), _lib.ptr(ws), ws.numel(), T, NN, _stream(),
                                                       _lib.ptr(active), active.numel() if active is not None else 0))
        ctx.plan = plan
        ctx.coef_shape = coef.shape
        ctx.active = active
        ctx.save_for_backward(Z)
        return h

    @staticmethod
    @nvtx("b200cam.ZernikeProject.backward")
    def backward(ctx, gh):
        plan: DevicePlan = ctx.plan
        (Z,) = ctx.saved_tensors
        T, NN = Z.shape[0], Z[0].numel()
        g = _as_f32(gh, plan.device)
        gc = torch.empty(T, dtype=torch.float32, device=plan.device)
        active = ctx.active
        with torch.cuda.device(plan.index):
            _lib.check(plan.lib.b200cam_zernike_bwd_ex(_lib.ptr(g), _lib.ptr(Z), _lib.ptr(gc), T, NN, _stream(),
                                                       _lib.ptr(active), active.numel() if active is not None else 0))
        return gc.reshape(ctx.coef_shape), None, None


def zernike_project(coef: torch.Tensor, volume: torch.Tensor, plan: DevicePlan) -> torch.Tensor:
    return ZernikeProject.apply(coef, volume, plan)


NOISE_RNGS = ("torch", "philox")


def check_noise_rng(rng) -> str:
    """The ``sensor_noise_rng`` module attribute of both cameras: "torch" (default) or "philox"."""
    if rng not in NOISE_RNGS:
        raise ValueError(f"sensor_noise_rng must be 'torch' or 'philox', got {rng!r}")
    return rng


def read_out(img: torch.Tensor, sigma: float, bits: int, noise: torch.Tensor | None = None, rng: str = "torch",
             first4: int = 0):
    """The opt-in sensor read-out of both cameras (``sensor_noise_sigma`` / ``sensor_quant_bits``): (noise, noise scale,
    quantisation bits) for the kernels' epilogue, or None when it is off (the reference).  A ``noise`` tensor given by the
    caller is used as it is.  Otherwise, with ``sigma > 0``:
    * ``rng="torch"``: the noise is drawn here with torch.randn shaped like ``img`` (torch's global generator: seed it to
      reproduce);
    * ``rng="philox"``: only a key is drawn here, with one torch.randint on the image's device (torch's generator, so seeded
      runs repeat and a CUDA graph draws a new key on every replay), and "noise" is the (2,) int64 seed block {key, first4}
      of include/b200cam.h (B200CAM_SENSOR_NOISE_PHILOX): the kernels draw the normals themselves.  ``first4`` is the counter
      of the batch's first four elements (non-zero for a shard of a larger batch, see :func:`shard_first4`)."""
    sigma, bits = float(sigma), int(bits)
    if noise is None and sigma > 0.0:
        if rng == "philox":
            key = torch.randint(2**63 - 1, (1,), dtype=torch.int64, device=img.device)
            noise = torch.cat((key, torch.full((1,), int(first4), dtype=torch.int64, device=img.device)))
        else:
            noise = torch.randn(img.shape, dtype=torch.float32, device=img.device)
    if noise is None and bits == 0:
        return None
    return (noise, sigma if noise is not None else 0.0, bits)


def noise_seed(epilogue) -> torch.Tensor | None:
    """The Philox seed block of a :func:`read_out` result, None when the noise is a tensor or there is none."""
    if epilogue is None or epilogue[0] is None or epilogue[0].dtype != torch.int64:
        return None
    return epilogue[0]


def shard_first4(img: torch.Tensor, process_group) -> int:
    """Philox counter of the first four elements of this rank's shard: rank * (elements per shard) / 4 for a batch sharded
    in equal parts over ``process_group`` (``data_parallel``), 0 without one.  Ranks seeded alike then draw the noise of the
    concatenated batch, as one GPU would."""
    if process_group is None:
        return 0
    import torch.distributed as dist
    if not dist.is_initialized():
        return 0
    return dist.get_rank(process_group) * (img.numel() // 4)


def philox_normal(seed_block: torch.Tensor, shape) -> torch.Tensor:
    """The standard normals the kernels draw for ``seed_block`` (the (2,) int64 {key, first4} of a Philox read-out), as an
    fp32 tensor of ``shape`` (numel % 4 == 0) on its device: b200cam_sensor_noise, bit for bit the values the normalise kernels
    add.  For tests, and for the geometries whose read-out runs as torch ops."""
    if seed_block.dtype != torch.int64 or seed_block.numel() != 2 or not seed_block.is_cuda:
        raise ValueError("seed_block must be a (2,) int64 CUDA tensor {key, first4}")
    seed = seed_block.contiguous()
    out = torch.empty(shape, dtype=torch.float32, device=seed.device)
    lib = _lib.load_library()
    with torch.cuda.device(seed.device):
        _lib.check(lib.b200cam_sensor_noise(_lib.ptr(seed), _lib.ptr(out), out.numel(), _stream()))
    return out


def epilogue_flags(epilogue, shape, device: torch.device):
    """(flags, noise, noise_scale, quant_bits) of the C ABI for a :func:`read_out` result: B200CAM_SENSOR_NOISE with an fp32
    tensor shaped like the images, B200CAM_SENSOR_NOISE_PHILOX with a seed block, B200CAM_SENSOR_QUANT with bits."""
    if epilogue is None:
        return 0, None, 0.0, 0
    noise, noise_scale, quant_bits = epilogue
    flags = 0
    if noise is not None and noise.dtype == torch.int64:
        if noise.numel() != 2 or noise.device != device:
            raise ValueError(f"a Philox seed block is a (2,) int64 tensor on {device}")
        noise = noise.contiguous()
        flags |= 4
    elif noise is not None:
        noise = _as_f32(noise.detach(), device)
        if tuple(noise.shape) != tuple(shape):
            raise ValueError(f"sensor noise must have the shape of the images {tuple(shape)}, got {tuple(noise.shape)}")
        flags |= 1
    if quant_bits:
        flags |= 2
    return flags, noise, noise_scale, quant_bits


SENSOR_DTYPES = (torch.float32, torch.bfloat16)


def check_sensor_dtype(dtype) -> torch.dtype:
    """The ``sensor_dtype`` module attribute of both cameras: torch.float32 (default) or torch.bfloat16."""
    if dtype not in SENSOR_DTYPES:
        raise ValueError(f"sensor_dtype must be torch.float32 or torch.bfloat16, got {dtype!r}")
    return dtype


def _check_img(img: torch.Tensor, N: int) -> None:
    if img.dim() != 4 or img.shape[1] != 3 or img.shape[2] != N or img.shape[3] != N:
        raise ValueError(f"expected img of shape (B,3,{N},{N}), got {tuple(img.shape)}")


class RowSpectra:
    """Result of :func:`sensor_rows`: the PSF-independent first half of the sensor forward (row transforms of the
    images, first half of ``rfftn`` in ``Face-DeId/Camera/Utils.py:8``)."""

    def __init__(self, x, spectrum, img_max, tie_count):
        self.x, self.spectrum, self.img_max, self.tie_count = x, spectrum, img_max, tie_count


def sensor_rows(img: torch.Tensor, plan: DevicePlan):
    """Enqueue the row transforms of ``img`` on the current stream (they need no PSF, so `Camera.forward` runs them
    while the PSF chain is busy on the plan's high-priority side stream).
    Returns None when the split entry points do not apply (empty batch, fused N=256 kernels).
    ``img`` is fp32 or uint8; a uint8 batch is read by the row kernel as it is (not with ``B200CAM_PLANE=1`` at N = 256:
    the finish call would then expect the plane layout, which only the fp32 row pass writes)."""
    N = plan.N
    _check_img(img, N)
    B = img.shape[0]
    if B == 0 or not plan.lib.b200cam_sensor_split_supported(N, B):
        return None
    x = _as_img(img.detach(), plan.device)
    spectrum = torch.empty(plan.lib.b200cam_spectrum_bytes(N, B) // 4, dtype=torch.float32, device=plan.device)
    img_max = torch.empty(B, dtype=torch.float32, device=plan.device)
    tie_count = torch.empty(B, dtype=torch.int32, device=plan.device)
    rows_fn = plan.lib.b200cam_sensor_rows_u8 if x.dtype == torch.uint8 else plan.lib.b200cam_sensor_rows
    with torch.cuda.device(plan.index):
        _lib.check(rows_fn(_lib.ptr(x), _lib.ptr(spectrum), _lib.ptr(img_max), _lib.ptr(tie_count), B, N, _stream()))
    return RowSpectra(x, spectrum, img_max, tie_count)


class SensorConv(torch.autograd.Function):
    @staticmethod
    @nvtx("b200cam.SensorConv.forward")
    def forward(ctx, img: torch.Tensor, psf: torch.Tensor, plan: DevicePlan, rows: RowSpectra | None = None, epilogue=None,
                out_dtype: torch.dtype = torch.float32):
        """`epilogue`: None (the reference's read-out: nothing) or (noise, noise_scale, quant_bits) of `read_out` - the opt-in
        sensor noise + quantisation of include/b200cam.h (B200CAM_SENSOR_NOISE, or _NOISE_PHILOX when `noise` is a seed block;
        _QUANT); straight-through in backward.
        `out_dtype` torch.bfloat16: the sensor image is written in bf16 (the fp32 result rounded to nearest-even, i.e.
        exactly ``fp32_result.to(torch.bfloat16)``) and the bf16 upstream gradient is read by the kernels as it is; the
        un-normalised fp32 image is a scratch buffer of the forward and is not kept.
        `img` fp32 or uint8: a uint8 batch is read by the kernels as it is (x * fp32(1/255) in registers, bit for bit the fp32
        call on ``img.float() / 255.0``) and the node saves it as it is; uint8 is not differentiable, so no dL/dimg."""
        N = plan.N
        flags, noise_t, noise_scale, quant_bits = epilogue_flags(epilogue, img.shape, plan.device)
        _check_img(img, N)
        x = rows.x if rows is not None else _as_img(img.detach(), plan.device)
        p = _as_f32(psf.detach(), plan.device).reshape(3, N, N)
        B = x.shape[0]
        bf16 = out_dtype == torch.bfloat16
        u8 = x.dtype == torch.uint8
        # bf16: `sensor` is the fp32 conv scratch (dropped after the forward), `out` the bf16 image handed downstream
        sensor = torch.empty(x.shape, dtype=torch.float32, device=x.device)
        out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device) if bf16 else sensor
        img_max = rows.img_max if rows is not None else torch.empty(B, dtype=torch.float32, device=plan.device)
        tie_count = rows.tie_count if rows is not None else torch.empty(B, dtype=torch.int32, device=plan.device)
        tie_pos = torch.empty(B, 8, dtype=torch.int32, device=plan.device)
        otf = torch.empty(plan.otf_floats, dtype=torch.float32, device=plan.device)
        # keep the image spectra for the backward (what autograd would save) only when a gradient is wanted
        spectrum = rows.spectrum if rows is not None else None
        if rows is None and B > 0 and any(ctx.needs_input_grad[:2]):
            spectrum = torch.empty(plan.lib.b200cam_spectrum_bytes(N, B) // 4, dtype=torch.float32, device=plan.device)
        if rows is not None:
            ws = plan.sensor_workspace(B)
            cached = plan.otf_cache
            otf_ready = int(cached is not None and cached[0] == p.data_ptr())
            if otf_ready:
                otf = cached[1]
            plan.otf_cache = None
            with torch.cuda.device(plan.index):
                if bf16:
                    _lib.check(plan.lib.b200cam_sensor_finish_bf16(
                        _lib.ptr(p), _lib.ptr(sensor), _lib.ptr(out), _lib.ptr(img_max), _lib.ptr(tie_count), _lib.ptr(tie_pos),
                        _lib.ptr(otf), _lib.ptr(spectrum), otf_ready, _lib.ptr(ws), ws.numel(), B, N, _stream(),
                        flags, _lib.ptr(noise_t), float(noise_scale), int(quant_bits)))
                else:
                    _lib.check(plan.lib.b200cam_sensor_finish_ex(
                        _lib.ptr(p), _lib.ptr(sensor), _lib.ptr(img_max), _lib.ptr(tie_count), _lib.ptr(tie_pos),
                        _lib.ptr(otf), _lib.ptr(spectrum), otf_ready, _lib.ptr(ws), ws.numel(), B, N, _stream(),
                        flags, _lib.ptr(noise_t), float(noise_scale), int(quant_bits)))
            if not any(ctx.needs_input_grad[:2]):
                spectrum = None
        elif B > 0:
            ws = plan.sensor_workspace(B)
            with torch.cuda.device(plan.index):
                if bf16:
                    fwd = plan.lib.b200cam_sensor_fwd_u8_bf16 if u8 else plan.lib.b200cam_sensor_fwd_bf16
                    _lib.check(fwd(
                        _lib.ptr(x), _lib.ptr(p), _lib.ptr(sensor), _lib.ptr(out), _lib.ptr(img_max), _lib.ptr(tie_count),
                        _lib.ptr(tie_pos), _lib.ptr(otf), _lib.ptr(spectrum), _lib.ptr(ws), ws.numel(), B, N, _stream(),
                        flags, _lib.ptr(noise_t), float(noise_scale), int(quant_bits)))
                else:
                    fwd = plan.lib.b200cam_sensor_fwd_u8 if u8 else plan.lib.b200cam_sensor_fwd_ex
                    _lib.check(fwd(
                        _lib.ptr(x), _lib.ptr(p), _lib.ptr(sensor), _lib.ptr(img_max), _lib.ptr(tie_count),
                        _lib.ptr(tie_pos), _lib.ptr(otf), _lib.ptr(spectrum), _lib.ptr(ws), ws.numel(), B, N, _stream(),
                        flags, _lib.ptr(noise_t), float(noise_scale), int(quant_bits)))
        elif bf16:
            out = sensor.to(torch.bfloat16)           # empty batch: nothing for the kernels to do
        ctx.plan = plan
        ctx.psf_shape = psf.shape
        ctx.spectrum = spectrum
        # the bf16 node keeps no image-sized fp32 sensor tensor (no backward kernel reads it); a uint8 batch is kept as uint8
        ctx.save_for_backward(x, p, None if bf16 else sensor, img_max, tie_count, tie_pos, otf)
        return out

    @staticmethod
    @nvtx("b200cam.SensorConv.backward")
    def backward(ctx, g):
        plan: DevicePlan = ctx.plan
        N = plan.N
        x, p, sensor, img_max, tie_count, tie_pos, otf = ctx.saved_tensors
        B = x.shape[0]
        want_img = ctx.needs_input_grad[0]
        # the kernels overwrite every element of grad_psf; only the empty batch needs explicit zeros
        grad_psf = (torch.empty if B > 0 else torch.zeros)(3, N, N, dtype=torch.float32, device=plan.device)
        grad_img = torch.empty_like(x) if want_img else None      # (never for uint8 images: not differentiable)
        u8 = x.dtype == torch.uint8
        if B > 0 and g.dtype == torch.bfloat16:
            if g.device != plan.device:
                raise RuntimeError(f"b200cam: tensor on {g.device}, camera tables on {plan.device}")
            gc = g.contiguous()
            ws = plan.sensor_workspace(B)
            bwd = plan.lib.b200cam_sensor_bwd_u8_bf16 if u8 else plan.lib.b200cam_sensor_bwd_bf16
            with torch.cuda.device(plan.index):
                _lib.check(bwd(
                    _lib.ptr(gc), _lib.ptr(x), _lib.ptr(img_max), _lib.ptr(tie_count), _lib.ptr(tie_pos), _lib.ptr(p),
                    _lib.ptr(otf), _lib.ptr(ctx.spectrum), _lib.ptr(grad_psf), _lib.ptr(grad_img),
                    _lib.ptr(ws), ws.numel(), B, N, _stream()))
        elif B > 0:
            gc = _as_f32(g, plan.device)
            ws = plan.sensor_workspace(B)
            bwd = plan.lib.b200cam_sensor_bwd_u8 if u8 else plan.lib.b200cam_sensor_bwd
            with torch.cuda.device(plan.index):
                _lib.check(bwd(
                    _lib.ptr(gc), _lib.ptr(x), _lib.ptr(sensor), _lib.ptr(img_max), _lib.ptr(tie_count),
                    _lib.ptr(tie_pos), _lib.ptr(p), _lib.ptr(otf), _lib.ptr(ctx.spectrum), _lib.ptr(grad_psf),
                    _lib.ptr(grad_img),
                    _lib.ptr(ws), ws.numel(), B, N, _stream()))
        return grad_img, grad_psf.reshape(ctx.psf_shape), None, None, None, None


def psf_synth(h: torch.Tensor, plan: DevicePlan, stream: torch.cuda.Stream | None = None):
    return PsfSynth.apply(h, plan, stream)


def sensor_conv(img: torch.Tensor, psf: torch.Tensor, plan: DevicePlan, rows: RowSpectra | None = None,
                epilogue=None, out_dtype: torch.dtype = torch.float32) -> torch.Tensor:
    return SensorConv.apply(img, psf, plan, rows, epilogue, out_dtype)
