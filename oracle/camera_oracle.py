"""TEST INFRASTRUCTURE ONLY - CPU restatement of the Face-DeId optical encoder.

This file is the *oracle* for the CUDA hot path: a plain ``torch`` (CPU)
restatement of the algorithm of the reference ``Camera`` module
(``Face-DeId/Camera/Optics.py``, helpers in ``Face-DeId/Camera/Utils.py``),
written from the maths, with every function citing the reference lines it
follows.  It is a floating-point path, so the oracle is torch fp32 (same
operation order as the reference where fp32 rounding of large phases matters)
and can also be evaluated in fp64 to attribute error.

Who may use it: ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs - as the checker or the timed CPU
baseline, never as the product.  The product package
(``privacy-preserving-vision_b200``) must not import anything from ``oracle/``.

Parity pinning: the reference ships no tests, golden vectors or usable
known-answer artefacts for this path (SURVEY.md section 4 / 8c).  The oracle is
pinned instead against outputs of the reference module itself, run in the build
container through ``oracle/ref_shim.py``: ``oracle/make_golden.py`` writes those
outputs to ``tests/golden/facedeid_*.npz`` and ``tests/test_oracle_vs_golden.py``
checks this file against them (and, when ``B200CAM_REFERENCE_ROOT`` names a
reference checkout, against the live reference module).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch

# ----------------------------------------------------------------------------
# constants (Optics.py:10-55)
# ----------------------------------------------------------------------------


def sellmeier_delta_n(lam_um: torch.Tensor) -> torch.Tensor:
    """abs(n_lens - n_air) for wavelength in micrometres (Utils.py:33-40, ``deta``)."""
    l2 = lam_um ** 2
    n_lens = torch.sqrt(1 + (0.6961663 * l2 / (l2 - 0.0684043 ** 2)
                             + 0.4079426 * l2 / (l2 - 0.1162414 ** 2)
                             + 0.8974794 * l2 / (l2 - 9.896161 ** 2)))
    inv2 = lam_um ** -2
    n_air = 1 + 0.05792105 / (238.0185 - inv2) + 0.00167917 / (57.362 - inv2)
    return torch.abs(n_lens - n_air)


@dataclass
class OracleConstants:
    N: int
    dtype: torch.dtype
    zi: float
    L_len: float
    L_sen: float
    px: float
    du: float
    dx2: float
    pi: torch.Tensor       # (1,)
    lamb: torch.Tensor     # (3,1,1)
    flmb: torch.Tensor     # (3,1,1)
    k: torch.Tensor        # (3,1,1)
    z: torch.Tensor        # (1,) object distances
    XY: torch.Tensor       # (N,N) pupil r^2
    rad: torch.Tensor      # (N,N) bool aperture
    FF: torch.Tensor       # (N,N) fft-ordered |f|^2
    XY2: torch.Tensor      # (N,N) sensor r^2
    rho: torch.Tensor      # (N,N) 0/1 outside-32px mask

    @property
    def kappa(self) -> torch.Tensor:
        """phase per metre of lens height, k*flmb (Optics.py:89-90)."""
        return self.k * self.flmb


def build_constants(N: int = 256, dtype: torch.dtype = torch.float32) -> OracleConstants:
    """Geometry and dispersion constants, Optics.py:13-55 (same torch calls, so same rounding)."""
    zi, z0 = 50e-3, 5.0
    f = 1 / (1 / zi + 1 / z0)
    R = f * sellmeier_delta_n(torch.tensor(550e-9 * 1e6, dtype=dtype))
    radii = 2.0e-3
    pi = torch.tensor([math.pi], dtype=dtype)
    L_len = 2 * radii * 2
    px = 3.713103e-6
    L_sen = px * N
    lamb = (torch.tensor([640, 550, 440]) * 1.e-9).to(dtype) if dtype == torch.float32 else \
        torch.tensor([640, 550, 440], dtype=dtype) * 1.e-9
    lamb = lamb.unsqueeze(-1).unsqueeze(-1)
    flmb = R / sellmeier_delta_n(lamb * 1e6)
    k = 2 * pi / lamb
    z = torch.tensor([0.75], dtype=dtype)

    du = L_len / N
    u = torch.arange(-1 * L_len / 2, L_len / 2, du, dtype=dtype)
    X, Y = torch.meshgrid(u, u, indexing="ij")
    XY = X * X + Y * Y
    rad = torch.sqrt(X ** 2 + Y ** 2) <= radii

    fx = torch.arange(-1 / (2 * du), 1 / (2 * du), 1 / L_len, dtype=dtype)
    fx = torch.roll(fx, -(N // 2), 0)
    FX, FY = torch.meshgrid(fx, fx, indexing="ij")
    FF = FX * FX + FY * FY

    dx2 = L_sen / N
    x2 = torch.arange(-1 * L_sen / 2, L_sen / 2, dx2, dtype=dtype)
    X2, Y2 = torch.meshgrid(x2, x2, indexing="ij")
    XY2 = X2 * X2 + Y2 * Y2
    rho = (torch.sqrt(X2 ** 2 + Y2 ** 2) > px * 32) * 1.0
    assert u.numel() == N and fx.numel() == N and x2.numel() == N
    return OracleConstants(N=N, dtype=dtype, zi=zi, L_len=L_len, L_sen=L_sen, px=px, du=du, dx2=dx2,
                           pi=pi, lamb=lamb, flmb=flmb, k=k, z=z, XY=XY, rad=rad, FF=FF, XY2=XY2,
                           rho=rho.to(dtype))


# ----------------------------------------------------------------------------
# forward restatement
# ----------------------------------------------------------------------------


def cexp(phase: torch.Tensor) -> torch.Tensor:
    """Euler exponent (Utils.py:55-57)."""
    return torch.complex(torch.cos(phase), torch.sin(phase))


def _shift(x: torch.Tensor, s: int) -> torch.Tensor:
    """roll both image dims by s (Utils.py:15-30; for even N fftshift == ifftshift == roll N/2)."""
    return torch.roll(x, (s, s), (-2, -1))


def phase_shift(h: torch.Tensor, C: OracleConstants) -> torch.Tensor:
    """(1,N,N) height [m] -> (3,N,N) phase [rad] (Optics.py:89-90)."""
    return C.k * C.flmb * h


def pupil_field(h: torch.Tensor, C: OracleConstants) -> torch.Tensor:
    """Field just behind the lens, pre-scaled for the two-step propagation (Optics.py:95-100)."""
    dis = C.z[0]
    t = cexp(-(C.k / (2 * C.flmb)) * C.XY)
    focus = cexp((C.k / (2 * dis)) * C.XY)
    ph = torch.mul(C.rad, torch.mul(t, focus)) * cexp(phase_shift(h, C))
    pre = cexp((C.pi / (C.lamb * C.zi * C.L_len) * (C.L_len - C.L_sen)) * C.XY)
    return torch.mul(ph, pre)


def transfer_function(C: OracleConstants) -> torch.Tensor:
    """H (3,N,N) of Optics.py:103 - NB it multiplies the *3-D* spectrum, so its first index
    is the DFT index across the wavelength axis, not a wavelength (SURVEY trap T1)."""
    return cexp(-(C.pi * C.lamb * C.zi * C.L_len / C.L_sen) * C.FF)


def propagate(vu: torch.Tensor, C: OracleConstants) -> torch.Tensor:
    """Optics.py:101-107: shift, fftn over ALL three dims, xH, ifftn over all dims, shift, post-phase."""
    N = C.N
    spec = torch.fft.fftn(_shift(vu, -(N // 2)))
    spec = torch.mul(spec, transfer_function(C))
    out = _shift(torch.fft.ifftn(spec), N // 2)
    post = cexp(-(C.pi / (C.lamb * C.zi * C.L_sen) * (C.L_len - C.L_sen)) * C.XY2)
    return (C.L_sen / C.L_len) * torch.multiply(out, post)


def psf_from_height(h: torch.Tensor, C: OracleConstants):
    """-> psfs (1,3,N,N), loss_rad (Optics.py:92-120)."""
    vu = propagate(pupil_field(h, C), C)
    psf = torch.square(torch.abs(vu * ((C.du * C.du) / (C.dx2 * C.dx2))))
    psf = psf / torch.sum(psf)
    loss_rad = torch.norm(C.rho * psf, "fro")
    return psf.unsqueeze(0), loss_rad


def centering_loss(psf: torch.Tensor, N: int) -> torch.Tensor:
    """Optics.py:124-125."""
    a = torch.mean(torch.square(psf - torch.roll(psf, shifts=N // 2, dims=-2)))
    return a + torch.mean(torch.square(psf - torch.roll(psf, shifts=N // 2, dims=-1)))


def circular_conv(img: torch.Tensor, kernel: torch.Tensor) -> torch.Tensor:
    """Utils.py:7-12 (``conv2D``): circular convolution through real FFTs, no padding."""
    return torch.fft.irfftn(torch.fft.rfftn(img, dim=(-2, -1)) * torch.fft.rfftn(kernel, dim=(-2, -1)),
                            dim=(-2, -1))


def sensor_from_psf(img: torch.Tensor, psf: torch.Tensor, N: int):
    """Optics.py:126-128: origin-centre the PSF, convolve, divide by the per-image max."""
    c = N // 2
    conv = circular_conv(img, _shift(psf, -c))
    m = conv.amax((1, 2, 3))
    return conv / m[:, None, None, None], conv, m


def camera_forward(img: torch.Tensor, h: torch.Tensor, C: OracleConstants) -> dict:
    """Whole forward (Optics.py:122-129). ``h`` is the (1,N,N) height map (Optics.py:79-83 output)."""
    psf, loss_rad = psf_from_height(h, C)
    closs = centering_loss(psf, C.N)
    y, conv, m = sensor_from_psf(img, psf, C.N)
    return {"sensor": y, "psf": psf, "loss_rad": loss_rad, "centering_loss": closs, "conv": conv, "max": m}


def height_map(zer_no_train: torch.Tensor, zer_train: torch.Tensor, zernike_volume: torch.Tensor) -> torch.Tensor:
    """Optics.py:79-83."""
    coefs = torch.cat((zer_no_train, zer_train), 0)
    return torch.sum(coefs * zernike_volume, dim=0).unsqueeze(0)


# ----------------------------------------------------------------------------
# closed-form backward (hand-derived adjoints; the CUDA kernels implement these,
# the tests check them against autograd of the forward above)
# ----------------------------------------------------------------------------


def sensor_backward(g: torch.Tensor, img: torch.Tensor, psf: torch.Tensor, N: int, want_img_grad: bool = False,
                    tie_mask: torch.Tensor | None = None):
    """Adjoint of ``sensor_from_psf`` w.r.t. psf (and optionally img).

    y = conv/m, m = amax(conv) per image.  dL/dconv = (g - s*tie/n)/m with s = sum(g*y) and
    ``tie`` the mask of positions equal to the max (torch's amax backward splits evenly).
    dL/dpsf0 = sum_b irfft2(conj(rfft2 x_b) * rfft2 dL/dconv_b); dL/dpsf = roll(dL/dpsf0, +N/2).
    """
    c = N // 2
    psf0 = _shift(psf, -c)
    K = torch.fft.rfftn(psf0, dim=(-2, -1))
    X = torch.fft.rfftn(img, dim=(-2, -1))
    conv = torch.fft.irfftn(X * K, dim=(-2, -1))
    m = conv.amax((1, 2, 3), keepdim=True)
    y = conv / m
    s = (g * y).sum((1, 2, 3), keepdim=True)
    tie = (conv == m).to(g.dtype) if tie_mask is None else tie_mask.to(g.dtype)   # override: test hook
    n = tie.sum((1, 2, 3), keepdim=True)
    gconv = (g - s * tie / n) / m
    G = torch.fft.rfftn(gconv, dim=(-2, -1))
    gpsf0 = torch.fft.irfftn((X.conj() * G).sum(0, keepdim=True), s=(N, N), dim=(-2, -1))
    gpsf = _shift(gpsf0, c)
    gimg = torch.fft.irfftn(K.conj() * G, s=(N, N), dim=(-2, -1)) if want_img_grad else None
    return gpsf, gimg


def regulariser_grads(psf: torch.Tensor, C: OracleConstants, g_rad: float, g_cen: float) -> torch.Tensor:
    """d(g_rad*loss_rad + g_cen*centering_loss)/dpsf, closed form."""
    N = C.N
    rp = C.rho * psf
    lr = torch.norm(rp, "fro")
    out = g_rad * C.rho * rp / lr
    n = psf.numel()
    out = out + g_cen * (4.0 / n) * (psf - torch.roll(psf, N // 2, -2))
    out = out + g_cen * (4.0 / n) * (psf - torch.roll(psf, N // 2, -1))
    return out


def psf_backward(gpsf: torch.Tensor, h: torch.Tensor, C: OracleConstants) -> torch.Tensor:
    """Adjoint of ``psf_from_height`` (psf output only): (1,3,N,N) grad -> (1,N,N) dL/dh.

    Uses: psf = I/S, I = |U|^2 (constant scalars and the unit-modulus post phase cancel);
    U = shift(IFFT3(H * FFT3(shift(V)))) is linear in V with adjoint of the same shape with conj(H);
    V = A exp(i kappa h)  =>  dL/dphi = Im(Gv * conj(V)), dL/dh = sum_lambda kappa * dL/dphi.
    """
    N = C.N
    V = pupil_field(h, C)
    Us = torch.fft.ifftn(torch.fft.fftn(_shift(V, -(N // 2))) * transfer_function(C))
    I = (Us.real ** 2 + Us.imag ** 2)
    S = I.sum()
    psf_s = I / S                                   # psf in the un-shifted (FFT) frame
    gp = _shift(gpsf.reshape(3, N, N), -(N // 2))   # bring the gradient into the same frame
    gI = (gp - (gp * psf_s).sum()) / S
    GU = 2.0 * gI * Us
    GVs = torch.fft.ifftn(torch.fft.fftn(GU) * transfer_function(C).conj())
    GV = _shift(GVs, N // 2)
    gphi = (GV * V.conj()).imag
    return (C.kappa * gphi).sum(0, keepdim=True)
