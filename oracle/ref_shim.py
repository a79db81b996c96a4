"""TEST INFRASTRUCTURE ONLY - import the *unmodified* reference camera modules.

The reference sources are not part of this repository.  They are used only when
the environment variable ``B200CAM_REFERENCE_ROOT`` names a checkout of
carlosh93/privacy-preserving-vision; without it ``reference_available()`` is
False and the tests that need the live reference skip.  Nothing under
``-m gpu``, ``smoke()`` or ``bench.py`` may call into this file.  Its two users
are ``oracle/make_golden.py`` (writes ``tests/golden/*.npz``) and the CPU tests
that pin ``oracle/camera_oracle.py`` / ``oracle/lens_oracle.py`` to the reference.

The reference imports ``matplotlib`` and ``poppy`` at module import time
(``Face-DeId/Camera/Optics.py:4``, ``Face-DeId/Camera/Utils.py:2-3``,
``Image_Caption/Camera/Utils.py:9``); neither is installed here, so they are
stubbed in ``sys.modules``.  ``poppy.zernike.zernike_basis`` is replaced by the
restatement in ``privacy-preserving-vision_b200/zernike.py`` (parity unpinned
vs. real poppy, see that file).  ``numpy.math`` (removed in numpy 2) is
aliased for ``Image_Caption/Camera/Utils.py:213``.
"""
from __future__ import annotations

import importlib
import importlib.util
import math
import os
import sys
import types
from pathlib import Path

REFERENCE_ROOT = Path(os.environ["B200CAM_REFERENCE_ROOT"]) if os.environ.get("B200CAM_REFERENCE_ROOT") else None
_REPO = Path(__file__).resolve().parent.parent


def reference_available() -> bool:
    if REFERENCE_ROOT is None:
        return False
    try:
        return (REFERENCE_ROOT / "Face-DeId" / "Camera" / "Optics.py").is_file()
    except OSError:                      # e.g. a path this user may not read
        return False


def _load_zernike():
    spec = importlib.util.spec_from_file_location(
        "_b200cam_zernike_for_shim", _REPO / "privacy-preserving-vision_b200" / "zernike.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _install_stubs() -> None:
    if "matplotlib" not in sys.modules:
        try:
            importlib.import_module("matplotlib.pyplot")
        except Exception:
            mpl = types.ModuleType("matplotlib")
            plt = types.ModuleType("matplotlib.pyplot")
            mpl.pyplot = plt
            sys.modules["matplotlib"] = mpl
            sys.modules["matplotlib.pyplot"] = plt
    if "poppy" not in sys.modules:
        try:
            importlib.import_module("poppy")
        except Exception:
            zern = _load_zernike()
            poppy = types.ModuleType("poppy")
            pz = types.ModuleType("poppy.zernike")
            pz.zernike_basis = zern.zernike_basis
            poppy.zernike = pz
            sys.modules["poppy"] = poppy
            sys.modules["poppy.zernike"] = pz
    import numpy as np
    if not hasattr(np, "math"):
        np.math = math  # Image_Caption/Camera/Utils.py:213 uses np.math.gcd


def _import_package(alias: str, pkg_dir: Path):
    """Import ``pkg_dir`` (a directory without __init__.py) as namespace package ``alias``."""
    if alias in sys.modules:
        return sys.modules[alias]
    pkg = types.ModuleType(alias)
    pkg.__path__ = [str(pkg_dir)]
    sys.modules[alias] = pkg
    return pkg


def load_face_deid_camera():
    """Returns the reference ``Camera`` class (Face-DeId/Camera/Optics.py:9)."""
    if not reference_available():
        raise RuntimeError(f"reference sources not found (B200CAM_REFERENCE_ROOT={REFERENCE_ROOT})")
    _install_stubs()
    _import_package("_ref_facedeid_camera", REFERENCE_ROOT / "Face-DeId" / "Camera")
    return importlib.import_module("_ref_facedeid_camera.Optics").Camera


def load_face_deid_utils():
    if not reference_available():
        raise RuntimeError(f"reference sources not found (B200CAM_REFERENCE_ROOT={REFERENCE_ROOT})")
    _install_stubs()
    _import_package("_ref_facedeid_camera", REFERENCE_ROOT / "Face-DeId" / "Camera")
    return importlib.import_module("_ref_facedeid_camera.Utils")


def load_image_caption_lens():
    """Returns the reference module ``Image_Caption/Camera/Lens.py`` (class OpticsZernike :11)."""
    if not reference_available():
        raise RuntimeError(f"reference sources not found (B200CAM_REFERENCE_ROOT={REFERENCE_ROOT})")
    _install_stubs()
    _import_package("_ref_caption_camera", REFERENCE_ROOT / "Image_Caption" / "Camera")
    return importlib.import_module("_ref_caption_camera.Lens")
