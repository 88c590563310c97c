"""ORACLE (test infrastructure, not product): run the reference's *own* ``_extract_eig`` in this container.

The reference's sources are only needed where the fixtures are generated, so no test, smoke() or bench.py imports
this file; oracle/make_golden.py uses it to record the fixtures under tests/golden/, which the tests compare with.

The reference's module imports packages that are not installed here (fire, accelerate, skimage, pymatting); they
are replaced by inert stubs *before* ``import extract``:
  fire.Fire, accelerate.Accelerator, skimage.morphology.binary_{dilation,erosion}  -> never called on this path
  pymatting.util.util.row_sum    -> A.dot(ones)           (published behaviour; used at extract_utils.py:217)
  pymatting.util.kdtree.knn      -> exact KNN stand-in    (used at extract_utils.py:177)
  pymatting.laplacian.rw_laplacian._rw_laplacian -> restated stencil weights (used at extract_utils.py:194,202)
With no GPU, ``Tensor.cuda`` (extract.py:146) is made a no-op so the matmul runs on the CPU in float32.
"""
from __future__ import annotations

import importlib.machinery
import sys
import types
from pathlib import Path

import numpy as np
import torch

REFERENCE_DIR = Path("/root/reference/extract")


def available() -> bool:
    return (REFERENCE_DIR / "extract.py").is_file()


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__spec__ = importlib.machinery.ModuleSpec(name, loader=None)  # keeps importlib.util.find_spec(name) happy
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


_ref = None


def load_reference():
    """Import /root/reference/extract/extract.py under stubs and return the module."""
    global _ref
    if _ref is not None:
        return _ref
    if not available():
        raise RuntimeError("reference sources are not present (only available in the dev container)")
    from . import eigs_ref

    def _never(*a, **k):
        raise RuntimeError("stubbed dependency called")

    transient = []  # stubs only needed while the reference's top-level imports run (removed again afterwards so
    #                 that other libraries probing e.g. `accelerate` do not mistake them for the real packages)
    if "fire" not in sys.modules:
        _stub("fire", Fire=_never); transient.append("fire")
    if "accelerate" not in sys.modules:
        _stub("accelerate", Accelerator=_never); transient.append("accelerate")
    try:
        import skimage.morphology  # noqa: F401
    except Exception:
        _stub("skimage")
        _stub("skimage.morphology", binary_dilation=_never, binary_erosion=_never)
        transient += ["skimage", "skimage.morphology"]
    try:
        import pymatting  # noqa: F401
    except Exception:
        _stub("pymatting")
        _stub("pymatting.util")
        _stub("pymatting.util.util", row_sum=eigs_ref.row_sum)
        _stub("pymatting.util.kdtree", knn=lambda data, query, k: eigs_ref.knn_exact(data, query, k))
        _stub("pymatting.laplacian")
        _stub("pymatting.laplacian.rw_laplacian", _rw_laplacian=eigs_ref.rw_laplacian_values)
    if not torch.cuda.is_available():
        torch.Tensor.cuda = lambda self, *a, **k: self  # extract.py:146 on a GPU-less box
    sys.path.insert(0, str(REFERENCE_DIR))
    try:
        import extract as ref_extract  # the reference's module, unmodified
    finally:
        sys.path.remove(str(REFERENCE_DIR))
        for name in transient:
            sys.modules.pop(name, None)
    _ref = ref_extract
    return _ref


def run_reference_extract_eig(feature_dict: dict, tmpdir, K: int, images_root=None, **kwargs):
    """Write ``feature_dict`` as a features .pth, call the reference's ``_extract_eig`` on it, load its output.

    kwargs are the reference's own keyword arguments (which_matrix, lapnorm, image_color_lambda, ...).
    Returns the dict the reference saved: {'eigenvalues', 'eigenvectors'}.
    """
    ref = load_reference()
    tmpdir = Path(tmpdir)
    fdir, odir = tmpdir / "features", tmpdir / "eigs"
    fdir.mkdir(parents=True, exist_ok=True)
    odir.mkdir(parents=True, exist_ok=True)
    ffile = fdir / f"{feature_dict['id']}.pth"
    torch.save(feature_dict, str(ffile))
    kwargs.setdefault("image_color_lambda", 0.0)
    ref._extract_eig((0, str(ffile)), K=K, images_root=str(images_root) if images_root else "", output_dir=str(odir),
                     **kwargs)
    image_id = feature_dict["file"][:-4]
    out = torch.load(str(odir / f"{image_id}.pth"), map_location="cpu", weights_only=False)
    return out


def reference_knn_affinity(image_lr: np.ndarray):
    """The reference's own utils.knn_affinity (extract_utils.py:151-188) with the stubbed pymatting knn."""
    ref = load_reference()
    return ref.utils.knn_affinity(image_lr)
