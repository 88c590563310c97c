"""CPU suite: the C-ABI library loads here (no GPU), exports every symbol include/dss_b200.h declares, validates its
arguments before touching the device, and its host-side positional-embedding interpolation matches upstream DINO."""
import ctypes as C
import re
from pathlib import Path

import pytest
import torch

from conftest import ROOT, load_pkg


def _declared_symbols():
    text = (ROOT / "include" / "dss_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dss_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    _lib = load_pkg("_lib")
    lib = _lib.load()
    names = _declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"libdss_b200.so does not export {n}"
    # and the ctypes prototype table covers the whole header
    assert set(names) == set(_lib.PROTOTYPES), set(names) ^ set(_lib.PROTOTYPES)
    assert lib.dss_version() >= 1


def test_bad_arguments_are_rejected_before_any_device_work():
    _lib = load_pkg("_lib")
    lib = _lib.load()
    launches_before = lib.dss_kernel_launch_count()     # the counter is per process: GPU tests may have run before
    assert lib.dss_affinity(None, 1, 10, 8, 3, None, 0.0, None, 12, None, None, 0, None) == -1
    assert b"null" in lib.dss_last_error()
    buf = torch.zeros(1 << 16, dtype=torch.uint8)
    p = (buf.data_ptr() + 255) // 256 * 256
    assert lib.dss_affinity(p, 1, 10, 8, 3, None, 0.0, p, 11, None, p, 1 << 15, None) == -1     # ldw not multiple of 4
    assert lib.dss_affinity(p, 1, 10, 8, 3, None, 0.0, p, 12, None, p, 16, None) == -3         # workspace too small
    assert lib.dss_eigsh_laplacian(p, None, 12, 1, 10, 10, 1, 0.0, 0, p, p, p, None, p, 1 << 15, None) == -1   # K >= N
    assert lib.dss_eigsh_laplacian(p, None, 12, 1, 10, 0, 1, 0.0, 0, p, p, p, None, p, 1 << 15, None) == -1    # K < 1
    assert lib.dss_op_gemm_f16(p, p, p, p, 16, 30, 64, 0, None, 0, 0, None) == -1           # N % 32
    assert lib.dss_op_layernorm_f16(p, p, p, p, 4, 100, 1e-6, None) == -1                   # unsupported width
    cfg = _lib.VitConfig(16, 384, 12, 5, 4, 14, 1e-6)                                       # 384 / 5 != 64
    h = C.c_void_p()
    assert lib.dss_vit_create(C.byref(cfg), C.byref(h)) == -1
    cfg = _lib.VitConfig(16, 384, 12, 6, 4, 14, 1e-6)
    assert lib.dss_vit_create(C.byref(cfg), C.byref(h)) == 0
    assert lib.dss_vit_workspace_bytes(h, 2, 224, 224) > 2 * 197 * 384 * 4
    assert lib.dss_vit_workspace_bytes(h, 2, 8, 224) == 0                                   # smaller than a patch
    assert lib.dss_vit_forward_k(h, p, 1, 224, 224, -1, p, p, 1 << 15, None) == -1          # weights not loaded
    lib.dss_vit_destroy(h)
    assert lib.dss_affinity_workspace_bytes(2, 900, 384) >= 2 * 900 * 384 * 4
    assert lib.dss_kernel_launch_count() == launches_before                                 # nothing was launched


@pytest.mark.parametrize("name,Hp,Wp", [("dino_vits16", 30, 30), ("dino_vits16", 23, 31), ("dino_vits16", 14, 14),
                                        ("dino_vits16", 7, 40), ("dino_vitb8", 60, 60), ("dino_vitb8", 28, 28)])
def test_pos_embed_interpolation_matches_upstream(name, Hp, Wp):
    from oracle import dino_vit
    vit = load_pkg("vit")
    ref = dino_vit.build(name, seed=3)
    P = ref.cfg.patch
    want = ref.interpolate_pos_encoding(Hp * Wp, Hp * P, Wp * P)[0]
    got = vit.pos_embed_interp_host(ref.pos_embed, ref.cfg.grid0, Hp, Wp)
    assert got.shape == want.shape
    assert (got - want).abs().max().item() <= 2e-6


def test_product_path_fails_loudly_without_cuda(tmp_path):
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    _lib = load_pkg("_lib")
    vit = load_pkg("vit")
    spectral = load_pkg("spectral")
    ex = load_pkg("extract")
    with pytest.raises(_lib.DssError):
        vit.get_model("dino_vits16", device="cpu", seed=0)
    with pytest.raises(_lib.DssError, match="pretrained DINO weights not found"):
        vit.get_model("dino_vits16", device="cpu")          # no checkpoint and no explicit opt-in to random weights
    with pytest.raises(_lib.DssError):
        spectral.affinity(torch.zeros(1, 16, 8))
    with pytest.raises(_lib.DssError):
        spectral.eigsh_laplacian(torch.zeros(1, 16, 16), 16, 3)
    (tmp_path / "list.txt").write_text("a.jpg\n")
    with pytest.raises(_lib.DssError):
        ex.extract_features(str(tmp_path / "list.txt"), str(tmp_path), "dino_vits16", 1, str(tmp_path / "out"), seed=0)
    with pytest.raises(ValueError):
        vit.get_model("resnet50")


def test_no_product_module_imports_the_oracle():
    pkg = ROOT / "deep-spectral-segmentation_b200"
    for f in list(pkg.glob("*.py")) + [ROOT / "extract" / "extract.py"]:
        src = f.read_text()
        assert "oracle" not in src.replace("# oracle", ""), f"{f} references the oracle"
