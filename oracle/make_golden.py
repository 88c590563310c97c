"""Generates tests/golden/*.npz by running the reference's OWN ``_extract_eig`` (imported from /root/reference through
oracle/ref_shim.py) on small seeded inputs. Run in the dev container only:

    python -m oracle.make_golden
    python -m oracle.make_golden --reference-calls    # only the ref_*.npz fixtures

Each fixture stores the inputs (features, optional JPEG bytes + the low-res image the reference derived from it)
and the tensors the reference saved. tests/test_cpu_oracle.py checks the oracle restatement against them;
tests/test_golden_gpu.py checks the CUDA path against them."""
from __future__ import annotations

import importlib
import io
import sys
import tempfile
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from oracle import ref_shim  # noqa: E402

synth = importlib.import_module("deep-spectral-segmentation_b200.synth")
GOLDEN = ROOT / "tests" / "golden"

CASES = [
    # name, N-grid (Hp, Wp), d, K, rank, seed, kwargs
    ("lap_196_k5", (14, 14), 64, 5, 6, 0, {}),
    ("lap_143_k5_odd", (11, 13), 64, 5, 4, 1, {}),
    ("lap_196_k8", (14, 14), 96, 8, 6, 2, {}),
    ("lap_100_nolapnorm", (10, 10), 64, 4, 4, 3, {"lapnorm": False}),
    ("lap_120_nonorm_nothr", (10, 12), 64, 5, 6, 4, {"normalize": False, "threshold_at_zero": False}),
    ("lap_196_color10", (14, 14), 64, 5, 6, 5, {"image_color_lambda": 10.0}),
    ("lap_150_color1", (10, 15), 64, 6, 6, 6, {"image_color_lambda": 1.0}),
    # round 2: odd N (N*N % 4 != 0) with the colour-KNN term, and the random-walk colour affinity
    ("lap_143_color10_odd", (11, 13), 64, 5, 4, 7, {"image_color_lambda": 10.0}),
    ("lap_713_color1_voc", (23, 31), 64, 5, 4, 8, {"image_color_lambda": 1.0}),
    ("lap_143_rw5_odd", (11, 13), 64, 5, 4, 9, {"image_color_lambda": 5.0, "which_color_matrix": "rw"}),
    ("lap_196_rw1", (14, 14), 64, 6, 6, 10, {"image_color_lambda": 1.0, "which_color_matrix": "rw"}),
]
ONLY_NEW = {"lap_143_color10_odd", "lap_713_color1_voc", "lap_143_rw5_odd", "lap_196_rw1"}   # keep round-1 files byte-stable

# segmentation fixtures: (name, (Hp, Wp), regions, seed, kwargs of the reference's multi-region worker). The grids are
# chosen so that no two bands tie for the largest border share: the reference breaks such a tie by LABEL NUMBER
# (np.argmax over np.unique's order), which depends on the unseeded K-means initialisation.
SEG_CASES = [
    ("seg_bands4_adaptive", (6, 10), 4, 0, dict(adaptive=True, non_adaptive_num_segments=4, infer_bg_index=True,
                                                 kmeans_baseline=False, num_eigenvectors=1_000_000)),
    ("seg_bands3_fixed3", (7, 10), 3, 1, dict(adaptive=False, non_adaptive_num_segments=3, infer_bg_index=True,
                                              kmeans_baseline=False, num_eigenvectors=1_000_000)),
    ("seg_bands5_nobg_2vec", (8, 15), 5, 2, dict(adaptive=False, non_adaptive_num_segments=5, infer_bg_index=False,
                                                  kmeans_baseline=False, num_eigenvectors=2)),
    ("seg_bands3_baseline", (6, 10), 3, 3, dict(adaptive=False, non_adaptive_num_segments=3, infer_bg_index=True,
                                                kmeans_baseline=True, num_eigenvectors=1_000_000)),
]


def planted_eigs(Hp, Wp, n_regions, seed):
    """Eigenvector-like embedding with well separated vertical bands (+ small noise), a spectrum whose largest gap
    sits after eigenvalue n_regions - 1, and band-structured 'k' features for the kmeans_baseline branch."""
    g = torch.Generator().manual_seed(seed)
    band = (torch.arange(Wp) * n_regions // Wp)[None, :].expand(Hp, Wp).reshape(-1)
    K = n_regions + 2
    vecs = torch.zeros(K, Hp * Wp)
    vecs[0] = 1.0 / (Hp * Wp) ** 0.5
    for k in range(1, K):
        centres = torch.randn(n_regions, generator=g) * 2.0
        vecs[k] = centres[band] + 0.01 * torch.randn(Hp * Wp, generator=g)
    vals = torch.cat([torch.linspace(0.0, 0.1, n_regions), torch.linspace(0.6, 0.7, K - n_regions)])
    feats = (torch.randn(n_regions, 16, generator=g) * 3.0)[band] + 0.05 * torch.randn(Hp * Wp, 16, generator=g)
    return vals, vecs, feats, band.reshape(Hp, Wp).numpy()


def make_segmentation_golden():
    from PIL import Image
    ref = ref_shim.load_reference()
    for name, (Hp, Wp), nr, seed, kw in SEG_CASES:
        P = 16
        H, W = Hp * P + 7, Wp * P + 2
        vals, vecs, feats, band = planted_eigs(Hp, Wp, nr, seed)
        with tempfile.TemporaryDirectory() as td:
            td = Path(td)
            fdir, edir, o1, o2 = td / "f", td / "e", td / "single", td / "multi"
            for d in (fdir, edir, o1, o2):
                d.mkdir()
            fd = {"k": feats[None].clone(), "indices": torch.tensor(0), "file": f"{name}.jpg", "id": name,
                  "model_name": "dino_vits16", "patch_size": P, "shape": (1, 3, H, W)}
            torch.save(fd, fdir / f"{name}.pth")
            torch.save({"eigenvalues": vals, "eigenvectors": vecs}, edir / f"{name}.pth")
            inp = ref.utils.get_paired_input_files(str(fdir), str(edir))[0]
            ref._extract_single_region_segmentations(inp, threshold=0.05, output_dir=str(o1))
            np.random.seed(1234)     # the reference's KMeans is unseeded: k-means++ draws from numpy's global RNG
            ref._extract_multi_region_segmentations(inp, output_dir=str(o2), **kw)
            single = np.array(Image.open(o1 / f"{name}.png"))
            multi = np.array(Image.open(o2 / f"{name}.png"))
            single_png = np.frombuffer((o1 / f"{name}.png").read_bytes(), np.uint8)
        np.savez_compressed(GOLDEN / f"{name}.npz", eigenvalues=vals.numpy(), eigenvectors=vecs.numpy(), feats=feats.numpy(),
                            shape=np.array([1, 3, H, W]), patch=P, band=band, kwargs=np.array(repr(kw)), threshold=0.05,
                            single=single, multi=multi, single_png=single_png)
        print(name, "labels:", np.unique(multi), "single on:", int((single > 0).sum()))


def make_reference_call_golden():
    """ref_*.npz: inputs and outputs of three direct calls of the reference's functions (its _extract_eig, its
    utils.knn_affinity, its two segmentation workers and utils.get_border_fraction). tests/test_cpu_oracle.py checks the
    oracle against these recorded outputs, so the checks run wherever the tests run."""
    from PIL import Image
    ref = ref_shim.load_reference()
    # _extract_eig with the default flags
    feats = synth.structured_features(150, 64, 6, 42)
    fd = {"k": feats[None], "indices": torch.tensor(0), "file": "x.jpg", "id": "x", "model_name": "dino_vits16",
          "patch_size": 16, "shape": (1, 3, 160, 240)}
    with tempfile.TemporaryDirectory() as td:
        out = ref_shim.run_reference_extract_eig(fd, td, K=6)
    np.savez_compressed(GOLDEN / "ref_extract_eig_150_k6.npz", feats=feats.numpy(), K=6,
                        eigenvalues=np.asarray(out["eigenvalues"]), eigenvectors=out["eigenvectors"].numpy())
    # utils.knn_affinity on a 12 x 15 low-resolution image
    img = synth.blobs_image(12 * 16, 15 * 16, 7).numpy()
    lr = np.array(Image.fromarray(img).resize((15, 12), Image.BILINEAR)) / 255.0
    W = ref_shim.reference_knn_affinity(lr).tocoo()
    np.savez_compressed(GOLDEN / "ref_knn_affinity_12x15.npz", image_lr=lr, shape=np.array(W.shape),
                        row=W.row.astype(np.int32), col=W.col.astype(np.int32), data=W.data)
    # the single- and multi-region workers on a 7 x 11 patch grid, and the border fractions of the multi-region PNG
    vals, vecs, feats, band = planted_eigs(7, 11, 4, 17)
    kw = dict(adaptive=True, non_adaptive_num_segments=4, infer_bg_index=True, kmeans_baseline=False, num_eigenvectors=3)
    with tempfile.TemporaryDirectory() as td:
        fdir, edir, o1, o2 = (Path(td) / n for n in ("f", "e", "s", "m"))
        for d in (fdir, edir, o1, o2):
            d.mkdir()
        fd = {"k": feats[None], "indices": torch.tensor(0), "file": "x.jpg", "id": "x", "model_name": "dino_vits16",
              "patch_size": 16, "shape": (1, 3, 7 * 16 + 3, 11 * 16)}
        torch.save(fd, fdir / "x.pth")
        torch.save({"eigenvalues": vals, "eigenvectors": vecs}, edir / "x.pth")
        inp = ref.utils.get_paired_input_files(str(fdir), str(edir))[0]
        ref._extract_single_region_segmentations(inp, threshold=0.0, output_dir=str(o1))
        np.random.seed(7)        # the reference's KMeans is unseeded: k-means++ draws from numpy's global RNG
        ref._extract_multi_region_segmentations(inp, output_dir=str(o2), **kw)
        single, multi = np.array(Image.open(o1 / "x.png")), np.array(Image.open(o2 / "x.png"))
    border_idx, border_frac = ref.utils.get_border_fraction(multi)
    np.savez_compressed(GOLDEN / "ref_segment_7x11.npz", eigenvalues=vals.numpy(), eigenvectors=vecs.numpy(),
                        feats=feats.numpy(), grid=np.array([7, 11]), kwargs=np.array(repr(kw)), threshold=0.0, rng_seed=7,
                        single=single, multi=multi, border_indices=np.asarray(border_idx),
                        border_fractions=np.asarray(border_frac))
    print("reference calls recorded: lambda", np.asarray(out["eigenvalues"]), "labels", np.unique(multi))


def main():
    assert ref_shim.available(), "reference sources not present"
    GOLDEN.mkdir(parents=True, exist_ok=True)
    from PIL import Image
    import sys as _sys
    if "--reference-calls" in _sys.argv:
        make_reference_call_golden()
        return
    regenerate_all = "--all" in _sys.argv
    for name, (Hp, Wp), d, K, rank, seed, kw in CASES:
        if not regenerate_all and name not in ONLY_NEW and (GOLDEN / f"{name}.npz").is_file():
            continue
        N = Hp * Wp
        P = 16
        H, W = Hp * P + 3, Wp * P + 5  # un-cropped size: exercises the crop arithmetic of get_image_sizes
        feats = synth.structured_features(N, d, rank, seed)
        if kw.get("normalize", True) is False:
            feats = feats - feats.min() + 0.1
        fd = {"k": feats[None].clone(), "indices": torch.tensor(0), "file": f"{name}.jpg", "id": name,
              "model_name": "dino_vits16", "patch_size": P, "shape": (1, 3, H, W)}
        jpeg = np.zeros(0, np.uint8)
        image_lr = np.zeros(0)
        with tempfile.TemporaryDirectory() as td:
            if kw.get("image_color_lambda", 0) > 0:
                img = synth.blobs_image(H, W, 100 + seed).numpy()
                buf = io.BytesIO()
                Image.fromarray(img).save(buf, format="JPEG", quality=95)
                jpeg = np.frombuffer(buf.getvalue(), np.uint8)
                (Path(td) / f"{name}.jpg").write_bytes(buf.getvalue())
                image_lr = np.array(Image.open(str(Path(td) / f"{name}.jpg")).resize((Wp, Hp), Image.BILINEAR)) / 255.0
            out = ref_shim.run_reference_extract_eig(fd, td, K=K, images_root=td, **kw)
        np.savez_compressed(GOLDEN / f"{name}.npz", feats=feats.numpy(), K=K, patch=P, shape=np.array([1, 3, H, W]),
                            kwargs=np.array(repr(kw)), jpeg=jpeg, image_lr=image_lr,
                            eigenvalues=np.asarray(out["eigenvalues"], dtype=np.float32),
                            eigenvectors=out["eigenvectors"].numpy())
        print(name, "lambda:", np.asarray(out["eigenvalues"]))
    make_segmentation_golden()


if __name__ == "__main__":
    main()
