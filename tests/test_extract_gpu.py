"""-m gpu: the image commands' host pipeline (extract.py) end to end -- a retried image's fused segmentations, and
extract_features on a data set with many image shapes."""
import numpy as np
import pytest
import torch

from conftest import load_pkg

pytestmark = pytest.mark.gpu


def _write_pngs(root, shapes, seed0=0):
    from PIL import Image
    synth = load_pkg("synth")
    root.mkdir(parents=True, exist_ok=True)
    names = []
    for i, (H, W) in enumerate(shapes):
        names.append(f"im{i:04d}.png")
        Image.fromarray(synth.blobs_image(H, W, seed0 + i).numpy()).save(root / names[-1])
    return names


def test_extract_all_retry_recomputes_the_fused_segmentations(cuda, tmp_path, monkeypatch):
    """The first solve of one image reports no convergence and comes back with eigenvector 1 negated. The retry
    replaces its eigenpairs, and its fused PNGs must come from those, i.e. equal what the two segmentation commands
    make from the written files."""
    from PIL import Image
    ex = load_pkg("extract")
    spectral = load_pkg("spectral")
    real = spectral.laplacian_eigs
    calls = []

    def first_pass_of_one_image_fails(feats, K, *args, max_steps=0, **kwargs):
        evals, evecs, info, resid = real(feats, K, *args, max_steps=max_steps, **kwargs)
        calls.append(max_steps)
        if len(calls) == 1:
            info[0, 1] = 0
            evecs[0, 1].neg_()
        return evals, evecs, info, resid
    monkeypatch.setattr(spectral, "laplacian_eigs", first_pass_of_one_image_fails)
    root = tmp_path / "images"
    names = _write_pngs(root, [(160, 208)] * 6)
    (tmp_path / "list.txt").write_text("\n".join(names) + "\n")
    fdir, edir, sdir, mdir = (tmp_path / n for n in ("features", "eigs", "single", "multi"))
    ex.extract_all(str(tmp_path / "list.txt"), str(root), "dino_vits16", str(fdir), str(edir), K=5, batch_size=4, seed=0,
                   single_region_dir=str(sdir), multi_region_dir=str(mdir), non_adaptive_num_segments=3)
    assert calls.count(0) == 2 and len(calls) == 3 and calls[2] == 10 * 13 - 1    # two batches, one retry
    ex.extract_single_region_segmentations(str(fdir), str(edir), str(tmp_path / "single2"))
    ex.extract_multi_region_segmentations(str(fdir), str(edir), str(tmp_path / "multi2"), non_adaptive_num_segments=3)
    for n in names:
        stem = n[:-4]
        for fused, two_stage in ((sdir, "single2"), (mdir, "multi2")):
            a = np.array(Image.open(fused / f"{stem}.png"))
            assert np.array_equal(a, np.array(Image.open(tmp_path / two_stage / f"{stem}.png"))), (stem, two_stage)


def test_extract_features_on_many_image_shapes(cuda, tmp_path):
    """14 image shapes with 2-3 images each: more shapes than the batch assembler gives full-size rings, and enough
    images in open batches that it closes some early. Every image is written once, with its own index / id / shape, and
    its k equals forward_k on that image alone, bit for bit."""
    ex = load_pkg("extract")
    utils = load_pkg("extract_utils")
    vit = load_pkg("vit")
    shapes = [(40 + 8 * s, 96 - 4 * s) for s in range(14)]
    per_image = [shapes[i % 14] for i in range(14 * 2 + 9)]              # 9 shapes with 3 images, 5 with 2
    root = tmp_path / "images"
    names = _write_pngs(root, per_image, seed0=100)
    (tmp_path / "list.txt").write_text("\n".join(names) + "\n")
    fdir = tmp_path / "features"
    ex.extract_features(str(tmp_path / "list.txt"), str(root), "dino_vits16", 4, str(fdir), seed=0)
    assert sorted(p.name for p in fdir.iterdir()) == [n[:-4] + ".pth" for n in names]
    model, _, _, _ = vit.get_model("dino_vits16", seed=0, device=cuda)
    for i, n in enumerate(names):
        d = torch.load(fdir / f"{n[:-4]}.pth", map_location="cpu")
        H, W = per_image[i]
        assert int(d["indices"]) == i and d["id"] == n[:-4] and d["file"] == n and d["shape"] == (1, 3, H, W)
        img = torch.from_numpy(utils.read_image_rgb(root / n))[None].to(cuda)
        k_alone = model.forward_k(img).cpu()
        assert d["k"].shape == k_alone.shape and torch.equal(d["k"], k_alone), n
