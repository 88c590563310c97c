"""CPU suite: the oracle (oracle/eigs_ref.py, oracle/dino_vit.py) is pinned against
  * the committed golden fixtures produced by the reference's own _extract_eig (tests/golden/, oracle/make_golden.py),
  * recorded outputs of direct calls of the reference's functions (tests/golden/ref_*.npz, same generator),
  * analytic known-answer cases and an independent ViT implementation (transformers.ViTModel)."""
import ast
import io
from pathlib import Path

import numpy as np
import pytest
import torch

from conftest import ROOT, load_pkg
from oracle import dino_vit, eigs_ref

GOLDEN_DIR = ROOT / "tests" / "golden"
GOLDEN = sorted(GOLDEN_DIR.glob("lap_*.npz"))
SEG_GOLDEN = sorted(GOLDEN_DIR.glob("seg_*.npz"))
torch.set_grad_enabled(False)


def _aligned_err(a, b):
    out = []
    for k in range(a.shape[0]):
        s = np.sign(np.dot(a[k], b[k])) or 1.0
        out.append(np.linalg.norm(a[k] - s * b[k]) / np.linalg.norm(b[k]))
    return np.array(out)


def gap_tolerance(feats, K, kw, floor=None, jitter=1e-6):
    """per-vector tolerance max(floor, jitter / gap_k), gap_k = distance of lambda_k to its nearest neighbour (float64
    spectrum). floor = max(2e-5, 5e-8 N): the run-to-run jitter of the reference's own float32 LU + ARPACK route (its
    start vector is unseeded) grows with the matrix size -- 1.3e-5 .. 2.3e-5 measured at N = 713."""
    if floor is None:
        floor = max(2e-5, 5e-8 * feats.shape[-2])
    kw = {k: v for k, v in kw.items() if k in ("normalize", "lapnorm", "threshold_at_zero")}
    vals, _ = eigs_ref.eigh_f64(feats, K + 1, **kw)
    scale = max(1.0, float(np.abs(vals).max()))
    gaps = np.array([min(abs(vals[k] - vals[j]) for j in range(K + 1) if j != k) for k in range(K)]) / scale
    return np.maximum(floor, jitter / np.maximum(gaps, 1e-12))


def load_golden(path):
    z = np.load(path, allow_pickle=False)
    kw = ast.literal_eval(str(z["kwargs"]))
    return z, kw


@pytest.mark.parametrize("path", GOLDEN, ids=[p.stem for p in GOLDEN])
def test_oracle_reproduces_reference_golden(path):
    z, kw = load_golden(path)
    feats = torch.from_numpy(z["feats"])
    image_lr = z["image_lr"] if z["image_lr"].size else None
    if image_lr is not None:
        # the low-res image is re-derived from the stored JPEG exactly as extract.py:199-204 does
        from PIL import Image
        H, W = int(z["shape"][2]), int(z["shape"][3])
        P = int(z["patch"])
        lr = np.array(Image.open(io.BytesIO(z["jpeg"].tobytes())).resize((W // P, H // P), Image.BILINEAR)) / 255.0
        assert np.array_equal(lr, image_lr)
    ev, vec = eigs_ref.extract_eig(feats, int(z["K"]), image_lr=image_lr, rng_seed=0, **kw)
    scale = max(1.0, float(np.abs(z["eigenvalues"]).max()))
    assert np.abs(np.asarray(ev) - z["eigenvalues"]).max() <= 2e-6 * scale
    # ARPACK's start vector is unseeded in the reference: agreement is limited by its own run-to-run jitter,
    # which an eigen-gap g amplifies to ~1e-7/g  (lap_120_nonorm_nothr has gaps of 1e-3)
    assert np.all(_aligned_err(vec.numpy(), z["eigenvectors"]) <= gap_tolerance(feats, int(z["K"]), kw))


def test_oracle_matches_live_reference():
    """Against what the reference's _extract_eig returned for these features (tests/golden/ref_extract_eig_150_k6.npz,
    recorded by ``python -m oracle.make_golden --reference-calls``)."""
    z = np.load(GOLDEN_DIR / "ref_extract_eig_150_k6.npz")
    ev, vec = eigs_ref.extract_eig(torch.from_numpy(z["feats"]), int(z["K"]), rng_seed=1)
    assert np.abs(ev.numpy() - z["eigenvalues"]).max() <= 2e-6
    assert _aligned_err(vec.numpy(), z["eigenvectors"]).max() <= 2e-5
    assert z["eigenvectors"].dtype == np.float32 and z["eigenvectors"].shape == (6, 150)


def test_knn_affinity_restatement_matches_reference_function():
    """Against the matrix the reference's utils.knn_affinity returned for this image (ref_knn_affinity_12x15.npz)."""
    from scipy.sparse import coo_matrix
    z = np.load(GOLDEN_DIR / "ref_knn_affinity_12x15.npz")
    lr = z["image_lr"]
    W_ref = coo_matrix((z["data"], (z["row"], z["col"])), shape=tuple(z["shape"])).toarray()
    W = eigs_ref.knn_affinity(lr).toarray()
    assert np.array_equal(W, W_ref)
    assert np.array_equal(W, W.T) and set(np.unique(W)) <= {0.0, 1.0, 2.0, 3.0, 4.0} and np.all(np.diag(W) == 4)


def test_knn_exact_against_kdtree():
    from scipy.spatial import cKDTree
    rng = np.random.default_rng(0)
    pts = rng.random((300, 5)).astype(np.float32)
    d, i = eigs_ref.knn_exact(pts, pts, 20)
    d2, i2 = cKDTree(pts).query(pts, 20)
    assert np.array_equal(i, i2)
    assert np.abs(d - d2).max() <= 1e-6


def test_oracle_known_answers():
    # complete graph K_n (W = 1 - I after removing self loops is not reachable through features; use eigh_f64 route):
    # two identical clusters of orthogonal features -> W block diagonal -> lambda_0 = lambda_1 = 0
    f = torch.zeros(40, 8)
    f[:20, 0] = 1.0
    f[20:, 1] = 1.0
    W, D = eigs_ref.affinity_matrices(f)
    assert np.allclose(W[:20, :20], 1) and np.allclose(W[:20, 20:], 0)
    assert np.allclose(np.diag(D), 20)
    vals, vecs = eigs_ref.eigh_f64(f, 3)
    assert abs(vals[0]) < 1e-12 and abs(vals[1]) < 1e-12 and abs(vals[2] - 1.0) < 1e-12
    # sign rule: at most half of the entries positive unless all of them are
    v = torch.tensor([[1.0, 1.0, 1.0, -1.0], [1.0, 1.0, 1.0, 1.0], [1.0, -1.0, -1.0, -1.0], [1.0, 1.0, -1.0, -1.0]])
    w = eigs_ref.sign_rule_(v.clone())
    assert torch.equal(w[0], -v[0]) and torch.equal(w[1], v[1]) and torch.equal(w[2], v[2]) and torch.equal(w[3], v[3])


def test_oracle_eigs_against_float64_truth():
    synth = load_pkg("synth")
    feats = synth.structured_features(196, 64, 6, 0)
    ev, vec = eigs_ref.extract_eig(feats, 5, rng_seed=0)
    ev64, vec64 = eigs_ref.eigh_f64(feats, 5)
    assert np.abs(ev.numpy() - ev64).max() <= 1e-5
    assert _aligned_err(vec.numpy(), vec64).max() <= 1e-4
    W, D = eigs_ref.affinity_matrices(feats)
    G = (vec.numpy().astype(np.float64) * np.diag(D)[None]) @ vec.numpy().astype(np.float64).T
    assert np.abs(G - np.eye(5)).max() <= 1e-4   # D-orthonormal, not unit 2-norm


def test_oracle_vit_block_math_against_transformers():
    """Independent implementation of the same architecture: HF ViTModel with the weights copied over (q/k/v split).
    Compared at the native 224 grid where no positional interpolation happens."""
    transformers = pytest.importorskip("transformers")
    ref = dino_vit.build("dino_vits16", seed=0)
    cfg = transformers.ViTConfig(hidden_size=384, num_hidden_layers=12, num_attention_heads=6, intermediate_size=1536,
                                 image_size=224, patch_size=16, layer_norm_eps=1e-6, qkv_bias=True, hidden_act="gelu")
    hf = transformers.ViTModel(cfg, add_pooling_layer=False).eval()
    sd = ref.state_dict()
    new = {"embeddings.cls_token": sd["cls_token"], "embeddings.position_embeddings": sd["pos_embed"],
           "embeddings.patch_embeddings.projection.weight": sd["patch_embed.proj.weight"],
           "embeddings.patch_embeddings.projection.bias": sd["patch_embed.proj.bias"],
           "layernorm.weight": sd["norm.weight"], "layernorm.bias": sd["norm.bias"]}
    d = 384
    for l in range(12):
        p, q = f"blocks.{l}.", f"encoder.layer.{l}."
        w, b = sd[p + "attn.qkv.weight"], sd[p + "attn.qkv.bias"]
        for i, n in enumerate(("query", "key", "value")):
            new[q + f"attention.attention.{n}.weight"] = w[i * d:(i + 1) * d]
            new[q + f"attention.attention.{n}.bias"] = b[i * d:(i + 1) * d]
        new[q + "attention.output.dense.weight"] = sd[p + "attn.proj.weight"]
        new[q + "attention.output.dense.bias"] = sd[p + "attn.proj.bias"]
        new[q + "layernorm_before.weight"] = sd[p + "norm1.weight"]; new[q + "layernorm_before.bias"] = sd[p + "norm1.bias"]
        new[q + "layernorm_after.weight"] = sd[p + "norm2.weight"]; new[q + "layernorm_after.bias"] = sd[p + "norm2.bias"]
        new[q + "intermediate.dense.weight"] = sd[p + "mlp.fc1.weight"]; new[q + "intermediate.dense.bias"] = sd[p + "mlp.fc1.bias"]
        new[q + "output.dense.weight"] = sd[p + "mlp.fc2.weight"]; new[q + "output.dense.bias"] = sd[p + "mlp.fc2.bias"]
    missing, unexpected = hf.load_state_dict(new, strict=False)
    assert not unexpected and all("pooler" in m for m in missing), (missing, unexpected)
    synth = load_pkg("synth")
    x = dino_vit.preprocess_u8(synth.blobs_image(224, 224, 0), 16)
    hs = hf(pixel_values=x, output_hidden_states=True).hidden_states  # hs[i] = residual stream after i blocks
    for n in (0, 1, 6, 11):
        mine = ref.forward_tokens(x, n)
        assert (mine - hs[n]).abs().max().item() <= 2e-4 * max(1.0, hs[n].abs().max().item()), n
    # the hooked K features of the last block, from HF's modules
    lay = hf.encoder.layer[11]
    k_hf = lay.attention.attention.key(lay.layernorm_before(hs[11]))[:, 1:]
    assert (ref.forward_k(x) - k_hf).abs().max().item() <= 2e-4


def test_preprocess_matches_torchvision_transform():
    tv = pytest.importorskip("torchvision")
    synth = load_pkg("synth")
    img = synth.blobs_image(250, 333, 2)
    t = tv.transforms.Compose([tv.transforms.ToTensor(), tv.transforms.Normalize((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))])
    want = t(img.numpy())[None, :, :240, :320]
    assert torch.equal(dino_vit.preprocess_u8(img, 16), want)


# ---------------------------------------------------------------------------------------------------------------
# round 2: segmentation workers (extract.py:283-411) and the random-walk colour affinity (extract_utils.py:191-204)
def load_seg_golden(path):
    z = np.load(path, allow_pickle=False)
    return z, ast.literal_eval(str(z["kwargs"]))


@pytest.mark.parametrize("path", SEG_GOLDEN, ids=[p.stem for p in SEG_GOLDEN])
def test_segmentation_oracle_reproduces_reference_golden(path):
    """oracle/segment_ref.py against the PNGs the reference's own functions wrote (oracle/make_golden.py)."""
    from oracle import segment_ref
    z, kw = load_seg_golden(path)
    P = int(z["patch"])
    Hp, Wp = int(z["shape"][2]) // P, int(z["shape"][3]) // P
    single = segment_ref.single_region(z["eigenvectors"], Hp, Wp, float(z["threshold"]))
    assert np.array_equal(single, z["single"])
    np.random.seed(1234)                       # same RNG state as the generating call: labels are then identical too
    multi = segment_ref.multi_region(z["eigenvalues"], z["eigenvectors"], z["feats"], Hp, Wp, **kw)
    assert np.array_equal(multi, z["multi"])
    assert segment_ref.same_partition(multi, z["band"])          # and it is the planted partition


def test_segmentation_oracle_matches_live_reference():
    """Against the PNGs the reference's two segmentation workers wrote for these eigenvectors and the border fractions
    its utils.get_border_fraction returned for the multi-region one (ref_segment_7x11.npz)."""
    from oracle import segment_ref
    z = np.load(GOLDEN_DIR / "ref_segment_7x11.npz")
    kw = ast.literal_eval(str(z["kwargs"]))
    Hp, Wp = (int(v) for v in z["grid"])
    vals, vecs, feats = z["eigenvalues"], z["eigenvectors"], z["feats"]
    assert np.array_equal(z["single"], segment_ref.single_region(vecs, Hp, Wp, float(z["threshold"])))
    np.random.seed(int(z["rng_seed"]))           # the RNG state the reference's K-means started from
    assert np.array_equal(z["multi"], segment_ref.multi_region(vals, vecs, feats, Hp, Wp, **kw))
    i1, c1 = segment_ref.get_border_fraction(z["multi"])
    assert np.array_equal(i1, z["border_indices"]) and np.array_equal(c1, z["border_fractions"])


def test_rw_affinity_restatement_properties():
    """pymatting's _rw_laplacian restated (oracle/eigs_ref.py): 3x3 clamped stencil, duplicates summed by csr_matrix."""
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (6, 9, 3)) / 255.0
    vals, ii, jj = eigs_ref.rw_laplacian_values(img, 0.033, 1)
    assert vals.shape == (6 * 9 * 9,) and ii.dtype == np.int32 and jj.dtype == np.int32
    # pymatting's loop order: pixel-major, offsets (dy, dx) fastest; first pixel (corner): 4 of its 9 entries are itself
    assert np.array_equal(ii[:9], np.zeros(9)) and list(jj[:9]) == [0, 0, 1, 0, 0, 1, 9, 9, 10]
    W = eigs_ref.rw_affinity(img).toarray()
    assert np.array_equal(W, W.T) and W[0, 0] == 4.0 and W[4, 4] == 2.0 and W[9 + 4, 9 + 4] == 1.0
    zi, zj = img[2, 3], img[3, 4]
    assert abs(W[2 * 9 + 3, 3 * 9 + 4] - np.exp(-900 * np.linalg.norm(zi - zj) ** 2)) < 1e-15
    assert (W > 0).sum(1).max() <= 9
