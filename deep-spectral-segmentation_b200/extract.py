"""Drop-in replacements for the reference's hot-path callables (extract/extract.py):

    extract_features  (:21-116)   images -> features/{id}.pth      {'k','indices','file','id','model_name','patch_size','shape'}
    _extract_eig      (:119-244)  one features file -> eigs/{image_id}.pth  {'eigenvalues','eigenvectors'}
    extract_eigs      (:247-280)  directory of features files -> eigs files (batched on the GPU)
    extract_all                   fused: images -> both file layouts (+ optional segmentations) without the disk round-trip
    extract_single_region_segmentations / extract_multi_region_segmentations  (:283-411)  eigs -> PNG masks (GPU kernels)
    extract_bbox_features (:500-544)  DINO CLS embedding of every bounding-box crop

Same argument names, defaults, file layouts and skip-if-exists behaviour; all arithmetic runs in libdss_b200. Host I/O
(decode, pinned staging, .pth / PNG writers) is threaded, see io_pipeline.py."""
from __future__ import annotations

from collections import defaultdict
from pathlib import Path
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from . import _lib, io_pipeline, segment, spectral
from . import extract_utils as utils

torch.set_grad_enabled(False)  # extract.py:838


def _rank_world() -> Tuple[int, int]:
    """(rank, world size) of a multi-process launch (torchrun or anything else that sets RANK / WORLD_SIZE); (0, 1)
    otherwise. Images are the only parallel axis of the path (SURVEY 8e): every command below gives rank r the items
    r, r + R, r + 2R, ... of its sorted work list, on the GPU LOCAL_RANK; the ranks exchange nothing and write
    disjoint files, so `torchrun --nproc-per-node 8 extract.py extract_all ...` is the multi-GPU form of the command."""
    import os
    world = int(os.environ.get("WORLD_SIZE", "1") or 1)
    rank = int(os.environ.get("RANK", "0") or 0)
    if world < 1 or not (0 <= rank < world):
        raise ValueError(f"RANK={rank} outside WORLD_SIZE={world}")
    return rank, world


def _my_share(items: list) -> list:
    rank, world = _rank_world()
    return items if world == 1 else items[rank::world]


def _device():
    if not torch.cuda.is_available():
        raise _lib.DssError("a CUDA device is required: the hot path has no CPU implementation")
    import os
    if _rank_world()[1] > 1 and os.environ.get("LOCAL_RANK") is not None:
        torch.cuda.set_device(int(os.environ["LOCAL_RANK"]) % torch.cuda.device_count())
    return torch.device("cuda", torch.cuda.current_device())


def _feature_dict(k: torch.Tensor, index: int, file: str, model_name: str, patch_size: int, H: int, W: int) -> dict:
    """The dict the reference saves at extract.py:98-110 (k is (1, N, d) fp32 on the CPU; shape is un-cropped)."""
    return {"k": k, "indices": torch.tensor(index), "file": file, "id": Path(file).stem, "model_name": model_name,
            "patch_size": patch_size, "shape": (1, 3, H, W)}


def _feature_items(output_dir, files_indices, model_name, patch_size, H, W):
    """Writer items (io_pipeline) for the feature dicts of one batch: extract.py:98-110, k taken from arrays['k']."""
    items = []
    for j, (file, index) in enumerate(files_indices):
        extra = {"file": file, "id": Path(file).stem, "model_name": model_name, "patch_size": patch_size, "shape": (1, 3, H, W)}
        items.append((str(Path(output_dir) / f"{Path(file).stem}.pth"), j, extra,
                      {"k": ("slice1", "k"), "indices": ("tensor0d", index)}))
    return items


def _eigs_items(output_dir, image_ids, which_matrix="laplacian", skip=()):
    """Writer items for the eigs dicts of one batch (extract.py:242). The 'affinity' branch of the reference keeps
    `eigenvalues` as the ascending numpy array eigsh returned while the eigenvectors are flipped (extract.py:171-172):
    the caller passes arrays['evals'] already flipped and it is saved as numpy."""
    how = "np_slice" if which_matrix == "affinity" else "slice"
    return [(str(Path(output_dir) / f"{image_id}.pth"), j, {}, {"eigenvalues": (how, "evals"), "eigenvectors": ("slice", "evecs")})
            for j, image_id in enumerate(image_ids) if j not in skip]


class _Batcher:
    """Groups items by a shape key. A group is handed to ``flush`` when it reaches ``batch_size``; when more than
    ``max_pending`` items are waiting in total (data sets with hundreds of distinct image sizes, e.g. VOC), the
    largest group is flushed early, so host memory stays bounded and outputs appear steadily."""

    def __init__(self, batch_size: int, flush, max_pending: Optional[int] = None):
        self.batch_size = max(1, int(batch_size))
        self.flush_fn = flush
        self.max_pending = max_pending if max_pending is not None else 8 * self.batch_size
        self.groups: Dict[object, list] = defaultdict(list)
        self.count = 0

    def _flush(self, key):
        items = self.groups.pop(key, [])
        self.count -= len(items)
        if items:
            self.flush_fn(key, items)

    def add(self, key, item):
        self.groups[key].append(item)
        self.count += 1
        if len(self.groups[key]) >= self.batch_size:
            self._flush(key)
        elif self.count > self.max_pending:
            self._flush(max(self.groups, key=lambda k: len(self.groups[k])))

    def finish(self):
        for key in list(self.groups.keys()):
            self._flush(key)


def extract_features(images_list: str, images_root: Optional[str], model_name: str, batch_size: int, output_dir: str,
                     which_block: int = -1, checkpoint: Optional[str] = None, seed: Optional[int] = None,
                     random_init: bool = False, yes: Optional[bool] = None, num_workers: Optional[int] = None,
                     num_workers_out: int = 4, writer: str = "process"):
    """
    Extract features from a list of images.

    Example:
        python extract.py extract_features \
            --images_list "./data/VOC2012/lists/images.txt" \
            --images_root "./data/VOC2012/images" \
            --output_dir "./data/VOC2012/features/dino_vits16" \
            --model_name dino_vits16 \
            --batch_size 1
    """
    utils.make_output_dir(output_dir, assume_yes=yes)
    model_name = model_name.lower()
    if not ("dino" in model_name or "mocov3" in model_name):
        raise ValueError(model_name)
    dev = _device()
    model, _, patch_size, _ = utils.get_model(model_name, checkpoint=checkpoint, seed=seed, device=dev,
                                              random_init=random_init)
    filenames = Path(images_list).read_text().splitlines()
    dataset = utils.ImagesDataset(filenames=filenames, images_root=images_root)
    print(f"Dataset size: {len(dataset)=}")
    rings: Dict[tuple, io_pipeline.PinnedRing] = {}

    with io_pipeline.make_writer(writer, num_workers_out) as wr:
        def flush(shape_key, items):
            H, W = shape_key
            ring = rings.get(shape_key)
            if ring is None:
                ring = rings[shape_key] = io_pipeline.PinnedRing(shape_key, max(1, int(batch_size)), dev)
            slot, host = ring.stage([it[0] for it in items])
            k = model.forward_k(ring.to_device(slot, host), which_block=which_block).cpu()
            wr.submit_batch({"k": k.numpy()}, _feature_items(output_dir, [(it[1], it[2]) for it in items], model_name,
                                                             patch_size, H, W))

        batcher = _Batcher(batch_size, flush)
        todo = []
        for i in _my_share(list(range(len(dataset)))):
            output_file = Path(output_dir) / f"{Path(dataset.filenames[i]).stem}.pth"
            if output_file.is_file():
                print(f"Skipping existing file {str(output_file)}")
            else:
                todo.append(i)
        for image, file, index in io_pipeline.ImagePrefetcher(dataset.__getitem__, todo, num_workers):
            batcher.add((int(image.shape[0]), int(image.shape[1])), (image, file, index))
        batcher.finish()
    print(f"Saved features to {output_dir}")


def _load_image_lr_u8(images_root: str, image_id: str, W_lr: int, H_lr: int) -> np.ndarray:
    """extract.py:199-203: PIL open (no .convert), BILINEAR resize of the WHOLE image to (W_lr, H_lr) -> uint8 pixels."""
    from PIL import Image
    image_file = str(Path(images_root) / f"{image_id}.jpg")
    return np.array(Image.open(image_file).resize((W_lr, H_lr), Image.BILINEAR))


def _load_image_lr(images_root: str, image_id: str, W_lr: int, H_lr: int) -> np.ndarray:
    """extract.py:199-204: the low-resolution image / 255 -> float64 (H_lr, W_lr, 3)."""
    return _load_image_lr_u8(images_root, image_id, W_lr, H_lr) / 255.0


def _check_supported(which_matrix, which_color_matrix, image_color_lambda):
    if which_matrix == "affinity_torch":
        raise RuntimeError("which_matrix='affinity_torch' calls torch.eig, which PyTorch removed (dead in the reference)")
    if which_matrix not in ("laplacian", "matting_laplacian", "affinity", "affinity_svd"):
        raise ValueError(f"unknown which_matrix={which_matrix!r}")
    if which_matrix in ("laplacian", "matting_laplacian") and image_color_lambda > 0 \
            and which_color_matrix not in ("knn", "rw"):
        raise ValueError(f"unknown which_color_matrix={which_color_matrix!r} (the reference knows 'knn' and 'rw')")


def _color_inputs(images_root, image_ids, W_lr, H_lr, which_color_matrix, dev):
    """Low-resolution colour images of a batch on the device: fp32 /255 for 'knn', the uint8 pixels for 'rw'."""
    lr = np.stack([_load_image_lr_u8(images_root, i, W_lr, H_lr) for i in image_ids]).reshape(len(image_ids), H_lr * W_lr, 3)
    if which_color_matrix == "rw":
        return torch.from_numpy(np.ascontiguousarray(lr)).to(dev)
    return torch.from_numpy((lr / 255.0).astype(np.float32)).to(dev)


def _bad_rows(evals: torch.Tensor, evecs: torch.Tensor, info: torch.Tensor) -> List[int]:
    """Rows of a batch (CPU tensors) whose solve did not reach the tolerance or came back non-finite. Three array
    operations per batch: a per-image Python loop here cost more main-thread time than launching the kernels did. They
    run in numpy, on this thread: torch would hand them to its intra-op pool, and with the decode threads holding every
    core each call waited ~27 ms for the pool's threads (measured on a 16-core B200 host: 0.43 s of 0.7 s for 2048
    images)."""
    B = len(info)
    ok = ((info[:, 1].numpy() != 0) & np.isfinite(evecs.numpy()).reshape(B, -1).all(1)
          & np.isfinite(evals.numpy()).reshape(B, -1).all(1))
    return np.flatnonzero(~ok).tolist()


def _solve_with_retry(solve, n_images: int, N: int):
    """Runs ``solve(sel, max_steps)`` (sel = None for the whole batch, else a list of batch rows) and retries the images
    whose Lanczos run did not reach its tolerance or came back non-finite with the largest possible Krylov space
    (max_steps = N - 1). The reference's own safety net is a second eigsh call (which='SM', extract.py:226-234).
    Returns (eigenvalues, eigenvectors, info, failed rows) on the CPU."""
    evals, evecs, info = (t.cpu() for t in solve(None, 0))
    bad = _bad_rows(evals, evecs, info)
    failed = []
    if bad:
        ev2, vec2, info2 = (t.cpu() for t in solve(bad, max(N - 1, 1)))
        for j, i in enumerate(bad):
            ok = int(info2[j, 1]) == 1 and bool(torch.isfinite(vec2[j]).all() and torch.isfinite(ev2[j]).all())
            if ok:
                evals[i], evecs[i], info[i] = ev2[j], vec2[j], info2[j]
            else:
                failed.append(i)
    return evals, evecs, info, failed


def _eigs_for_group(data_dicts: List[dict], K: int, images_root, which_features, normalize, lapnorm, threshold_at_zero,
                    image_downsample_factor, image_color_lambda, dev, which_matrix="laplacian", which_color_matrix="knn"
                    ) -> Tuple[torch.Tensor, torch.Tensor, List[int]]:
    """One GPU batch: feature dicts whose patch grids have the same size -> (eigenvalues [B,K], eigenvectors [B,K,N],
    rows whose solve failed even after the retry) on the CPU."""
    feats = torch.stack([d[which_features].squeeze() for d in data_dicts]).to(torch.float32)
    feats = feats.pin_memory().to(dev, non_blocking=True)
    if which_matrix in ("affinity", "affinity_svd"):
        def solve(sel, max_steps):
            f = feats if sel is None else feats[sel]
            return spectral.affinity_eigs(f, K, which_matrix, normalize, threshold_at_zero, max_steps=max_steps)
    else:
        rgb_lr, lr_size = None, None
        sizes = utils.get_image_sizes(data_dicts[0])
        P, H_patch, W_patch, H_pad, W_pad = sizes[4:]
        factor = P if image_downsample_factor is None else image_downsample_factor
        H_lr, W_lr = H_pad // factor, W_pad // factor
        if (H_patch, W_patch) != (H_lr, W_lr):
            # extract.py:148,179-188: normalise first, then bilinear up-sampling (no re-normalisation afterwards)
            if normalize:
                feats = spectral.normalize_rows(feats)
                normalize = False
            feats = spectral.upsample_bilinear(feats, H_patch, W_patch, H_lr, W_lr)
        if image_color_lambda > 0:
            rgb_lr = _color_inputs(images_root, [d["file"][:-4] for d in data_dicts], W_lr, H_lr, which_color_matrix, dev)
            lr_size = (H_lr, W_lr)

        def solve(sel, max_steps):
            f = feats if sel is None else feats[sel]
            rgb = rgb_lr if (sel is None or rgb_lr is None) else rgb_lr[sel]
            return spectral.laplacian_eigs(f, K, normalize, threshold_at_zero, lapnorm, rgb, lr_size, image_color_lambda,
                                           max_steps=max_steps, which_color_matrix=which_color_matrix)[:3]
    evals, evecs, info, failed = _solve_with_retry(solve, len(data_dicts), feats.shape[1])
    if failed:
        print(f"Warning: eigensolver did not converge for {[data_dicts[i]['id'] for i in failed]}; no file is written for them")
    if which_matrix == "affinity" and bool((info[:, 2] != 0).any()):
        print("Warning: a negative eigenvalue exceeds the K-th largest in magnitude; eigsh(which='LM') would pick it")
    return evals, evecs, failed


def _eigs_dict(which_matrix, evals_k: torch.Tensor, evecs_k: torch.Tensor) -> dict:
    """extract.py:242. The 'affinity' branch of the reference keeps `eigenvalues` as the ascending numpy array eigsh
    returned while the eigenvectors are flipped to descending order (extract.py:171-172); mirrored here."""
    eigenvalues = evals_k.flip(0).numpy().copy() if which_matrix == "affinity" else evals_k.clone()
    return {"eigenvalues": eigenvalues, "eigenvectors": evecs_k.clone()}


def _save_eigs(output_file, which_matrix, evals_k: torch.Tensor, evecs_k: torch.Tensor):
    Path(output_file).parent.mkdir(parents=True, exist_ok=True)
    torch.save(_eigs_dict(which_matrix, evals_k, evecs_k), str(output_file))


def _extract_eig(inp: Tuple[int, str], K: int, images_root: str, output_dir: str, which_matrix: str = "laplacian",
                 which_features: str = "k", normalize: bool = True, lapnorm: bool = True,
                 which_color_matrix: str = "knn", threshold_at_zero: bool = True,
                 image_downsample_factor: Optional[int] = None, image_color_lambda: float = 10):
    """Single-image worker with the reference's signature (extract.py:119-132); writes {output_dir}/{image_id}.pth."""
    index, features_file = inp
    data_dict = torch.load(features_file, map_location="cpu")
    image_id = data_dict["file"][:-4]
    output_file = str(Path(output_dir) / f"{image_id}.pth")
    if Path(output_file).is_file():
        print(f"Skipping existing file {str(output_file)}")
        return
    _check_supported(which_matrix, which_color_matrix, image_color_lambda)
    evals, evecs, failed = _eigs_for_group([data_dict], K, images_root, which_features, normalize, lapnorm,
                                           threshold_at_zero, image_downsample_factor, image_color_lambda, _device(),
                                           which_matrix, which_color_matrix)
    if failed:
        raise _lib.DssError(f"eigensolver did not converge for {image_id}")
    _save_eigs(output_file, which_matrix, evals[0], evecs[0])


def extract_eigs(images_root: str, features_dir: str, output_dir: str, which_matrix: str = "laplacian",
                 which_color_matrix: str = "knn", which_features: str = "k", normalize: bool = True,
                 threshold_at_zero: bool = True, lapnorm: bool = True, K: int = 20,
                 image_downsample_factor: Optional[int] = None, image_color_lambda: float = 0.0,
                 multiprocessing: int = 0, batch_size: int = 128, yes: Optional[bool] = None,
                 num_workers: Optional[int] = None, num_workers_out: int = 4, writer: str = "process"):
    """
    Extracts eigenvalues from features.

    Example:
        python extract.py extract_eigs \
            --images_root "./data/VOC2012/images" \
            --features_dir "./data/VOC2012/features/dino_vits16" \
            --which_matrix "laplacian" \
            --output_dir "./data/VOC2012/eigs/laplacian" \
            --K 5
    """
    utils.make_output_dir(output_dir, assume_yes=yes)
    kwargs = dict(K=K, which_matrix=which_matrix, which_features=which_features, which_color_matrix=which_color_matrix,
                  normalize=normalize, threshold_at_zero=threshold_at_zero, images_root=images_root,
                  output_dir=output_dir, image_downsample_factor=image_downsample_factor,
                  image_color_lambda=image_color_lambda, lapnorm=lapnorm)
    print(kwargs)
    if multiprocessing:
        print(f"Note: multiprocessing={multiprocessing} is ignored: images are batched inside the GPU kernels "
              f"({batch_size} per launch) instead of forked CPU workers")
    _check_supported(which_matrix, which_color_matrix, image_color_lambda)
    dev = _device()
    inputs = _my_share(list(enumerate(sorted(Path(features_dir).iterdir()))))
    import time
    start = time.time()
    all_failed: List[str] = []

    with io_pipeline.make_writer(writer, num_workers_out) as wr:
        def flush(key, dds):
            evals, evecs, failed = _eigs_for_group(dds, K, images_root, which_features, normalize, lapnorm,
                                                   threshold_at_zero, image_downsample_factor, image_color_lambda, dev,
                                                   which_matrix, which_color_matrix)
            all_failed.extend(dds[j]["id"] for j in failed)
            ev = evals.flip(1) if which_matrix == "affinity" else evals
            wr.submit_batch({"evals": ev.numpy(), "evecs": evecs.numpy()},
                            _eigs_items(output_dir, [d["file"][:-4] for d in dds], which_matrix, skip=failed))

        batcher = _Batcher(batch_size, flush)
        load = lambda i: torch.load(str(inputs[i][1]), map_location="cpu")   # noqa: E731  (file reads overlap on threads)
        for data_dict in io_pipeline.ImagePrefetcher(load, range(len(inputs)), num_workers):
            image_id = data_dict["file"][:-4]
            if (Path(output_dir) / f"{image_id}.pth").is_file():
                print(f"Skipping existing file {str(Path(output_dir) / (image_id + '.pth'))}")
                continue
            batcher.add((tuple(data_dict[which_features].shape[-2:]), tuple(data_dict["shape"])), data_dict)
        batcher.finish()
    print(f"Finished in {time.time() - start:.1f}s")
    if all_failed:
        raise _lib.DssError(f"eigensolver did not converge for {len(all_failed)} image(s): {all_failed[:8]} -- their files "
                            "were not written (all other outputs were)")


# ---------------------------------------------------------------------------------------------------------------
# Segmentations (SURVEY 8f rank 1): device kernels on batches of eigenvector files
def _png_writer_pool(num_threads: int):
    from concurrent.futures import ThreadPoolExecutor
    return ThreadPoolExecutor(max(1, num_threads), thread_name_prefix="dss-png")


def _save_png(arr_u8: np.ndarray, path: str):
    from PIL import Image
    Image.fromarray(arr_u8, mode="L").save(path)


def _paired_dicts(inputs, output_dir, num_workers):
    """Loads (features, eigs) file pairs on threads, skipping pairs whose PNG exists (extract.py:300-304)."""
    def load(i):
        _, (feature_path, eigs_path) = inputs[i]
        data_dict = torch.load(str(feature_path), map_location="cpu")
        data_dict.update(torch.load(str(eigs_path), map_location="cpu", weights_only=False))
        return data_dict
    for data_dict in io_pipeline.ImagePrefetcher(load, range(len(inputs)), num_workers):
        output_file = str(Path(output_dir) / f"{Path(data_dict['id'])}.png")
        if Path(output_file).is_file():
            print(f"Skipping existing file {str(output_file)}")
            continue
        yield data_dict, output_file


def extract_single_region_segmentations(features_dir: str, eigs_dir: str, output_dir: str, threshold: float = 0.0,
                                        multiprocessing: int = 0, yes: Optional[bool] = None, batch_size: int = 256,
                                        num_workers: Optional[int] = None):
    """
    Thresholds the Fiedler-like eigenvector of every image into a patch-grid mask (reference
    extract/extract.py:364-411), same command / file contract; the threshold runs on the GPU for a batch of images.

    Example:
    python extract.py extract_single_region_segmentations \
        --features_dir "./data/VOC2012/features/dino_vits16" \
        --eigs_dir "./data/VOC2012/eigs/laplacian" \
        --output_dir "./data/VOC2012/single_region_segmentation/patches" \
    """
    utils.make_output_dir(output_dir, assume_yes=yes)
    inputs = _my_share(utils.get_paired_input_files(features_dir, eigs_dir))
    dev = _device()
    with _png_writer_pool(4) as pool:
        def flush(key, items):
            evecs = torch.stack([torch.as_tensor(d["eigenvectors"]) for d, _ in items]).to(dev)
            masks = segment.threshold_masks(evecs, threshold, which=1).cpu().numpy()
            for j, (d, output_file) in enumerate(items):
                _, _, _, _, _, H_patch, W_patch, _, _ = utils.get_image_sizes(d)
                pool.submit(_save_png, masks[j].reshape(H_patch, W_patch).copy(), output_file)

        batcher = _Batcher(batch_size, flush)
        for d, output_file in _paired_dicts(inputs, output_dir, num_workers):
            batcher.add(tuple(torch.as_tensor(d["eigenvectors"]).shape), (d, output_file))
        batcher.finish()


def extract_multi_region_segmentations(features_dir: str, eigs_dir: str, output_dir: str, adaptive: bool = False,
                                       non_adaptive_num_segments: int = 4, infer_bg_index: bool = True,
                                       kmeans_baseline: bool = False, num_eigenvectors: int = 1_000_000,
                                       multiprocessing: int = 0, random_state: Optional[int] = None,
                                       yes: Optional[bool] = None, batch_size: int = 256,
                                       num_workers: Optional[int] = None):
    """
    K-means on the non-constant eigenvectors (or on the raw features, ``kmeans_baseline``) of every image -> label map
    on the patch grid, background label swapped to 0 (reference extract/extract.py:283-376), same command / file
    contract. The clustering is the batched device K-means of csrc/segment.cu (k-means++ / Lloyd with scikit-learn's
    stopping rules); the reference's KMeans is unseeded, so label NUMBERS differ from run to run there and only the
    partition is comparable. ``random_state`` seeds the device generator (default 0: reproducible).

    Example:
    python extract.py extract_multi_region_segmentations \
        --features_dir "./data/VOC2012/features/dino_vits16" \
        --eigs_dir "./data/VOC2012/eigs/laplacian" \
        --output_dir "./data/VOC2012/multi_region_segmentation/fixed" \
    """
    utils.make_output_dir(output_dir, assume_yes=yes)
    inputs = _my_share(utils.get_paired_input_files(features_dir, eigs_dir))
    dev = _device()
    seed = 0 if random_state is None else int(random_state)
    with _png_writer_pool(4) as pool:
        def flush(key, items):
            dicts = [d for d, _ in items]
            ks = [segment.adaptive_num_clusters(torch.as_tensor(d["eigenvalues"]).numpy()) if adaptive
                  else non_adaptive_num_segments for d in dicts]
            _, _, _, _, _, H_patch, W_patch, _, _ = utils.get_image_sizes(dicts[0])
            if kmeans_baseline:
                pts = torch.stack([d["k"].squeeze() for d in dicts]).to(dev)
                n_pts, layout = pts.shape[1], "features"
            else:
                pts = torch.stack([torch.as_tensor(d["eigenvectors"])[1:1 + num_eigenvectors] for d in dicts]).to(dev)
                n_pts, layout = pts.shape[2], "eigenvectors"
            if n_pts == H_patch * W_patch:     # extract.py:328-333
                grid = (H_patch, W_patch)
            elif n_pts == H_patch * W_patch * 4:
                grid = (H_patch * 2, W_patch * 2)
            else:
                raise ValueError(f"{n_pts} labels do not fit a {H_patch} x {W_patch} patch grid")
            labels, _, _ = segment.kmeans_labels(pts, ks, grid, infer_bg_index, layout, seed,
                                                 image_keys=[int(d["indices"]) for d in dicts])
            labels = labels.cpu().numpy()
            for j, (_, output_file) in enumerate(items):
                pool.submit(_save_png, labels[j].reshape(grid).copy(), output_file)

        batcher = _Batcher(batch_size, flush)
        for d, output_file in _paired_dicts(inputs, output_dir, num_workers):
            key = (tuple(torch.as_tensor(d["eigenvectors"]).shape), tuple(d["k"].shape), tuple(d["shape"]))
            batcher.add(key, (d, output_file))
        batcher.finish()


# ---------------------------------------------------------------------------------------------------------------
def extract_bbox_features(images_root: str, bbox_file: str, model_name: str, output_file: str,
                          checkpoint: Optional[str] = None, seed: Optional[int] = None, random_init: bool = False,
                          batch_size: int = 64):
    """
    DINO CLS embedding of every bounding-box crop (reference extract/extract.py:500-544), same command / file
    contract: each dict of ``bbox_file`` gains 'features' [n_boxes, d] fp32. Crops of equal size are batched.

    Example:
        python extract.py extract_bbox_features \
            --model_name dino_vits16 \
            --images_root "./data/VOC2012/images" \
            --bbox_file "./data/VOC2012/multi_region_bboxes/fixed/bboxes_e2_d5.pth" \
            --output_file "./data/VOC2012/multi_region_bboxes/fixed/bbox_features_e2_d5.pth" \
    """
    from PIL import Image
    bbox_list = torch.load(bbox_file, weights_only=False)
    total_num_boxes = sum(len(d["bboxes"]) for d in bbox_list)
    print(f"Loaded bounding box list. There are {total_num_boxes} total bounding boxes.")
    dev = _device()
    model, _, patch_size, _ = utils.get_model(model_name.lower(), checkpoint=checkpoint, seed=seed, device=dev,
                                              random_init=random_init)
    feats: Dict[Tuple[int, int], torch.Tensor] = {}   # (image row, box row) -> [d]

    def flush(shape_key, items):
        batch = torch.stack([it[0] for it in items]).to(dev)
        cls = model.forward_cls(batch).cpu()
        for j, (_, where) in enumerate(items):
            feats[where] = cls[j].clone()

    batcher = _Batcher(batch_size, flush)
    for bi, bbox_dict in enumerate(bbox_list):
        image_filename = str(Path(images_root) / f"{bbox_dict['id']}.jpg")
        image = torch.from_numpy(np.ascontiguousarray(np.asarray(Image.open(image_filename).convert("RGB"))))
        for ji, (xmin, ymin, xmax, ymax) in enumerate(bbox_dict["bboxes_original_resolution"]):
            crop = image[ymin:ymax, xmin:xmax].contiguous()          # image[:, :, ymin:ymax, xmin:xmax] at :539
            if crop.shape[0] < patch_size or crop.shape[1] < patch_size:
                raise ValueError(f"{bbox_dict['id']}: box {(xmin, ymin, xmax, ymax)} is smaller than one patch")
            batcher.add((int(crop.shape[0]), int(crop.shape[1])), (crop, (bi, ji)))
    batcher.finish()
    for bi, bbox_dict in enumerate(bbox_list):
        bbox_dict["features"] = torch.stack([feats[(bi, ji)] for ji in range(len(bbox_dict["bboxes"]))], dim=0)
    torch.save(bbox_list, output_file)
    print(f"Saved features to {output_file}")


# ---------------------------------------------------------------------------------------------------------------
def extract_all(images_list: str, images_root: Optional[str], model_name: str, features_dir: Optional[str],
                eigs_dir: str, K: int = 20, batch_size: int = 64, which_block: int = -1, normalize: bool = True,
                threshold_at_zero: bool = True, lapnorm: bool = True, image_color_lambda: float = 0.0,
                which_color_matrix: str = "knn", checkpoint: Optional[str] = None, seed: Optional[int] = None,
                random_init: bool = False, yes: Optional[bool] = None, single_region_dir: Optional[str] = None,
                multi_region_dir: Optional[str] = None, non_adaptive_num_segments: int = 4, adaptive: bool = False,
                infer_bg_index: bool = True, threshold: float = 0.0, num_workers: Optional[int] = None,
                num_workers_out: int = 4, writer: str = "process"):
    """Fused extract_features + extract_eigs (+ the two segmentation commands): features and eigenvectors never leave
    the GPU between the stages. Writes the eigs files and, if the directories are given, the features files and the
    single- / multi-region segmentation PNGs, all in the reference's layouts. Decoding, pinned staging and the file
    writers run on threads (io_pipeline.py)."""
    for dname in (features_dir, eigs_dir, single_region_dir, multi_region_dir):
        if dname:
            utils.make_output_dir(dname, assume_yes=yes)
    wr = io_pipeline.make_writer(writer, num_workers_out)   # first: writer processes import torch while the model is set up
    model_name = model_name.lower()
    _check_supported("laplacian", which_color_matrix, image_color_lambda)
    dev = _device()
    model, _, patch_size, _ = utils.get_model(model_name, checkpoint=checkpoint, seed=seed, device=dev,
                                              random_init=random_init)
    filenames = Path(images_list).read_text().splitlines()
    dataset = utils.ImagesDataset(filenames=filenames, images_root=images_root)
    all_failed: List[str] = []
    decode_threads: dict = {}
    import time
    t_start = time.perf_counter()   # model set-up (weights, packing) is done: what follows is the per-image pipeline

    tm = {"decode_wait": 0.0, "pinned_alloc": 0.0, "launch": 0.0, "wait_gpu": 0.0, "submit": 0.0}
    in_flight: List[dict] = []       # batches whose kernels / read-back copies are still running (software pipeline)
    with wr, _png_writer_pool(2) as png_pool:
        def finish(h):
            """Second half of a batch: wait for its read-back, retry stragglers, hand everything to the writers."""
            ta = time.perf_counter()
            h["event"].synchronize()
            assembler.release(h["batch"])     # its host->device copy is long done: the decode threads may refill it
            tb = time.perf_counter()
            items, H, W, Hp, Wp = h["items"], h["H"], h["W"], h["Hp"], h["Wp"]
            evals, evecs, info = h["evals"], h["evecs"], h["info"]
            n_img = len(items)
            bad = _bad_rows(evals, evecs, info)
            failed = []
            if bad:   # rare: largest possible Krylov space for the images that did not reach the tolerance
                ev2, vec2, info2 = (t.cpu() for t in h["solve"](bad, max(Hp * Wp - 1, 1)))
                for j, i in enumerate(bad):
                    if int(info2[j, 1]) == 1 and bool(torch.isfinite(vec2[j]).all()):
                        evals[i], evecs[i] = ev2[j], vec2[j]
                    else:
                        failed.append(i)
            all_failed.extend(items[j][1] for j in failed)
            if features_dir:
                wr.submit_batch({"k": h["k"].numpy()}, [it_ for j, it_ in enumerate(_feature_items(
                    features_dir, [(it[1], it[2]) for it in items], model_name, patch_size, H, W)) if j not in failed])
            wr.submit_batch({"evals": evals.numpy(), "evecs": evecs.numpy()},
                            _eigs_items(eigs_dir, [it[1][:-4] for it in items], skip=failed))
            for j, (_, file, index) in enumerate(items):
                if j in failed:
                    continue
                if h["masks"] is not None:
                    png_pool.submit(_save_png, h["masks"][j].numpy().reshape(Hp, Wp).copy(),
                                    str(Path(single_region_dir) / f"{Path(file).stem}.png"))
                if h["labels"] is not None:
                    png_pool.submit(_save_png, h["labels"][j].numpy().reshape(Hp, Wp).copy(),
                                    str(Path(multi_region_dir) / f"{Path(file).stem}.png"))
            tm["wait_gpu"] += tb - ta
            tm["submit"] += time.perf_counter() - tb

        def flush(batch):
            """First half of a batch: start the H2D copy of the page-locked batch the decode threads filled, enqueue every
            kernel and the read-back copies; then finish the PREVIOUS batch while this one runs."""
            H, W = batch.key
            tb = time.perf_counter()
            items = [(None, file, index) for file, index in batch.items]
            host = batch.host[:len(items)]
            k = model.forward_k(host.to(dev, non_blocking=True), which_block=which_block)
            Hp, Wp = H // patch_size, W // patch_size
            rgb_lr, lr_size = None, None
            if image_color_lambda > 0:
                rgb_lr = _color_inputs(images_root, [it[1][:-4] for it in items], Wp, Hp, which_color_matrix, dev)
                lr_size = (Hp, Wp)

            def solve(sel, max_steps):
                f = k if sel is None else k[sel]
                rgb = rgb_lr if (sel is None or rgb_lr is None) else rgb_lr[sel]
                return spectral.laplacian_eigs(f, K, normalize, threshold_at_zero, lapnorm, rgb, lr_size, image_color_lambda,
                                               max_steps=max_steps, which_color_matrix=which_color_matrix)[:3]
            evals_d, evecs_d, info_d = solve(None, 0)
            masks_d = labels_d = None
            if single_region_dir:
                masks_d = segment.threshold_masks(evecs_d, threshold, which=1)
            if multi_region_dir:
                if adaptive:   # the per-image cluster count comes from the eigenvalues (host arithmetic on K numbers)
                    ks = [segment.adaptive_num_clusters(e.numpy()) for e in evals_d.cpu()]
                else:
                    ks = [non_adaptive_num_segments] * len(items)
                labels_d = segment.kmeans_labels(evecs_d[:, 1:], ks, (Hp, Wp), infer_bg_index,
                                                 image_keys=[it[2] for it in items])[0]

            def to_host(t):
                if t is None:
                    return None
                h_ = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
                h_.copy_(t, non_blocking=True)
                return h_
            h = {"items": items, "H": H, "W": W, "Hp": Hp, "Wp": Wp, "solve": solve, "evals": to_host(evals_d),
                 "evecs": to_host(evecs_d), "info": to_host(info_d), "masks": to_host(masks_d), "labels": to_host(labels_d),
                 "k": to_host(k) if features_dir else None, "keep": (k, evals_d, evecs_d, info_d, masks_d, labels_d),
                 "batch": batch}
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(dev))
            h["event"] = ev
            tm["launch"] += time.perf_counter() - tb
            in_flight.append(h)
            while len(in_flight) > 1:
                finish(in_flight.pop(0))

        todo = []
        for i in _my_share(list(range(len(dataset)))):
            file = dataset.filenames[i]
            if (Path(eigs_dir) / f"{file[:-4]}.pth").is_file():
                print(f"Skipping existing file {str(Path(eigs_dir) / (file[:-4] + '.pth'))}")
            else:
                todo.append(i)
        # The decode threads group the images by shape and write them straight into page-locked batches
        # (io_pipeline.BatchAssembler); this thread only sees completed batches.
        if dataset.transform is None:
            load = dataset.load_raw
        else:
            def load(i):
                image, file, index = dataset[i]
                return image.numpy(), False, file, index
        assembler = io_pipeline.BatchAssembler(load, todo, max(1, int(batch_size)), num_workers)
        it = iter(assembler)
        while True:
            ta = time.perf_counter()
            batch = next(it, None)
            tm["decode_wait"] += time.perf_counter() - ta
            if batch is None:
                break
            flush(batch)
        tm["pinned_alloc"] = assembler.alloc_seconds
        decode_threads = {k_: round(v_, 3) for k_, v_ in assembler.worker_seconds.items()}
        decode_threads["threads"] = len(assembler.threads)
        if assembler.trace is not None:
            decode_threads["trace"] = [(round(t_ - t_start, 4), ev_, d_) for t_, ev_, d_ in sorted(assembler.trace)]
        while in_flight:
            finish(in_flight.pop(0))
    seconds = time.perf_counter() - t_start
    print(f"Saved eigs to {eigs_dir} ({len(todo)} images in {seconds:.2f}s after model set-up: "
          f"{len(todo) / max(seconds, 1e-9):.0f} images/s incl. decode and file writes; main thread: "
          + ", ".join(f"{k_} {v_:.2f}s" for k_, v_ in tm.items()) + ")")
    if all_failed:
        raise _lib.DssError(f"eigensolver did not converge for {len(all_failed)} image(s): {all_failed[:8]}")
    return {"images": len(todo), "seconds": seconds, "images_per_s": len(todo) / max(seconds, 1e-9),
            "decode_thread_seconds_summed": decode_threads,
            "main_thread_seconds": {"waiting_for_decoders": tm["decode_wait"],
                                    "pinned_alloc_in_decoders": tm["pinned_alloc"], "kernel_launches": tm["launch"],
                                    "waiting_for_gpu": tm["wait_gpu"], "writer_submit": tm["submit"], "total": seconds}}
