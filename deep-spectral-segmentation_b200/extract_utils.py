"""Host utilities of the hot path, under the reference's names (extract/extract_utils.py).

Five-line helpers that ARE the file/CLI contract are kept as the reference has them and say so in their docstrings
(get_image_sizes :73-79, _get_files :82-88, get_paired_input_files :91-95, ImagesDataset.__init__/__len__ :17-24,36-37);
everything with behaviour of its own (decode, get_model, make_output_dir, parallel_process, get_border_fraction) is
written for this package."""
from __future__ import annotations

import sys
import time
from pathlib import Path
from typing import Callable, Iterable, Optional

import numpy as np
import torch

from .vit import get_model  # noqa: F401  (re-exported under the reference's name)


def read_image_raw(path):
    """cv2.imread -> (pixels uint8 (H, W, 3), is_bgr); PIL is the fallback decoder (RGB). The colour swap is left to the
    caller so that it can write the RGB image straight into a page-locked batch row (io_pipeline.BatchAssembler)
    instead of into a temporary that is then copied."""
    try:
        import cv2
        img = cv2.imread(str(path))
        if img is None:
            raise IOError(f"cannot decode {path}")
        return img, True
    except ImportError:
        from PIL import Image
        return np.asarray(Image.open(str(path)).convert("RGB")), False


def read_image_rgb(path) -> np.ndarray:
    """cv2.imread + BGR->RGB (extract_utils.py:30-31) -> uint8 (H, W, 3)."""
    pixels, is_bgr = read_image_raw(path)
    if not is_bgr:
        return pixels
    import cv2
    return cv2.cvtColor(pixels, cv2.COLOR_BGR2RGB)


class ImagesDataset:
    """De-duplicated, sorted list of image files; items are (uint8 RGB HWC tensor, path, index).

    The reference's transform (ToTensor + Normalize) is fused into the device patch-embedding kernel, so items stay
    uint8: 4x fewer bytes over PCIe than the reference's fp32 CHW tensors."""

    def __init__(self, filenames, images_root: Optional[str] = None, transform: Optional[Callable] = None,
                 prepare_filenames: bool = True) -> None:
        # copied from extract_utils.py:18-24 (de-duplicate + sort: the order defines the `indices` field of the .pth files)
        self.root = None if images_root is None else Path(images_root)
        self.filenames = sorted(list(set(filenames))) if prepare_filenames else list(filenames)
        self.transform = transform

    def __getitem__(self, index: int):
        path = self.filenames[index]
        full_path = Path(path) if self.root is None else self.root / path
        assert full_path.is_file(), f"Not a file: {full_path}"
        image = torch.from_numpy(np.ascontiguousarray(read_image_rgb(full_path)))
        if self.transform is not None:
            image = self.transform(image)
        return image, path, index

    def load_raw(self, index: int):
        """(decoded pixels, is_bgr, path, index): __getitem__ without the BGR->RGB pass (see read_image_raw)."""
        path = self.filenames[index]
        full_path = Path(path) if self.root is None else self.root / path
        assert full_path.is_file(), f"Not a file: {full_path}"
        pixels, is_bgr = read_image_raw(full_path)
        return pixels, is_bgr, path, index

    def __len__(self) -> int:
        return len(self.filenames)


def get_image_sizes(data_dict: dict, downsample_factor: Optional[int] = None):
    """Copied from extract_utils.py:73-79 (the arithmetic every consumer of features/*.pth shares: crop to patch
    multiples, B must be 1)."""
    P = data_dict["patch_size"] if downsample_factor is None else downsample_factor
    B, C, H, W = data_dict["shape"]
    assert B == 1, "assumption violated :("
    H_patch, W_patch = H // P, W // P
    H_pad, W_pad = H_patch * P, W_patch * P
    return (B, C, H, W, P, H_patch, W_patch, H_pad, W_pad)


def _get_files(p: str):
    """Copied from extract_utils.py:82-88."""
    if Path(p).is_dir():
        return sorted(Path(p).iterdir())
    elif Path(p).is_file():
        return Path(p).read_text().splitlines()
    else:
        raise ValueError(p)


def get_paired_input_files(path1: str, path2: str):
    """Copied from extract_utils.py:91-95: pairs the sorted entries of two directories (or list files)."""
    files1 = _get_files(path1)
    files2 = _get_files(path2)
    assert len(files1) == len(files2)
    return list(enumerate(zip(files1, files2)))


def make_output_dir(output_dir, check_if_empty=True, assume_yes: Optional[bool] = None):
    """Creates the directory; like the reference it asks before writing into a non-empty one. When stdin is not a
    terminal (batch jobs, tests) or assume_yes is set, it continues without blocking (skip-if-exists makes that safe)."""
    output_dir = Path(output_dir)
    output_dir.mkdir(exist_ok=True, parents=True)
    if check_if_empty and (len(list(output_dir.iterdir())) > 0):
        print(f"Output dir: {str(output_dir)}")
        if assume_yes or (assume_yes is None and not sys.stdin.isatty()):
            print("Output dir already contains files. Continuing (existing outputs are skipped).")
            return
        if input("Output dir already contains files. Continue? (y/n) >> ") != "y":
            sys.exit()


def get_border_fraction(segmap: np.ndarray):
    """extract_utils.py:124-135 restated: per label, its share of the 2(H+W) border cells (corners count twice)."""
    labels = np.unique(segmap)
    counts = {int(v): 0 for v in labels}
    for edge in (segmap[:, 0], segmap[:, -1], segmap[0, :], segmap[-1, :]):
        vals, n = np.unique(edge, return_counts=True)
        for v, c in zip(vals.tolist(), n.tolist()):
            counts[v] += c
    perimeter = 2 * (segmap.shape[0] + segmap.shape[1])
    return np.array(list(counts.keys())), np.array(list(counts.values())) / perimeter


def parallel_process(inputs: Iterable, fn: Callable, multiprocessing: int = 0):
    """Serial driver with the reference's timing print (extract_utils.py:138-148). ``multiprocessing`` is accepted for
    CLI compatibility and ignored with a notice: the GPU path batches images inside each kernel instead of forking
    CPU workers (a forked worker could not share the CUDA context anyway)."""
    if multiprocessing:
        print(f"Note: multiprocessing={multiprocessing} is ignored (images are batched on the GPU, not over CPU workers)")
    start = time.time()
    for inp in inputs:
        fn(inp)
    print(f"Finished in {time.time() - start:.1f}s")
