"""Batched end-to-end driver of the hot path: uint8 images -> K features -> affinity -> eigenvectors.

Used by bench.py and the multi-GPU launcher. Images are the only parallel axis of this workload
(SURVEY 8e): ranks take a strided shard of the image list, the DINO weights are broadcast once from rank 0, and no
other collective exists on the data path."""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch

from . import _lib, spectral
from .vit import DinoViT, flat_param_order, random_state_dict


def shard_indices(n_items: int, rank: int, world_size: int) -> List[int]:
    """Rank r of R processes items r, r+R, r+2R, ... of the sorted, de-duplicated list (balances VOC-shaped sizes)."""
    if not (0 <= rank < world_size):
        raise ValueError(f"rank {rank} outside world of {world_size}")
    return list(range(rank, n_items, world_size))


def flatten_state_dict(sd: Dict[str, torch.Tensor], name: str, device=None) -> torch.Tensor:
    keys = flat_param_order(name)
    return torch.cat([sd[k].detach().reshape(-1).to(torch.float32) for k in keys]).to(device or "cpu").contiguous()


def unflatten_state_dict(flat: torch.Tensor, like: Dict[str, torch.Tensor], name: str) -> Dict[str, torch.Tensor]:
    out, off = {}, 0
    for k in flat_param_order(name):
        n = like[k].numel()
        out[k] = flat[off:off + n].view_as(like[k]).clone()
        off += n
    assert off == flat.numel()
    return out


def broadcast_weights(name: str, seed: int = 0, device=None, src: int = 0, state_dict=None) -> Dict[str, torch.Tensor]:
    """The one collective of the path: rank `src` materialises the DINO weights, everyone else receives them in a
    single broadcast of one flat fp32 buffer (86 MB for ViT-S, 341 MB for ViT-B) over NCCL (NVLink) or gloo (CPU tests)."""
    import torch.distributed as dist
    template = random_state_dict(name, seed)  # shapes only on non-src ranks
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return state_dict if state_dict is not None else template
    rank = dist.get_rank()
    if rank == src:
        flat = flatten_state_dict(state_dict if state_dict is not None else template, name, device)
    else:
        n = sum(template[k].numel() for k in flat_param_order(name))
        flat = torch.empty(n, dtype=torch.float32, device=device or "cpu")
    dist.broadcast(flat, src=src)
    return unflatten_state_dict(flat, template, name)


class SpectralPipeline:
    """images_u8 -> (eigenvalues [B,K], eigenvectors [B,K,N]) for which_matrix='laplacian' (extract.py:175-240)."""

    def __init__(self, model_name: str = "dino_vits16", K: int = 5, device="cuda", state_dict=None, seed: int = 0,
                 vit_batch: int = 32, which_block: int = -1, normalize=True, threshold_at_zero=True, lapnorm=True,
                 tol: float = 0.0, max_steps: int = 0, model: Optional[DinoViT] = None):
        self.device = torch.device(device)
        # ``model``: share one weight handle between several pipelines (one per image shape: buffers are per pipeline)
        self.model = model if model is not None else DinoViT(
            model_name, state_dict if state_dict is not None else random_state_dict(model_name, seed), device=self.device)
        self.K, self.vit_batch, self.which_block = K, vit_batch, which_block
        self.normalize, self.threshold_at_zero, self.lapnorm = normalize, threshold_at_zero, lapnorm
        self.tol, self.max_steps = tol, max_steps
        self._copy_stream = torch.cuda.Stream(self.device)
        self._bufs: dict = {}

    def _buf(self, key, shape, dtype, pinned=False):
        b = self._bufs.get(key)
        if b is None or tuple(b.shape) != tuple(shape):
            b = (torch.empty(shape, dtype=dtype).pin_memory() if pinned
                 else torch.empty(shape, dtype=dtype, device=self.device))
            self._bufs[key] = b
        return b

    @torch.no_grad()
    def run_device(self, images_u8: torch.Tensor, events: Optional[list] = None, slot: int = 0):
        """images_u8 [B,H,W,3] already in HBM. `events[i]` (optional) gates ViT sub-batch i on its H2D copy. ``slot``
        selects one of the feature buffers (the streaming driver alternates two so that the D2H copy of one batch's
        features overlaps the next batch's compute)."""
        B, H, W, _ = images_u8.shape
        P, d = self.model.patch_size, self.model.dim
        N = (H // P) * (W // P)
        feats = self._buf(("feats", slot), (B, N, d), torch.float32)
        self._bufs["feats"] = feats   # most recent features (parity checks read them)
        vb = self.vit_batch
        for i, s in enumerate(range(0, B, vb)):
            if events is not None:
                torch.cuda.current_stream(self.device).wait_event(events[i])
            self.model.forward_k(images_u8[s:s + vb], which_block=self.which_block, out=feats[s:s + vb])
        Wm = self._buf("W", (B, N, spectral.pitch(N)), torch.float32)
        deg = self._buf("deg", (B, N), torch.float32)
        spectral.affinity(feats, self.normalize, self.threshold_at_zero, out=Wm, degree=deg)
        evals, evecs, info, resid = spectral.eigsh_laplacian(Wm, N, self.K, self.lapnorm, self.tol, self.max_steps,
                                                             degree=deg)
        return evals, evecs, info

    @torch.no_grad()
    def run_host(self, images_u8_host: torch.Tensor):
        """Public end-to-end call: HOST uint8 images [B,H,W,3] (pinned for async copies) -> host (eigenvalues,
        eigenvectors, info). H2D copies are chunked on a side stream so they overlap the ViT of earlier chunks."""
        assert not images_u8_host.is_cuda and images_u8_host.dtype == torch.uint8
        B = images_u8_host.shape[0]
        dev_imgs = self._buf("imgs", tuple(images_u8_host.shape), torch.uint8)
        events = []
        cur = torch.cuda.current_stream(self.device)
        self._copy_stream.wait_stream(cur)  # previous users of dev_imgs are done
        with torch.cuda.stream(self._copy_stream):
            for s in range(0, B, self.vit_batch):
                dev_imgs[s:s + self.vit_batch].copy_(images_u8_host[s:s + self.vit_batch], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self._copy_stream)
                events.append(ev)
        evals, evecs, info = self.run_device(dev_imgs, events)
        h_evals = self._buf("h_evals", tuple(evals.shape), torch.float32, pinned=True)
        h_evecs = self._buf("h_evecs", tuple(evecs.shape), torch.float32, pinned=True)
        h_info = self._buf("h_info", tuple(info.shape), torch.int32, pinned=True)
        h_evals.copy_(evals, non_blocking=True)
        h_evecs.copy_(evecs, non_blocking=True)
        h_info.copy_(info, non_blocking=True)
        cur.synchronize()
        return h_evals, h_evecs, h_info

    @torch.no_grad()
    def run_host_pipelined(self, batches, copy_chunk: int = 32, features: bool = False):
        """Streaming form of run_host for a sequence of equally shaped HOST batches: the H2D copy of batch i+1 runs
        on the copy stream while batch i is being computed, and the D2H copies of batch i (on a third stream) complete
        while batch i+1 runs. Yields (eigenvalues, eigenvectors, info[, features]) per batch, in order; the yielded
        tensors are pinned buffers that stay valid until two further batches have been submitted. ``features=True``
        also brings the K features [B, N, d] back (what extract_features writes to features/*.pth)."""
        cur = torch.cuda.current_stream(self.device)
        if not hasattr(self, "_d2h_stream"):
            self._d2h_stream = torch.cuda.Stream(self.device)
        done = [None, None]      # per slot: event recorded after the D2H of the batch that used the slot
        keep = [None, None]      # per slot: device outputs kept alive until their D2H has completed
        pending = None           # (slot, outputs) of the previous batch
        for i, hb in enumerate(batches):
            assert not hb.is_cuda and hb.dtype == torch.uint8
            slot = i & 1
            B = hb.shape[0]
            dev_imgs = self._buf(("imgs", slot), tuple(hb.shape), torch.uint8)
            if done[slot] is not None:
                # the batch that used this slot two steps ago has been read back: its image / feature buffers are free
                self._copy_stream.wait_event(done[slot])
                cur.wait_event(done[slot])
            vb = self.vit_batch
            events = []
            with torch.cuda.stream(self._copy_stream):
                for s in range(0, B, vb):
                    for c in range(s, min(s + vb, B), copy_chunk):
                        e = min(c + copy_chunk, s + vb, B)
                        dev_imgs[c:e].copy_(hb[c:e], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(self._copy_stream)
                    events.append(ev)
            evals, evecs, info = self.run_device(dev_imgs, events, slot=slot)
            feats = self._bufs[("feats", slot)]
            computed = torch.cuda.Event()
            computed.record(cur)
            outs = [self._buf(("h_evals", slot), tuple(evals.shape), torch.float32, pinned=True),
                    self._buf(("h_evecs", slot), tuple(evecs.shape), torch.float32, pinned=True),
                    self._buf(("h_info", slot), tuple(info.shape), torch.int32, pinned=True)]
            if features:
                outs.append(self._buf(("h_feats", slot), tuple(feats.shape), torch.float32, pinned=True))
            with torch.cuda.stream(self._d2h_stream):
                self._d2h_stream.wait_event(computed)
                outs[0].copy_(evals, non_blocking=True)
                outs[1].copy_(evecs, non_blocking=True)
                outs[2].copy_(info, non_blocking=True)
                if features:
                    outs[3].copy_(feats, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self._d2h_stream)
            done[slot] = ev
            keep[slot] = (evals, evecs, info)
            if pending is not None:
                done[pending[0]].synchronize()
                yield tuple(pending[1])
            pending = (slot, outs)
        if pending is not None:
            done[pending[0]].synchronize()
            yield tuple(pending[1])
        cur.wait_stream(self._d2h_stream)

    @staticmethod
    def launches_per_call(depth: int, which_block: int, n_vit_batches: int) -> int:
        """Kernels libdss_b200 launches for one run_device call (cross-checked against dss_kernel_launch_count)."""
        blk = which_block % depth
        vit = 3 + 7 * blk + 2
        return n_vit_batches * vit + 3 + 1   # rownorm/split, affinity GEMM, degree reduce; eigensolver
