"""Flat parameter buffer + gradient bucket of the view-sharded step (SURVEY.md §8e), and the
round-robin view assignment.  Pure torch: shared by the product step (bloomscene_b200/multiview.py)
and the reference arm of bench.py, which must not load the product's native libraries."""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from .synthetic import Scene

_ORDER = ("means3D", "scales", "rotations", "opacities", "shs", "colors_precomp")


class GaussianParams:
    """Gaussian parameters packed in one flat fp32 buffer with a matching flat gradient bucket.

    Each parameter tensor is a leaf view into `flat`, and its `.grad` is preset to the matching view
    of `grad_bucket`, so every view's gradients land straight in the bucket (added by the kernel itself
    with the native rasterizer, by autograd otherwise) and a single allreduce covers all parameters
    ((44 + 12 M) bytes per Gaussian, SURVEY.md §8e).

    `densify_stats=True` adds 2 P words to the all-reduced buffer, between the gradients and the loss / flag words:
    `densify = {"grad_norm": [P], "count": [P]}`, the step's densification statistics (sum over this step's views
    of |means2D.grad[i, :2]| and the number of views with radii[i] > 0).  They ride in the step's one all-reduce and
    are cleared by `zero_grad()` like the gradients: per step, not running totals (a running total would be
    multiplied by the world size at the next all-reduce), so callers add them into their own accumulators."""

    def __init__(self, scene: Scene, densify_stats: bool = False):
        tensors = {k: v for k, v in scene.tensors().items()}
        self.names = [n for n in _ORDER if n in tensors]
        self.sh_degree = scene.sh_degree
        dev = scene.means3D.device
        sizes = [tensors[n].numel() for n in self.names]
        G = sum(sizes)
        S = 2 * tensors["means3D"].shape[0] if densify_stats else 0
        self.flat = torch.empty(G, dtype=torch.float32, device=dev)
        # two extra words behind the gradients (and the statistics) carry the step loss and a "some rank must repeat
        # this step" count, so that a multi-rank step needs ONE collective
        self._bucket_ext = torch.zeros(G + S + 2, dtype=torch.float32, device=dev)
        self.grad_bucket = self._bucket_ext[:G]
        self.densify = ({"grad_norm": self._bucket_ext[G:G + S // 2], "count": self._bucket_ext[G + S // 2:G + S]}
                        if densify_stats else None)
        self.loss_slot = self._bucket_ext[G + S:G + S + 1]
        self.flag_slot = self._bucket_ext[G + S + 1:]
        self.tensors: Dict[str, torch.Tensor] = {}
        self._zero_means2D = None
        off = 0
        for n, sz in zip(self.names, sizes):
            seg = self.flat[off:off + sz].view(tensors[n].shape)
            seg.copy_(tensors[n])
            seg.requires_grad_(True)
            seg.grad = self.grad_bucket[off:off + sz].view(tensors[n].shape)
            self.tensors[n] = seg
            off += sz

    @property
    def P(self) -> int:
        return self.tensors["means3D"].shape[0]

    def zero_grad(self):
        self._bucket_ext.zero_()

    def reduce_buffer(self) -> torch.Tensor:
        """What a multi-rank step all-reduces: the gradient bucket, the densification statistics if any, then the loss
        and the repeat-flag words."""
        return self._bucket_ext

    def zero_means2D(self) -> torch.Tensor:
        """The all-zero `means2D` input every view passes in (reference gaussian_renderer/__init__.py:224-229
        creates a fresh zeros_like per call); it is only a gradient carrier, so one buffer serves all views."""
        if self._zero_means2D is None:
            self._zero_means2D = torch.zeros_like(self.tensors["means3D"].detach())
        return self._zero_means2D

    def grads(self) -> Dict[str, torch.Tensor]:
        return {n: t.grad for n, t in self.tensors.items()}

    def get(self, name: str) -> Optional[torch.Tensor]:
        return self.tensors.get(name)


def shard_views(n_views: int, rank: int, world: int) -> List[int]:
    """Round-robin view assignment: rank r renders views r, r+N, r+2N, ..."""
    return list(range(rank, n_views, world))
