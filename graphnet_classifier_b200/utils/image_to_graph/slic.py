"""Device SLIC (csrc/slic.cu): the segmentation stage of the superpixel builder.

The reference calls ``skimage.segmentation.slic(img, n_segments, compactness, start_label=0)``
(reference image_to_graph_superpixel.py:31).  scikit-image is un-vendored, unpinned and absent
here, so label parity is UNPINNED; this follows the published SLIC algorithm with
scikit-image's conventions (Lab colour space, colour / compactness, 10 iterations).
"""
from __future__ import annotations

import torch
from torch import Tensor

from ... import _lib
from ..._lib import check
from ...ops import _require_cuda, _stream, _workspace


def enforce_connectivity(labels: Tensor, min_size: int) -> Tensor:
    """scikit-image's default SLIC post-pass on int32 label maps ``[B, H, W]``: connected components of equal labels,
    components smaller than ``min_size`` dissolved into a neighbour, survivors renumbered in scan order (the exact rule:
    csrc/slic_connect.cu; parity unpinned)."""
    _require_cuda(labels)
    lab = labels if labels.dim() == 3 else labels.unsqueeze(0)
    lab = lab.to(torch.int32).contiguous()
    B, H, W = lab.shape
    lib = _lib.load()
    out = torch.empty_like(lab)
    n_work = int(lib.gnc_slic_connectivity_workspace(B, H, W))
    work = _workspace(lab.device, n_work, torch.int32)
    check(lib.gnc_slic_enforce_connectivity(lab.data_ptr(), B, H, W, int(min_size), out.data_ptr(), None, work.data_ptr(),
                                            n_work, _stream()), "slic_enforce_connectivity")
    return out


def connectivity_min_size(H: int, W: int, n_segments: int, min_size_factor: float = 0.5) -> int:
    """``min_size`` of the connectivity post-pass of ``slic_labels``: ``int(min_size_factor * H * W / n_centres)``."""
    n_centres = int(_lib.load().gnc_slic_num_centers(int(H), int(W), int(n_segments)))
    return int(min_size_factor * H * W / max(n_centres, 1))


def slic_labels(images: Tensor, n_segments: int = 100, compactness: float = 10.0, max_num_iter: int = 10,
                enforce_connectivity_: bool = True, min_size_factor: float = 0.5) -> Tensor:
    """uint8 ``[B, H, W, 3]`` (or ``[H, W, 3]``) on the device -> int32 labels ``[B, H, W]``.  As scikit-image's
    ``slic`` does by default, the k-means labels go through the connectivity post-pass with
    ``min_size = int(min_size_factor * H * W / n_centres)``."""
    img = images if images.dim() == 4 else images.unsqueeze(0)
    _require_cuda(img)
    if img.dtype != torch.uint8 or img.shape[-1] != 3:
        raise TypeError("slic_labels expects uint8 [B, H, W, 3]")
    img = img.contiguous()
    B, H, W, _ = img.shape
    lib = _lib.load()
    labels = torch.empty(B, H, W, dtype=torch.int32, device=img.device)
    nbytes = int(lib.gnc_slic_workspace_bytes(B, H, W, int(n_segments)))
    work = _workspace(img.device, (nbytes + 7) // 8, torch.int64)
    check(lib.gnc_slic_labels_u8(img.data_ptr(), B, H, W, int(n_segments), float(compactness), int(max_num_iter),
                                 labels.data_ptr(), work.data_ptr(), _stream()), "slic_labels")
    if enforce_connectivity_:
        labels = enforce_connectivity(labels, connectivity_min_size(H, W, n_segments, min_size_factor))
    return labels
