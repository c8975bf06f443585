"""Ragged batches: point clouds of different sizes in one batched call (model.vcrnet_model.vcrnetIterRagged).

A ragged batch is a padded tensor [B, 3, N_max] plus int32 lengths [B] on the device: cloud b is x[b, :, :lengths[b]].
The kernels read the lengths on the device only and clamp them into range; this module builds such batches and checks
the lengths on the host.
"""
from __future__ import annotations

import torch

# the kNN graphs of LPDNet rank k + 1 = 21 candidates per point (rank 0 is the point itself)
MIN_POINTS = 21


def check_lengths(lengths, n_max: int):
    """Raise ValueError unless every length is in [MIN_POINTS, n_max]."""
    ls = [int(n) for n in (lengths.tolist() if isinstance(lengths, torch.Tensor) else lengths)]
    bad = [n for n in ls if not MIN_POINTS <= n <= n_max]
    if bad:
        raise ValueError(f"ragged batch: cloud lengths must be in [{MIN_POINTS}, {n_max}], got {bad}")


def pad_clouds(clouds, n_max: int | None = None, device=None):
    """List of [3, N_b] clouds -> (padded fp32 [B, 3, N_max] with zero padding, lengths int32 [B]), both on ``device``
    (default: the first cloud's device, which must then be a CUDA device).  ``n_max`` defaults to the longest cloud."""
    if len(clouds) == 0:
        raise ValueError("ragged batch: no clouds")
    for c in clouds:
        if c.dim() != 2 or c.shape[0] != 3:
            raise ValueError(f"ragged batch: every cloud must be [3, N], got {tuple(c.shape)}")
    lengths = [int(c.shape[1]) for c in clouds]
    n_max = max(lengths) if n_max is None else int(n_max)
    check_lengths(lengths, n_max)
    device = torch.device(device) if device is not None else clouds[0].device
    if device.type != "cuda":
        raise ValueError("ragged batch: the padded batch must live on a CUDA device")
    out = torch.zeros((len(clouds), 3, n_max), dtype=torch.float32, device=device)
    for b, c in enumerate(clouds):
        out[b, :, :lengths[b]].copy_(c)
    return out, torch.tensor(lengths, dtype=torch.int32, device=device)


# Per-pair counts of the partial path (model/transformer.py:41, model/vcrnet_model.py:200-201, :283), evaluated on the
# device with Python's arithmetic: fp64 products left to right, truncated toward zero.  Each is non-decreasing in n, so
# buffers sized from N_max hold every pair.
def _trunc(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.int32)


def key_counts(nk: torch.Tensor, overlap2: float) -> torch.Tensor:
    """int(nk * overlap2): the keys the partial cross attention keeps."""
    return _trunc(nk.double() * float(overlap2))


def select_counts(n: torch.Tensor, overlap2: float) -> torch.Tensor:
    """int(n * 0.84 * overlap2): the points selectCom keeps of a cloud."""
    return _trunc(n.double() * 0.84 * float(overlap2))


def copair_counts(sel: torch.Tensor, overlap2: float) -> torch.Tensor:
    """int(sel * 0.52 * overlap2): the correspondences getCopair keeps of sel selected sources."""
    return _trunc(sel.double() * 0.52 * float(overlap2))


def corr_lengths(src_len: torch.Tensor, overlap2: float) -> torch.Tensor:
    """int(int(ns * 0.84 * overlap2) * 0.52 * overlap2): the correspondences getCopair keeps of pair b, the valid columns
    of vcrnetIterRaggedPartial's srcK / src_corrK (int32 [B] on the lengths' device)."""
    return copair_counts(select_counts(src_len, overlap2), overlap2)
