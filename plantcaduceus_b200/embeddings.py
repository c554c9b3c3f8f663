"""Embedding extraction on the B200 engine -- the model-facing half of the reference's ``src/train_XGBoost.py``
(``extract_embeddings``, :96-114): the final hidden state at ``tokenIdx`` of every window, forward and reverse-complement
halves averaged as ``(fwd + rev[..., ::-1]) / 2``.  The XGBoost classifier around it is CPU post-processing and stays with
the caller.

The reference materialises ``hidden_states[-1]`` ([B, L, 2d]) to read one position; here ``pcad_hidden_at`` taps the
requested position(s) only, windows travel as ASCII bytes and are tokenised with the byte LUT (the reference's dataset for
this script does NOT mask ``tokenIdx``: the embedding is taken from the unmasked window).
"""
from __future__ import annotations

import numbers
from typing import Sequence, Union

import numpy as np
import torch


def average_strands(embeddings: np.ndarray) -> np.ndarray:
    """``(forward + reverse[..., ::-1]) / 2`` over the last axis split in two (train_XGBoost.py:108-113)."""
    hidden_size = embeddings.shape[-1] // 2
    forward = embeddings[..., 0:hidden_size]
    reverse = embeddings[..., hidden_size:][..., ::-1]
    return (forward + reverse) / 2


def extract_embeddings(model, tokenizer, sequences: Union[Sequence[str], np.ndarray], tokenIdx: int = 255,
                       batch_size: int = 128, average: bool = True, layer: Union[int, Sequence[int]] = -1,
                       pooling: str = "token", ranges=None) -> np.ndarray:
    """float32 [n, d_model] averaged embeddings (or [n, 2*d_model] raw halves with ``average=False``) at ``tokenIdx``.
    ``sequences``: equal-length strings or a uint8 ASCII matrix [n, L].

    ``layer`` indexes the reference's ``hidden_states`` (n_layer + 1 entries; -1, the default, is the final normed state
    the reference takes; 0 the embedding; k the mixer output of layer k-1).  A sequence of indices returns
    [len(layer), n, ...], entry i from hidden_states[layer[i]].  Intermediate entries have the same RCPS layout, so the
    strand average applies to them as is.  The forward stops after the deepest requested layer.

    ``pooling="mean"`` replaces the position ``tokenIdx`` by the mean over each window's positions (``model.hidden_mean``:
    one vector per window and per layer, float32, in a fixed summation order); ``ranges`` ([n, 2] integers (s, e), or
    None for the whole window) restricts window i to positions [s_i, e_i), e.g. a gene body or the part of a window that
    is not N padding.  The states inside a range still see the whole window through the bidirectional scans.  An invalid
    range gives a NaN row.  ``ranges`` needs ``pooling="mean"``."""
    from .modeling import hidden_layer_indices, hidden_mean_ranges   # ValueError for malformed arguments, before any work
    if pooling not in ("token", "mean"):
        raise ValueError(f"pooling must be 'token' or 'mean', not {pooling!r}")
    if ranges is not None and pooling != "mean":
        raise ValueError("ranges apply to pooling='mean' only")
    many = not isinstance(layer, numbers.Integral) or isinstance(layer, bool)
    if many:
        layers = hidden_layer_indices(layer, model.config.n_layer)
    else:
        layers = None if int(layer) == -1 else hidden_layer_indices([layer], model.config.n_layer)   # -1: hidden_at's own path
    if isinstance(sequences, np.ndarray):
        ascii_mat = np.ascontiguousarray(sequences, dtype=np.uint8)
    else:
        seqs = [str(s) for s in sequences]
        ascii_mat = tokenizer.windows_to_ascii(seqs, len(seqs[0])) if seqs else np.zeros((0, 0), dtype=np.uint8)
    n = len(ascii_mat)
    rng = None if ranges is None else hidden_mean_ranges(ranges, n, ascii_mat.shape[1])
    n_out = len(layers) if layers is not None else 1
    out = np.zeros((n_out, n, 2 * model.config.d_model), dtype=np.float32)
    for s in range(0, n, batch_size):
        ids = tokenizer.encode_bytes(ascii_mat[s:s + batch_size])
        if pooling == "mean":
            r = rng[s:s + len(ids)] if rng is not None else None
            h = model.hidden_mean(torch.from_numpy(ids), r, layers=layers)
            out[:, s:s + len(ids)] = (h[None] if layers is None else h).cpu().numpy()
            continue
        pos = torch.full((len(ids), 1), int(tokenIdx), dtype=torch.int32)
        if layers is None:
            h = model.hidden_at(torch.from_numpy(ids), pos)[None, :, 0]
        else:
            h = model.hidden_at(torch.from_numpy(ids), pos, layers=layers)[:, :, 0]
        out[:, s:s + len(ids)] = h.to(torch.float32).cpu().numpy()
    out = out if many else out[0]
    return average_strands(out) if average else out
