"""Direct ingestion of the on-disk embedding formats the reference's extraction scripts write (SURVEY.md §8f.1), so the
filter can run on pre-extracted galleries at the N x M scales of BASELINE configs 2-4 without the CNN in the loop.

Formats (paths relative to the reference, face_detection_and_extraction/face_extraction/):
  * ``<image>.pkl``   pickle of a list of ``{"det_score": float, "normed_feature": ndarray[D]}``, one entry per detected
                      face, features already L2-normalised      (extract_and_clean_imdb_wiki_faces.py:149-156)
  * ``data.npy``      ``np.save`` of a list of ``{"image_path", "age", "gender", "feature": ndarray[D]}``
                                                                 (extract_and_clean_imdb_wiki_faces.py:232-252)
  * ``<media>.npy``   ``np.save`` of ONE dict with ``"feature"``: either a single [D] / [1, D] vector
                      (extract_features_from_face_dataset.py:126-140) or the concatenation of all per-face vectors of a
                      video, zero padded to a fixed length (extract_faces_from_dataset.py:352-363) -- pass
                      ``feature_size`` to split it; all-zero padding rows are dropped.

Everything is returned as contiguous float32 ``[n, D]`` plus a provenance list ``(path, index_in_file)`` so that
``best_idx`` / ``keep`` can be mapped back to files.
"""
from __future__ import annotations

import os
import pickle
from typing import Iterable, List, Optional, Sequence, Tuple

import numpy as np

Provenance = List[Tuple[str, int]]


def load_pkl_faces(path: str, min_det_score: Optional[float] = None) -> Tuple[np.ndarray, np.ndarray]:
    """``<image>.pkl`` -> (features [n, D] float32, det_scores [n] float32)."""
    with open(path, "rb") as f:
        faces = pickle.load(f)
    feats = [np.asarray(d["normed_feature"], dtype=np.float32).reshape(-1) for d in faces]
    scores = np.asarray([float(d.get("det_score", 1.0)) for d in faces], dtype=np.float32)
    if not feats:
        return np.zeros((0, 0), dtype=np.float32), scores
    x = np.stack(feats)
    if min_det_score is not None:
        sel = scores >= min_det_score
        x, scores = x[sel], scores[sel]
    return np.ascontiguousarray(x), scores


def load_data_npy(path: str) -> Tuple[np.ndarray, List[dict]]:
    """aggregated ``data.npy`` -> (features [n, D] float32, list of the remaining metadata dicts)."""
    data = np.load(path, allow_pickle=True)
    items = list(data.tolist() if isinstance(data, np.ndarray) else data)
    feats = np.stack([np.asarray(d["feature"], dtype=np.float32).reshape(-1) for d in items]) if items else \
        np.zeros((0, 0), dtype=np.float32)
    meta = [{k: v for k, v in d.items() if k != "feature"} for d in items]
    return np.ascontiguousarray(feats), meta


def load_media_npy(path: str, feature_size: Optional[int] = None) -> Tuple[np.ndarray, dict]:
    """per-media ``.npy`` -> (features [k, D] float32, the remaining annotation dict)."""
    d = np.load(path, allow_pickle=True).item()
    feat = np.asarray(d["feature"], dtype=np.float32)
    if feature_size is None:
        feature_size = feat.shape[-1] if feat.ndim > 1 else feat.size
    if feat.size % feature_size != 0:
        raise ValueError(f"{path}: feature of size {feat.size} is not a multiple of feature_size {feature_size}")
    x = feat.reshape(-1, feature_size)
    x = x[np.any(x != 0, axis=1)]                           # zero padding of short videos
    return np.ascontiguousarray(x), {k: v for k, v in d.items() if k != "feature"}


def load_embeddings(paths: Iterable[str], feature_size: Optional[int] = None) -> Tuple[np.ndarray, Provenance]:
    """Concatenate any mix of the three formats into one [n, D] float32 matrix."""
    mats, prov = [], []
    for p in paths:
        if p.endswith(".pkl"):
            x, _ = load_pkl_faces(p)
        elif os.path.basename(p) == "data.npy":
            x, _ = load_data_npy(p)
        elif p.endswith(".npy"):
            x, _ = load_media_npy(p, feature_size)
        else:
            raise ValueError(f"unknown embedding file type: {p}")
        if x.shape[0]:
            mats.append(x)
            prov += [(p, i) for i in range(x.shape[0])]
    if not mats:
        return np.zeros((0, 0), dtype=np.float32), prov
    dims = {m.shape[1] for m in mats}
    if len(dims) != 1:
        raise ValueError(f"mixed embedding sizes {sorted(dims)}")
    return np.ascontiguousarray(np.concatenate(mats, axis=0)), prov


def filter_embedding_files(ref_paths: Sequence[str], cand_paths: Sequence[str], thr: float, metric: str = "cosine",
                           feature_size: Optional[int] = None, device: int = 0, chunk_cand: int = 1 << 18):
    """Gallery filter straight from files: every candidate embedding against all reference embeddings on the GPU
    (host-buffer pipeline, candidates streamed in chunks).  Returns (keep, best_idx, best_val, cand_prov, ref_prov)."""
    from . import ops
    ref, ref_prov = load_embeddings(ref_paths, feature_size)
    cand, cand_prov = load_embeddings(cand_paths, feature_size)
    if ref.shape[0] == 0:
        raise ValueError("no reference embeddings found")
    if cand.shape[0] and cand.shape[1] != ref.shape[1]:
        raise ValueError(f"candidate embeddings are {cand.shape[1]}-d, references {ref.shape[1]}-d")
    hf = ops.HostFilter(device=device, max_ref=ref.shape[0], chunk_cand=max(1, min(chunk_cand, max(cand.shape[0], 1))),
                        max_dim=ref.shape[1])
    try:
        keep, idx, val = hf(ref, cand.reshape(-1, ref.shape[1]), thr, metric=metric)
    finally:
        hf.close()
    return keep, idx, val, cand_prov, ref_prov


def group_embedding_files(paths: Sequence[str], thr: float, metric: str = "cosine", feature_size: Optional[int] = None,
                          device: int = 0):
    """Near-duplicate groups straight from files (the cleaner's ``.pkl`` / ``data.npy`` / media ``.npy`` output): all embeddings
    of ``paths`` are loaded into one set and grouped on the GPU (``ops.self_groups``).  Returns (labels int32 [n] NumPy, the
    number of groups, provenance): ``labels[k]`` is the smallest row of row k's group, and ``prov[k]`` / ``prov[labels[k]]``
    name the file and the index in it of row k and of its group's first occurrence."""
    import torch

    from . import ops
    x, prov = load_embeddings(paths, feature_size)
    if x.shape[0] == 0:
        raise ValueError("no embeddings found")
    res = ops.self_groups(torch.from_numpy(x).to(torch.device("cuda", device)), thr, metric=metric)
    return res.labels.cpu().numpy(), res.n_groups, prov
