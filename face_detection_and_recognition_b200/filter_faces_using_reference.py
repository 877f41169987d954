"""Drop-in replacement for the reference's ``similar_face_filtering/filter_faces_using_reference.py``.

Same entry point, same flags (``--ud --rd --td -m -b -r``), same importable helpers
(``_fix_path_for_globbing``, ``get_class_name_list``, ``read_and_preprocess_img``,
``get_ref_mean_vec_and_thres_from_imgs``), same ``TARGET/{clean,unclean}/<class>/<img>`` output tree and the same
per-class summary line (reference :198-199).  What changes is where the arithmetic runs:

  reference (NumPy, one row at a time)                              here (libffr_b200.so, sm_100a)
  ---------------------------------------------------------------   --------------------------------------------
  np.mean / max_i np.linalg.norm(mu - ref_i)          :85-99         ffr_ref_mean_and_thres        (K5)
  np.linalg.norm(out - mu) <= thres per row           :186-189       ffr_filter metric=euclid N=1  (K2s, fp32)
  (new) gallery mode: all reference embeddings, cosine + threshold   ffr_filter metric=cosine      (K1+K2+K3, tcgen05)
  (new) gallery mode, --metric euclid: smallest distance <= threshold ffr_filter metric=euclid     (K1+K2+K3, tcgen05)

Embedding extraction stays in the reference's own PyTorch ``MobileFaceNet`` (imported from the reference
checkout, never copied): ``-m`` is reinterpreted as the path of its state dict.  Any object with
``predict(batch, verbose=0) -> np.ndarray[b, D]`` works as ``model`` (the contract of reference :84,184).

Differences from the reference, on purpose: class directories and image files are visited in sorted order (the
reference relies on unsorted ``glob`` order, :75,138-143,168); TensorFlow is not needed.
"""
from __future__ import annotations

import argparse
import glob
import os
import shutil
import sys
from typing import List, Tuple

import numpy as np
import torch

from . import ops

SEED = 42                      # reference :24
np.random.seed(SEED)


def _fix_path_for_globbing(dir: str) -> str:
    """Add * at the end of paths for proper globbing (reference :29-38)."""
    if dir[-1] == '/':
        dir += '*'
    elif dir[-1] != '*':
        dir += '/*'
    return dir


def get_class_name_list(base_dir: str) -> List[str]:
    """Sorted class sub-directory names of ``base_dir`` (reference :41-57)."""
    return [p.split('/')[-1] for p in sorted(glob.glob(_fix_path_for_globbing(base_dir)))]


def read_and_preprocess_img(img_path: str, in_size: Tuple[int, int] = (160, 160),
                            dct_method: str = "INTEGER_FAST") -> torch.Tensor:
    """jpeg -> RGB float32 in [0,1] -> bilinear resize to ``in_size`` -> per-image standardisation
    ``(x - mean) / max(std, 1/sqrt(N))`` (reference :60-68).  Returns an [H, W, 3] float32 CPU tensor.
    ``dct_method`` is accepted for signature compatibility (libjpeg-turbo picks its own DCT here)."""
    from PIL import Image
    with Image.open(img_path) as im:
        arr = np.asarray(im.convert("RGB"), dtype=np.uint8)
    img = torch.from_numpy(arr.copy()).to(torch.float32).div_(255.0)
    if tuple(img.shape[:2]) != tuple(in_size):
        img = torch.nn.functional.interpolate(img.permute(2, 0, 1)[None], size=tuple(in_size), mode="bilinear",
                                              align_corners=False, antialias=False)[0].permute(1, 2, 0).contiguous()
    n = img.numel()
    mean = img.mean()
    std = img.std(unbiased=False)
    adj = torch.clamp(std, min=1.0 / float(np.sqrt(n)))
    return (img - mean) / adj


class MobileFaceNetModel:
    """``model.predict`` adapter around the REFERENCE's own torch MobileFaceNet
    (face_detection_and_extraction/modules/mobile_facenet/mobile_facenet.py:104-154), imported from
    ``mobilefacenet_dir`` -- the class is not re-implemented here."""

    def __init__(self, weights_path: str, mobilefacenet_dir: str, device: str = "cuda:0", embedding_size: int = 512,
                 allow_random_init: bool = False):
        if not os.path.isfile(os.path.join(mobilefacenet_dir, "mobile_facenet.py")):
            raise FileNotFoundError(
                f"reference MobileFaceNet not found in {mobilefacenet_dir!r}; pass --mobilefacenet_dir or set "
                "FFR_MOBILEFACENET_DIR to <reference>/face_detection_and_extraction/modules/mobile_facenet")
        sys.path.insert(0, mobilefacenet_dir)
        try:
            import mobile_facenet as ref_mfn
        finally:
            sys.path.remove(mobilefacenet_dir)
        self.device = torch.device(device)
        net = ref_mfn.MobileFaceNet(embedding_size)
        if os.path.isfile(weights_path):
            net.load_state_dict(torch.load(weights_path, map_location="cpu"))
        elif not allow_random_init:
            raise FileNotFoundError(f"MobileFaceNet weights {weights_path!r} not found (use --allow_random_init to test)")
        self.net = net.eval().to(self.device)
        self.inputs = "[b, H, W, 3] float32 standardised (resized to 112x112 internally)"
        self.outputs = f"[b, {embedding_size}] float32, unit L2 norm"

    @torch.no_grad()
    def embed(self, img_batch) -> torch.Tensor:
        x = torch.as_tensor(np.asarray(img_batch) if not isinstance(img_batch, torch.Tensor) else img_batch)
        x = x.to(self.device, dtype=torch.float32).permute(0, 3, 1, 2)
        if x.shape[-2:] != (112, 112):
            x = torch.nn.functional.interpolate(x, size=(112, 112), mode="bilinear", align_corners=False)
        return self.net(x)

    def predict(self, img_batch, verbose=0) -> np.ndarray:
        return self.embed(img_batch).float().cpu().numpy()


def _embed_paths(model, paths: List[str], batch_size: int) -> np.ndarray:
    outs = []
    for s in range(0, len(paths), batch_size):
        batch = torch.stack([read_and_preprocess_img(p) for p in paths[s:s + batch_size]]).numpy()
        outs.append(np.asarray(model.predict(batch, verbose=0), dtype=np.float32))
    return np.concatenate(outs, axis=0) if outs else np.zeros((0, 0), dtype=np.float32)


# ---- embedding producer on the GPU (SURVEY §8f row 3) -------------------------------------------------------------
# The reference decodes, resizes and standardises one image at a time on the host (tf.io.decode_jpeg -> tf.image.resize ->
# per_image_standardization, :60-68), embeds the references with batch size 1 (:77-84) and hands every batch to the model
# as a NumPy array (:168-184).  Here a model that can take CUDA tensors (``embed``) is fed from a device-side pipeline:
# file bytes are read by a small thread pool, the whole batch is decoded by nvJPEG in one call
# (torchvision.io.decode_jpeg(device=cuda)), resize + standardisation run on the GPU, the next batch's files are read while
# the model works on the current one, and the embeddings go to the filter without leaving the device.

def preprocess_decoded_device(imgs: List[torch.Tensor], in_size: Tuple[int, int] = (160, 160)) -> torch.Tensor:
    """uint8 [3, H, W] CUDA images (any sizes) -> [B, h, w, 3] float32: [0, 1] scaling, bilinear resize (no antialias,
    half-pixel centres: what tf.image.resize / read_and_preprocess_img do), per-image standardisation
    ``(x - mean) / max(std, 1/sqrt(N))``.  Images of equal size are resized in one call."""
    h, w = in_size
    out = torch.empty((len(imgs), 3, h, w), dtype=torch.float32, device=imgs[0].device)
    groups = {}
    for i, im in enumerate(imgs):
        groups.setdefault(tuple(im.shape[-2:]), []).append(i)
    for shape, idxs in groups.items():
        x = torch.stack([imgs[i] for i in idxs]).to(torch.float32).div_(255.0)
        if shape != (h, w):
            x = torch.nn.functional.interpolate(x, size=(h, w), mode="bilinear", align_corners=False, antialias=False)
        out[torch.as_tensor(idxs, device=out.device)] = x
    n = out[0].numel()
    mean = out.mean(dim=(1, 2, 3), keepdim=True)
    std = out.var(dim=(1, 2, 3), unbiased=False, keepdim=True).sqrt_()
    out = (out - mean) / torch.clamp(std, min=1.0 / float(np.sqrt(n)))
    return out.permute(0, 2, 3, 1).contiguous()


def read_and_preprocess_batch_device(paths: List[str], device: torch.device, in_size: Tuple[int, int] = (160, 160),
                                     datas: List[torch.Tensor] = None) -> torch.Tensor:
    """``read_and_preprocess_img`` for a whole batch on the GPU: one batched nvJPEG decode + GPU resize / standardise.
    ``datas`` = the files' bytes if the caller has already read them (prefetch)."""
    from torchvision.io import ImageReadMode, decode_jpeg, read_file
    if datas is None:
        datas = [read_file(p) for p in paths]
    imgs = decode_jpeg(datas, mode=ImageReadMode.RGB, device=device)
    return preprocess_decoded_device(imgs, in_size)


def _embed_paths_device(model, paths: List[str], batch_size: int, device: torch.device,
                        in_size: Tuple[int, int] = (160, 160), stats: dict = None) -> torch.Tensor:
    """Embeddings as a float32 CUDA tensor.  A model that offers ``embed(batch) -> CUDA tensor`` (MobileFaceNetModel)
    is fed by the device-side pipeline above and its output goes straight into the filter: no PIL, no NumPy round trip
    (the reference goes device -> NumPy -> Python loop per row, :184-189).  Any other model goes through ``predict``
    (the reference's contract).  ``stats`` (optional dict) receives ``{"images", "seconds", "decoder"}``."""
    import time
    t0 = time.perf_counter()
    if not hasattr(model, "embed") or device.type != "cuda":
        out = torch.from_numpy(_embed_paths(model, paths, batch_size)).to(device)
        if stats is not None:
            stats.update(images=len(paths), seconds=time.perf_counter() - t0, decoder="PIL (host)")
        return out
    from concurrent.futures import ThreadPoolExecutor
    from torchvision.io import read_file
    outs = []
    chunks = [paths[s:s + batch_size] for s in range(0, len(paths), batch_size)]
    with ThreadPoolExecutor(max_workers=8) as pool:
        def read_chunk(chunk):
            return list(pool.map(read_file, chunk))
        with ThreadPoolExecutor(max_workers=1) as ahead:         # the NEXT batch's file reads overlap this batch's GPU work
            nxt = ahead.submit(read_chunk, chunks[0]) if chunks else None
            for k, chunk in enumerate(chunks):
                datas = nxt.result()
                nxt = ahead.submit(read_chunk, chunks[k + 1]) if k + 1 < len(chunks) else None
                batch = read_and_preprocess_batch_device(chunk, device, in_size, datas=datas)
                outs.append(model.embed(batch).float())
    out = torch.cat(outs, dim=0) if outs else torch.zeros((0, 0), dtype=torch.float32, device=device)
    if stats is not None:
        torch.cuda.synchronize(device)
        stats.update(images=len(paths), seconds=time.perf_counter() - t0, decoder="nvJPEG (torchvision.io.decode_jpeg, device)")
    return out


def get_ref_mean_vec_and_thres_from_imgs(model, ref_class_path: str,
                                         max_ref_img_count: int = 32) -> Tuple[np.ndarray, np.float32]:
    """Reference :71-100.  Embeds at most ``max_ref_img_count`` reference images one at a time (batch 1, like
    the reference), then mean vector and max distance from it are computed on the GPU (K5).
    Returns (mean (1, D) float32, thres float32) as NumPy, the reference's contract."""
    X_imgs = sorted(glob.glob(ref_class_path + "/*.jpg"))
    ref_num = min(max_ref_img_count, len(X_imgs))
    ref_feat = _embed_paths(model, X_imgs[:ref_num], 1)                       # (R, D)
    mean, thres = ops.ref_mean_and_thres(torch.from_numpy(ref_feat).cuda())
    ref_mean_vec = mean.cpu().numpy()
    max_dist_from_mean = np.float32(thres.item())
    print(f"number of samples considered for reference={ref_num}",
          f"ref mean shape={ref_mean_vec.shape}",
          f"ref feat shape={(ref_num, 1, ref_feat.shape[1])}")
    print("max dist from mean in the reference batch: ", max_dist_from_mean)
    return ref_mean_vec, max_dist_from_mean


def get_parsed_args(argv=None):
    parser = argparse.ArgumentParser()
    parser.add_argument('--ud', '--unfiltered_data_path', dest="unfiltered_data_path", type=str, required=True,
                        help='Unfiltered raw face dataset path with class imgs in subdirs')
    parser.add_argument('--rd', '--reference_data_path', dest="reference_data_path", type=str, required=True,
                        help='Reference face dataset path with class imgs in each subdirs that are manually prefiltered')
    parser.add_argument('--td', '--target_data_path', dest="target_data_path", type=str, default="data/faces_filtered",
                        help='Dataset path where subdirs clean and unclean contain respective filtered classes')
    parser.add_argument('-m', '--savedmodel_path', type=str, default="models/facenet/facenet_keras_p38",
                        help='Path to the MobileFaceNet state dict. (default: %(default)s)')
    parser.add_argument('-b', '--batch_size', type=int, default=32, help='Dataloader batch size. (default: %(default)s)')
    parser.add_argument('-r', '--ref_img_per_class', type=int, default=32,
                        help='Number of reference images to consider per class: %(default)s)')
    # optional additions (defaults reproduce the reference's behaviour)
    parser.add_argument('--gallery', action='store_true',
                        help='match every candidate against ALL reference embeddings (tensor cores) instead of '
                             'the class mean vector')
    parser.add_argument('--metric', choices=['cosine', 'euclid'], default='cosine',
                        help='decision rule of --gallery mode: best cosine >= threshold, or smallest Euclid distance <= threshold')
    parser.add_argument('--threshold', type=float, default=0.5,
                        help='threshold of --gallery mode: a cosine similarity, or a distance with --metric euclid')
    parser.add_argument('--mobilefacenet_dir', type=str,
                        default=os.environ.get("FFR_MOBILEFACENET_DIR",
                                               "../face_detection_and_extraction/modules/mobile_facenet"))
    parser.add_argument('--device', type=str, default="cuda:0")
    parser.add_argument('--ngpus', type=int, default=1,
                        help='distribute the classes (independent problems, reference :161) over this many GPUs: one worker '
                             'thread and one model replica per GPU')
    parser.add_argument('--allow_random_init', action='store_true')
    return parser.parse_args(argv)


def filter_class(model, ref_class_path: str, unfiltered_class_path: str, clean_dir: str, unclean_dir: str,
                 batch_size: int = 32, ref_img_per_class: int = 32, gallery: bool = False, threshold: float = 0.5,
                 device: str = "cuda:0", ref_stats=None, metric: str = "cosine"):
    """One iteration of the reference's per-class loop (:161-199).  Returns (similar_cnt, total, keep mask).
    ``ref_stats`` = (mean [1, D] CUDA, thres float) when the caller computed all classes' statistics up front; ``metric`` is the
    decision rule of gallery mode."""
    dev = torch.device(device)
    cls = unfiltered_class_path.split('/')[-1]
    filtered_class_clean_dir = os.path.join(clean_dir, cls)
    filtered_class_unclean_dir = os.path.join(unclean_dir, cls)
    os.makedirs(filtered_class_clean_dir, exist_ok=True)
    os.makedirs(filtered_class_unclean_dir, exist_ok=True)

    X_imgs = sorted(glob.glob(unfiltered_class_path + "/*.jpg"))
    if gallery:
        ref_imgs = sorted(glob.glob(ref_class_path + "/*.jpg"))[:ref_img_per_class]
        ref = _embed_paths_device(model, ref_imgs, batch_size, dev)
        thr = threshold
    elif ref_stats is not None:
        ref, thr, metric = ref_stats[0].reshape(1, -1), float(ref_stats[1]), "euclid"
    else:
        print(f"Calculating ref mean vector for {ref_class_path}")
        ref_mean_vec, thres = get_ref_mean_vec_and_thres_from_imgs(model, ref_class_path, max_ref_img_count=ref_img_per_class)
        ref = torch.from_numpy(np.ascontiguousarray(ref_mean_vec.reshape(1, -1))).to(dev)
        thr, metric = float(thres), "euclid"
    total = len(X_imgs)
    if total == 0:
        return 0, 0, np.zeros(0, dtype=np.uint8)
    cand = _embed_paths_device(model, X_imgs, batch_size, dev)
    keep = ops.face_filter(ref, cand, thr, metric=metric).keep.cpu().numpy()      # the hot path (:186-189)
    similar_cnt = int(keep.sum())
    for path, k in zip(X_imgs, keep):
        name = path.split('/')[-1]
        shutil.copy(path, os.path.join(filtered_class_clean_dir if k else filtered_class_unclean_dir, name))
    return similar_cnt, total, keep


def all_ref_stats(model, ref_class_paths: List[str], ref_img_per_class: int, device: str = "cuda:0"):
    """Mean vector and threshold of EVERY class in one kernel launch (K5 batched): the reference embeds and reduces
    one class at a time (:161-164).  Returns a list of (mean [1, D] CUDA tensor, thres float)."""
    dev = torch.device(device)
    feats, counts = [], []
    for path in ref_class_paths:
        imgs = sorted(glob.glob(path + "/*.jpg"))[:ref_img_per_class]
        # the reference embeds its references with batch size 1 (:77); a device-side model takes them as ONE batch
        f = _embed_paths_device(model, imgs, max(1, len(imgs)) if hasattr(model, "embed") else 1, dev)
        print(f"Calculating ref mean vector for {path}")
        print(f"number of samples considered for reference={len(imgs)}", f"ref mean shape={(1, f.shape[1]) if len(imgs) else None}",
              f"ref feat shape={(len(imgs), 1, f.shape[1] if len(imgs) else 0)}")
        feats.append(f)
        counts.append(len(imgs))
    dim = max((f.shape[1] for f in feats if f.numel()), default=0)
    feats = [f if f.numel() else torch.zeros((0, dim), dtype=torch.float32, device=dev) for f in feats]
    mean, thres = ops.ref_mean_and_thres_batched(torch.cat(feats, dim=0), counts)
    thres_h = thres.cpu().numpy()
    for t in thres_h:
        print("max dist from mean in the reference batch: ", t)
    return [(mean[i:i + 1], float(thres_h[i])) for i in range(len(counts))]


def main(argv=None, model=None, model_factory=None):
    """``model``: any object with the reference's ``predict`` contract (:84,184); ``model_factory(device) -> model`` builds
    the per-GPU replicas of ``--ngpus`` > 1 (default: MobileFaceNetModel on that device)."""
    args = get_parsed_args(argv)
    print(args)
    if model is None and model_factory is not None:
        model = model_factory(args.device)
    if model is None:
        model = MobileFaceNetModel(args.savedmodel_path, args.mobilefacenet_dir, device=args.device,
                                   allow_random_init=args.allow_random_init)
    print(f"Printing signature of model from {args.savedmodel_path}")
    print("\tInput:", getattr(model, "inputs", None))
    print("\tOutput:", getattr(model, "outputs", None))

    UNFILTERED_ROOT = _fix_path_for_globbing(args.unfiltered_data_path)
    REFERENCE_ROOT = _fix_path_for_globbing(args.reference_data_path)
    TARGET_ROOT = args.target_data_path
    ref_class_paths = sorted(glob.glob(REFERENCE_ROOT))
    unfiltered_class_paths = sorted(glob.glob(UNFILTERED_ROOT))
    if len(unfiltered_class_paths) != len(ref_class_paths):
        raise Exception(f"Class number Error. Unfiltered root {UNFILTERED_ROOT} and reference root {REFERENCE_ROOT} "
                        "must have the same number of classes")
    for i in range(len(ref_class_paths)):
        if ref_class_paths[i].split('/')[-1] != unfiltered_class_paths[i].split('/')[-1]:
            raise Exception(f"class {ref_class_paths[i]} and {unfiltered_class_paths[i]} did not match")

    clean_dir = os.path.join(TARGET_ROOT, 'clean')
    unclean_dir = os.path.join(TARGET_ROOT, 'unclean')
    os.makedirs(clean_dir, exist_ok=True)
    os.makedirs(unclean_dir, exist_ok=True)

    def run_classes(indices, mdl, device, progress=None, say=None):
        """The reference's per-class loop (:161-199) over ``indices`` on one device; returns {class index: summary line}
        (``say``: print each line as soon as its class is done, like the reference)."""
        paths = [ref_class_paths[i] for i in indices]
        stats = None if args.gallery else all_ref_stats(mdl, paths, args.ref_img_per_class, device)
        lines = {}
        for k, i in enumerate(indices):
            similar_cnt, total, _ = filter_class(mdl, ref_class_paths[i], unfiltered_class_paths[i], clean_dir, unclean_dir,
                                                 batch_size=args.batch_size, ref_img_per_class=args.ref_img_per_class,
                                                 gallery=args.gallery, threshold=args.threshold, device=device, metric=args.metric,
                                                 ref_stats=None if stats is None else stats[k])
            # the reference divides unconditionally (ZeroDivisionError on an empty class, :199); keep that behaviour
            lines[i] = f"Similar images percentage={similar_cnt/total:2.2f}%, positive={similar_cnt}, total={total}"
            if say is not None:
                say(lines[i])
            if progress is not None:
                progress.update(1)
        return lines

    try:
        import tqdm
        bar = tqdm.tqdm(total=len(ref_class_paths))
    except ImportError:
        bar = None
    n_gpus = max(1, min(int(args.ngpus), torch.cuda.device_count() or 1, max(1, len(ref_class_paths))))
    if n_gpus == 1:
        run_classes(list(range(len(ref_class_paths))), model, args.device, bar, say=print)
        lines = {}
    else:
        # classes are independent problems: class i goes to GPU i mod n (one worker thread + one model replica per GPU; the
        # library is re-entrant per device and stream).  Summary lines are printed in class order afterwards.
        from concurrent.futures import ThreadPoolExecutor
        replicas = [model_factory(f"cuda:{g}") if model_factory is not None else None for g in range(n_gpus)]
        if any(r is None for r in replicas):
            replicas = [MobileFaceNetModel(args.savedmodel_path, args.mobilefacenet_dir, device=f"cuda:{g}",
                                           allow_random_init=args.allow_random_init) for g in range(n_gpus)]
        def worker(g):
            with torch.cuda.device(g):
                return run_classes(list(range(g, len(ref_class_paths), n_gpus)), replicas[g], f"cuda:{g}", bar)
        with ThreadPoolExecutor(max_workers=n_gpus) as pool:
            lines = {}
            for part in pool.map(worker, range(n_gpus)):
                lines.update(part)
    if bar is not None:
        bar.close()
    for i in sorted(lines):
        print(lines[i])


if __name__ == "__main__":
    main()
