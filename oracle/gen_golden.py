#!/usr/bin/env python
"""Generate tests/golden/*.npz by EXECUTING THE UNMODIFIED REFERENCE in the authoring container.

Run once, here (``/root/reference`` is mounted read-only; it does not exist on the GPU box):

    python oracle/gen_golden.py [--reference /root/reference] [--out tests/golden]

What is executed from the reference, unmodified:

1. ``similar_face_filtering/filter_faces_using_reference.py`` -- imported with ``oracle/tf_shim``
   standing in for TensorFlow's I/O, then ``main()`` is run on the bundled faces
   (``similar_face_filtering/data/faces_{reference,unfiltered}``, BASELINE.json configs[0]).
   Every ``model.predict`` output, every ``(mean, thres)`` returned by
   ``get_ref_mean_vec_and_thres_from_imgs`` (:71-100) and the clean/unclean decision the script
   took for every file (:189-196) are recorded.  Two embedding models are used:
     * ``mobilefacenet``: the reference's own torch ``MobileFaceNet(512)`` (seeded random init, eval,
       CPU; trained weights are not in the repo) -> unit-norm 512-d;
     * ``facenetlike``: a fixed random projection to 128-d, un-normalised, norms ~10 like the Keras
       FaceNet the script was written for (golden thres 7.58 in the reference test).
2. ``face_detection_and_extraction/modules/mobile_facenet/mobile_facenet.py::l2_norm`` (:30-33).
3. ``face_detection_and_extraction/face_extraction/extract_and_label_faces_from_dataset.py::
   Net.check_if_face_exists`` (:101-116), called on an instance built with ``Net.__new__`` (the
   constructor loads ONNX/OpenVINO weights that are not in the repo); ``onnxruntime`` / ``openvino``
   are stubbed as empty modules because the module imports them at top level.

The resulting arrays are small and are committed; tests read only the committed files.
"""
from __future__ import annotations

import argparse
import contextlib
import glob as _glob
import io
import os
import sys
import tempfile
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import tf_shim  # noqa: E402


def _mobilefacenet_factory(reference_root):
    import torch
    import torch.nn.functional as F
    sys.path.insert(0, os.path.join(reference_root, "face_detection_and_extraction", "modules", "mobile_facenet"))
    import mobile_facenet as ref_mfn
    torch.manual_seed(42)
    net = ref_mfn.MobileFaceNet(512).eval()
    # Trained weights are not in the repo.  With untouched random-init BatchNorm statistics the
    # embedding is almost independent of the image (all pairwise distances ~1e-5), which would make
    # the fixture hinge on fp32 summation noise.  Calibrate the BatchNorm running statistics on the
    # bundled reference faces (train-mode forward passes, no gradient step): weights stay random, but
    # the embedding now varies across images like a real model's does.
    sff = os.path.join(reference_root, "similar_face_filtering", "data", "faces_reference")
    files = sorted(_glob.glob(os.path.join(sff, "*", "*.jpg")))[::2][:80]
    imgs = np.stack([tf_shim._per_image_standardization(tf_shim._resize(
        tf_shim._convert_image_dtype(tf_shim._decode_jpeg(tf_shim._read_file(f)), np.float32), (112, 112))) for f in files])
    calib = torch.from_numpy(imgs).permute(0, 3, 1, 2).contiguous()
    for m in net.modules():
        if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
            m.momentum = None                      # cumulative average -> exact calibration-batch statistics
            m.reset_running_stats()
    net.train()
    with torch.no_grad():
        for _ in range(3):
            net(calib)
    net.eval()

    class Adapter:
        inputs = "[b,160,160,3] f32 (NHWC, standardised)"
        outputs = "[b,512] f32 unit-norm (reference MobileFaceNet)"

        def predict(self, batch, verbose=0):
            x = torch.from_numpy(np.ascontiguousarray(batch)).permute(0, 3, 1, 2)
            x = F.interpolate(x, size=(112, 112), mode="bilinear", align_corners=False)
            with torch.no_grad():
                return net(x).numpy().astype(np.float32)
    return lambda path: Adapter()


def _facenetlike_factory():
    rng = np.random.default_rng(42)
    w = rng.standard_normal((16 * 16 * 3, 128)).astype(np.float32) * np.float32(0.035)

    class Adapter:
        inputs = "[b,160,160,3] f32"
        outputs = "[b,128] f32 un-normalised"

        def predict(self, batch, verbose=0):
            b = np.asarray(batch, dtype=np.float32)
            pooled = b.reshape(b.shape[0], 16, 10, 16, 10, 3).mean(axis=(2, 4)).reshape(b.shape[0], -1)
            return (pooled @ w).astype(np.float32)
    return lambda path: Adapter()


def sample_candidates(out, n_rows, seed=0):
    """Cuts every class's candidate embeddings in ``out`` to ``n_rows`` rows: the quarter nearest to the threshold (where a
    last-bit difference flips a decision) plus a seeded draw of the others.  ``c<i>_cand_rows`` lists the rows kept;
    the decisions, names and summary line of all candidates stay.  Keeps a 512-d fixture under 1 MB."""
    rng = np.random.default_rng(seed)
    for c in range(int(out["n_classes"])):
        cand = out[f"c{c}_cand"]
        if cand.shape[0] <= n_rows:
            continue
        d = np.linalg.norm(cand.astype(np.float64) - out[f"c{c}_mu"].astype(np.float64), axis=1)
        order = np.argsort(np.abs(d - float(out[f"c{c}_thres"])), kind="stable")
        near, rest = order[:n_rows // 4], order[n_rows // 4:]
        rows = np.sort(np.concatenate([near, rng.choice(rest, n_rows - len(near), replace=False)]))
        out[f"c{c}_cand"] = cand[rows]
        out[f"c{c}_cand_rows"] = rows.astype(np.int32)


def run_reference_main(reference_root, factory, out_path, tag, max_cand=None):
    sff = os.path.join(reference_root, "similar_face_filtering")
    calls = []                        # ("predict", ndarray) | ("stats", path, mu, thres) | ("glob", pattern, list)

    def rec_factory(path):
        model = factory(path)
        inner = model.predict

        def predict(batch, verbose=0):
            out = inner(batch, verbose=verbose)
            calls.append(("predict", np.array(out, copy=True)))
            return out
        model.predict = predict
        return model

    tf_shim.install(rec_factory)
    sys.path.insert(0, sff)
    sys.modules.pop("filter_faces_using_reference", None)
    import filter_faces_using_reference as ref_mod

    orig_stats = ref_mod.get_ref_mean_vec_and_thres_from_imgs

    def stats(model, path, max_ref_img_count=32):
        mu, thres = orig_stats(model, path, max_ref_img_count=max_ref_img_count)
        calls.append(("stats", path, np.array(mu, copy=True), np.float32(thres)))
        return mu, thres
    ref_mod.get_ref_mean_vec_and_thres_from_imgs = stats

    orig_glob = _glob.glob

    def rec_glob(pattern, *a, **k):
        res = orig_glob(pattern, *a, **k)
        calls.append(("glob", pattern, list(res)))
        return res
    ref_mod.glob.glob = rec_glob

    target = tempfile.mkdtemp(prefix="ffr_golden_")
    argv = sys.argv
    sys.argv = ["filter_faces_using_reference.py",
                "--ud", os.path.join(sff, "data", "faces_unfiltered"),
                "--rd", os.path.join(sff, "data", "faces_reference"),
                "--td", target, "-b", "32", "-r", "32"]
    buf = io.StringIO()
    try:
        with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(io.StringIO()):
            ref_mod.main()
    finally:
        sys.argv = argv
        ref_mod.glob.glob = orig_glob
        sys.path.remove(sff)
    summary = [ln for ln in buf.getvalue().splitlines() if ln.startswith("Similar images percentage")]

    # split the call log per class: [glob refs] predict*R stats [glob cands] predict*ceil(M/32)
    out = {}
    cls_i = 0
    i = 0
    while i < len(calls):
        if calls[i][0] == "stats":
            _, ref_path, mu, thres = calls[i]
            j = i - 1
            ref_feat = []
            while j >= 0 and calls[j][0] == "predict" and calls[j][1].shape[0] == 1 and len(ref_feat) < 32:
                ref_feat.append(calls[j][1])
                j -= 1
            ref_feat = np.asarray(ref_feat[::-1])                  # (R,1,D) like :85
            assert calls[i + 1][0] == "glob", calls[i + 1][0]
            names = calls[i + 1][2]
            k = i + 2
            cand = []
            while k < len(calls) and calls[k][0] == "predict" and sum(c.shape[0] for c in cand) < len(names):
                cand.append(calls[k][1])
                k += 1
            cand = np.concatenate(cand, axis=0)
            assert cand.shape[0] == len(names)
            cls = os.path.basename(ref_path)
            keep = np.array([os.path.exists(os.path.join(target, "clean", cls, os.path.basename(n))) for n in names],
                            dtype=np.uint8)
            unclean = np.array([os.path.exists(os.path.join(target, "unclean", cls, os.path.basename(n))) for n in names],
                               dtype=np.uint8)
            assert np.all(keep + unclean == 1)
            out[f"c{cls_i}_class"] = np.array(cls)
            out[f"c{cls_i}_ref_feat"] = ref_feat.astype(np.float32)
            out[f"c{cls_i}_mu"] = mu.astype(np.float32)
            out[f"c{cls_i}_thres"] = np.float32(thres)
            out[f"c{cls_i}_cand"] = cand.astype(np.float32)
            out[f"c{cls_i}_keep"] = keep
            out[f"c{cls_i}_names"] = np.array([os.path.basename(n) for n in names])
            out[f"c{cls_i}_summary"] = np.array(summary[cls_i])
            cls_i += 1
            i = k
        else:
            i += 1
    out["n_classes"] = np.int32(cls_i)
    if max_cand is not None:
        sample_candidates(out, max_cand)
    np.savez_compressed(out_path, **out)
    print(f"[{tag}] {cls_i} classes ->", out_path, {k: (v.shape if hasattr(v, 'shape') else v) for k, v in out.items()
                                                     if k.endswith(('_cand', '_thres'))})
    for s in summary:
        print("   ", s)


def run_l2norm(reference_root, out_path):
    import torch
    sys.path.insert(0, os.path.join(reference_root, "face_detection_and_extraction", "modules", "mobile_facenet"))
    import mobile_facenet as ref_mfn
    rng = np.random.default_rng(42)
    out = {}
    for name, shape, scale in (("a", (37, 128), 1.0), ("b", (16, 512), 9.0), ("c", (5, 256), 1e-3), ("d", (3, 100), 50.0)):
        x = (rng.standard_normal(shape) * scale).astype(np.float32)
        y = ref_mfn.l2_norm(torch.from_numpy(x), axis=1).numpy()
        out[f"{name}_x"], out[f"{name}_y"] = x, y
    np.savez_compressed(out_path, **out)
    print("[l2norm] ->", out_path)


def run_label_scan(reference_root, out_path):
    fde = os.path.join(reference_root, "face_detection_and_extraction")
    for stub in ("onnxruntime", "openvino"):
        sys.modules.setdefault(stub, types.ModuleType(stub))
    cwd = os.getcwd()
    tmp = tempfile.mkdtemp(prefix="ffr_label_")
    os.chdir(tmp)                                   # the module creates ./logs at import
    sys.path.insert(0, fde)
    try:
        sys.path.insert(0, os.path.join(fde, "face_extraction"))
        import extract_and_label_faces_from_dataset as lab
    finally:
        os.chdir(cwd)
    rng = np.random.default_rng(7)
    out = {}
    for tag, net_type, dim, unit in (("mfn", "MOBILE_FACENET", 512, True), ("reid", "FACE_REID_MNV3", 256, False)):
        net = lab.Net.__new__(lab.Net)
        net.feat_net_type = net_type
        net.face_feat_bbox_age_gender_list = []
        net.normal_thres, net.harsh_thres = 1., 0.72
        net.use_bbox_iou = True
        net.max_faceid = 0
        ids = rng.standard_normal((12, dim)).astype(np.float32)
        ids /= np.linalg.norm(ids, axis=1, keepdims=True)
        feats, bboxes, found, faceids = [], [], [], []
        for q in range(160):
            k = int(rng.integers(0, 12))
            noise = rng.standard_normal(dim).astype(np.float32)
            noise /= np.linalg.norm(noise)
            mix = np.float32(rng.uniform(0.2, 1.0))
            f = mix * ids[k] + np.sqrt(np.float32(1) - mix * mix) * noise
            f = (f / np.linalg.norm(f)).astype(np.float32)
            if not unit:
                f = (f * np.float32(rng.uniform(2.0, 9.0))).astype(np.float32)
            x0, y0 = rng.integers(0, 400, 2)
            bbox = np.array([x0, y0, x0 + rng.integers(30, 120), y0 + rng.integers(30, 120)], dtype=np.float32)
            with contextlib.redirect_stdout(io.StringIO()):
                ok, fid, _, _ = net.check_if_face_exists(f, bbox)
                if not ok:
                    net.add_face(f, bbox, 0, 0)
            feats.append(f)
            bboxes.append(bbox)
            found.append(ok)
            faceids.append(-1 if fid is None else fid)
        out[f"{tag}_feats"] = np.asarray(feats, dtype=np.float32)
        out[f"{tag}_bboxes"] = np.asarray(bboxes, dtype=np.float32)
        out[f"{tag}_found"] = np.asarray(found, dtype=np.uint8)
        out[f"{tag}_faceid"] = np.asarray(faceids, dtype=np.int32)
        print(f"[label_scan:{tag}] found {int(np.sum(found))}/160, gallery {net.max_faceid}")
    np.savez_compressed(out_path, **out)
    print("[label_scan] ->", out_path)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default="/root/reference")
    ap.add_argument("--out", default=os.path.join(os.path.dirname(HERE), "tests", "golden"))
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    run_l2norm(args.reference, os.path.join(args.out, "l2norm_ref.npz"))
    run_label_scan(args.reference, os.path.join(args.out, "label_scan_ref.npz"))
    run_reference_main(args.reference, _facenetlike_factory(), os.path.join(args.out, "ref_main_facenetlike.npz"),
                       "facenetlike")
    run_reference_main(args.reference, _mobilefacenet_factory(args.reference),
                       os.path.join(args.out, "ref_main_mobilefacenet.npz"), "mobilefacenet", max_cand=64)


if __name__ == "__main__":
    main()
