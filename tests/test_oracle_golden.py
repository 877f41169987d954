"""CPU: the oracle (oracle/oracle.py) pinned against outputs of the reference itself (tests/golden/*.npz)."""
import os

import numpy as np
import pytest

from oracle import oracle


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def _cand_rows(g, c):
    """Which of class c's candidates are stored: a fixture may hold a sample of the embeddings (oracle/gen_golden.py)."""
    key = f"c{c}_cand_rows"
    return g[key] if key in g.files else slice(None)


@pytest.mark.parametrize("name", ["ref_main_facenetlike.npz", "ref_main_mobilefacenet.npz"])
def test_mean_thres_and_keep_match_reference_main(golden_dir, name):
    """oracle.ref_mean_vec_and_thres / euclid_keep_literal == what the reference's main() computed
    (filter_faces_using_reference.py:85-99, :186-189)."""
    g = _load(golden_dir, name)
    assert int(g["n_classes"]) == 3
    for c in range(3):
        ref_feat, mu_ref, thres_ref = g[f"c{c}_ref_feat"], g[f"c{c}_mu"], g[f"c{c}_thres"]
        mu, thres = oracle.ref_mean_vec_and_thres(ref_feat, 32)
        assert mu.shape == mu_ref.shape == (1, ref_feat.shape[2])
        np.testing.assert_array_equal(mu, mu_ref)                 # same NumPy calls -> bit exact
        assert np.float32(thres) == np.float32(thres_ref)
        keep = oracle.euclid_keep_literal(g[f"c{c}_cand"], mu, thres)
        np.testing.assert_array_equal(keep, g[f"c{c}_keep"][_cand_rows(g, c)])
        # the reference's printed summary (positive=..., total=...) counts the decisions of every candidate
        summary = str(g[f"c{c}_summary"])
        assert f"positive={int(g[f'c{c}_keep'].sum())}, total={len(g[f'c{c}_keep'])}" in summary
        # vectorised restatement agrees with the literal loop
        k2, i2, d2 = oracle.filter_euclid(mu.reshape(1, -1), g[f"c{c}_cand"], thres)
        np.testing.assert_array_equal(k2, keep)
        assert np.all(i2 == 0)


def test_l2_norm_matches_reference(golden_dir):
    """oracle.l2_norm == mobile_facenet.py:30-33 run in torch (1-ulp tolerance: different reduction order)."""
    g = _load(golden_dir, "l2norm_ref.npz")
    for k in "abcd":
        x, y = g[f"{k}_x"], g[f"{k}_y"]
        np.testing.assert_allclose(oracle.l2_norm(x), y, rtol=3e-7, atol=1e-9)
        np.testing.assert_allclose(np.stack([oracle.l2_normalise_vec(r) for r in x]), y, rtol=3e-7, atol=1e-9)


@pytest.mark.parametrize("tag,metric", [("mfn", oracle.METRIC_EUCLID), ("reid", oracle.METRIC_COSINE)])
def test_first_match_scan_matches_reference(golden_dir, tag, metric):
    """oracle.first_match_scan == Net.check_if_face_exists (extract_and_label_faces_from_dataset.py:101-116)."""
    g = _load(golden_dir, "label_scan_ref.npz")
    feats, bboxes = g[f"{tag}_feats"], g[f"{tag}_bboxes"]

    def iou(a, b):                                                # restates modules/utils/image.py:124-143
        xd = min(a[2], b[2]) - max(a[0], b[0])
        yd = min(a[3], b[3]) - max(a[1], b[1])
        if xd < 0 or yd < 0:
            return 0
        inter = xd * yd
        return inter / (((a[2] - a[0]) * (a[3] - a[1])) + ((b[2] - b[0]) * (b[3] - b[1])) - inter)

    gal_feat, gal_box, gal_id = [], [], []
    mism = 0
    for q in range(len(feats)):
        ious = [iou(b, bboxes[q]) for b in gal_box]
        found, pos = oracle.first_match_scan(gal_feat, feats[q], metric, ious=ious)
        if found != bool(g[f"{tag}_found"][q]) or (found and gal_id[pos] != int(g[f"{tag}_faceid"][q])):
            mism += 1
        if bool(g[f"{tag}_found"][q]):                            # follow the reference's trajectory
            pos = gal_id.index(int(g[f"{tag}_faceid"][q]))
            gal_feat[pos], gal_box[pos] = feats[q], bboxes[q]
        else:
            gal_feat.append(feats[q]); gal_box.append(bboxes[q]); gal_id.append(len(gal_id) + 1)
    assert mism == 0, mism


def test_cosine_euclid_equivalence_on_unit_norm():
    """d <= t  <=>  cos >= 1 - t^2/2 for unit-norm rows (SURVEY §0): both oracle filters agree away from the band."""
    ref, cand = oracle.make_synthetic(50, 2000, 128, seed=3)
    t = 1.0
    kc, ic, sc = oracle.filter_cosine(ref, cand, 1 - t * t / 2)
    ke, ie, de = oracle.filter_euclid(ref, cand, t)
    safe = np.abs(sc - (1 - t * t / 2)) > 1e-5
    np.testing.assert_array_equal(kc[safe], ke[safe])
    gap_ok = np.abs(de - np.sqrt(np.maximum(2 - 2 * sc, 0))) < 1e-3
    assert gap_ok.all()
    np.testing.assert_array_equal(ic[safe], ie[safe])


def test_first_argmax_on_duplicates():
    ref, cand = oracle.make_synthetic(64, 500, 64, seed=5, n_dup_refs=16)
    k, i, s = oracle.filter_cosine(ref, cand, 0.5)
    rn = ref / np.linalg.norm(ref, axis=1, keepdims=True)
    cn = cand / np.linalg.norm(cand, axis=1, keepdims=True)
    sim = rn @ cn.T
    for j in range(0, 500, 37):
        assert i[j] == int(np.flatnonzero(sim[:, j] == sim[:, j].max())[0])


def test_literal_and_vectorised_cosine_agree():
    ref, cand = oracle.make_synthetic(7, 40, 128, seed=9, unit_norm=False)
    k, i, s = oracle.filter_cosine(ref, cand, 0.5)
    for j in range(40):
        lit = np.array([1 - oracle.cosine_dist_literal(r, cand[j]) for r in ref], dtype=np.float32)
        assert abs(lit.max() - s[j]) < 2e-6
        assert int(np.argmax(lit)) == i[j] or abs(np.sort(lit)[-1] - np.sort(lit)[-2]) < 1e-6
