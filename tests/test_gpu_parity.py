"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the reference's golden outputs.

Bars (BASELINE.md): similarities within 1e-3 absolute of the fp32 oracle; keep mask and best index exact,
except (a) rows whose fp64 best lies within the tolerance band of the threshold (listed) and (b) rows whose two
leading fp64 scores differ by less than fp32 summation noise (1e-6), where "the fp32 argmax" is itself
ill-defined.  Integer outputs are otherwise compared bit-exactly.
"""
import os

import numpy as np
import pytest
import torch

from oracle import oracle

pytestmark = pytest.mark.gpu

VAL_TOL = 1e-3          # north_star: similarities within 1e-3 absolute
TIE_EPS = 1e-6          # fp32 summation-order noise on a unit-norm dot product


@pytest.fixture(scope="module")
def ops(ffr_lib, cuda_dev):
    from face_detection_and_recognition_b200 import ops as _ops
    return _ops


def _top2_gap64(ref, cand, block=512):
    """fp64 shadow: (gap between the two leading scores, best score) per candidate, blocked over the candidates so that
    100 k references stay within a few hundred MB."""
    r = ref.astype(np.float64)
    r /= np.linalg.norm(r, axis=1, keepdims=True)
    gap = np.empty(len(cand))
    best = np.empty(len(cand))
    for s0 in range(0, len(cand), block):
        c = cand[s0:s0 + block].astype(np.float64)
        c /= np.linalg.norm(c, axis=1, keepdims=True)
        s = r @ c.T
        if s.shape[0] == 1:
            gap[s0:s0 + block], best[s0:s0 + block] = np.inf, s[0]
            continue
        b1 = s.max(axis=0)
        a1 = s.argmax(axis=0)
        s[a1, np.arange(s.shape[1])] = -np.inf
        gap[s0:s0 + block], best[s0:s0 + block] = b1 - s.max(axis=0), b1
    return gap, best


def _check_cosine(ops, ref, cand, thr, flags=0, band_tol=1e-3, sample=None):
    """GPU filter over ALL candidates against the oracle (+ fp64 shadow); ``sample`` = row subset the oracle is run on (the
    band listing is then checked on that subset)."""
    dev = torch.device("cuda:0")
    res = ops.face_filter(torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev), thr, metric="cosine",
                          band_tol=band_tol, flags=flags, want_stats=True)
    torch.cuda.synchronize()
    keep, idx, val = res.keep.cpu().numpy(), res.best_idx.cpu().numpy(), res.best_val.cpu().numpy()
    if sample is not None:
        sample = np.sort(np.asarray(sample))
        keep, idx, val, cand = keep[sample], idx[sample], val[sample], cand[sample]
    ko, io, so = oracle.filter_cosine(ref, cand, thr, block=1024 if len(ref) > 20_000 else 8192)
    gap, best64 = _top2_gap64(ref, cand)
    assert np.max(np.abs(val - so)) <= VAL_TOL, f"max |sim - oracle| = {np.max(np.abs(val - so))}"
    unamb = gap > TIE_EPS
    bad_idx = np.flatnonzero((idx != io) & unamb)
    assert bad_idx.size == 0, (f"{bad_idx.size} index mismatches outside fp32-tie rows, e.g. row {bad_idx[:5]} "
                               f"got {idx[bad_idx[:5]]} want {io[bad_idx[:5]]} gap {gap[bad_idx[:5]]} stats {res.stats}")
    band = oracle.tolerance_band(best64, thr, TIE_EPS)
    outside = np.ones(len(keep), bool)
    outside[band] = False
    bad_keep = np.flatnonzero((keep != ko) & outside)
    assert bad_keep.size == 0, f"{bad_keep.size} keep mismatches outside the band, e.g. {bad_keep[:5]} {best64[bad_keep[:5]]}"
    # the listed band must contain every row whose fp64 best is within band_tol - noise of thr
    if band_tol is not None:
        listed = set(res.band_rows.cpu().numpy().tolist())
        if sample is not None:
            pos = {int(r): i for i, r in enumerate(sample)}
            listed = {pos[r] for r in listed if r in pos}
        must = set(np.flatnonzero(np.abs(best64 - thr) <= band_tol - 1e-5).tolist())
        may = set(np.flatnonzero(np.abs(best64 - thr) <= band_tol + 1e-5).tolist())
        assert must <= listed <= may, (len(must - listed), len(listed - may))
    return res


# ---------------------------------------------------------------- K1
@pytest.mark.parametrize("rows,dim", [(1, 128), (37, 128), (1000, 512), (333, 256), (64, 384), (7, 1024), (19, 100),
                                      (5, 3), (4097, 128)])
def test_l2norm_rows(ops, rows, dim):
    rng = np.random.default_rng(rows * 1000 + dim)
    x = (rng.standard_normal((rows, dim)) * rng.uniform(0.01, 30)).astype(np.float32)
    out = ops.l2norm_rows(torch.from_numpy(x).cuda(), want_f16=True, want_f32=True, want_norms=True)
    torch.cuda.synchronize()
    y = oracle.l2_norm(x)
    np.testing.assert_allclose(out["f32"].cpu().numpy(), y, rtol=4e-7, atol=1e-9)
    np.testing.assert_allclose(out["norms"].cpu().numpy(), oracle.row_norms(x), rtol=4e-7)
    y16 = out["f16"].cpu().numpy()
    ld = (dim + 63) // 64 * 64
    assert y16.shape == (rows, ld) and y16.dtype == np.float16
    # fp16 copy = round-to-nearest of the fp32 result (allow 1 fp16 ulp where the fp32 values differ by an ulp)
    np.testing.assert_allclose(y16[:, :dim].astype(np.float32), y, rtol=1e-3, atol=1e-7)
    assert np.all(y16[:, dim:] == 0)


def test_l2norm_golden(ops, golden_dir):
    """K1 against the reference's own l2_norm outputs (mobile_facenet.py:30-33)."""
    g = np.load(os.path.join(golden_dir, "l2norm_ref.npz"))
    for k in "abcd":
        out = ops.l2norm_rows(torch.from_numpy(g[f"{k}_x"]).cuda())
        np.testing.assert_allclose(out["f32"].cpu().numpy(), g[f"{k}_y"], rtol=4e-7, atol=1e-9)


# ---------------------------------------------------------------- K5 + K2s against the reference's main()
@pytest.mark.parametrize("name", ["ref_main_facenetlike.npz", "ref_main_mobilefacenet.npz"])
def test_reference_main_golden(ops, golden_dir, name):
    """BASELINE configs[0]: mean vector, threshold and the clean/unclean decision of every stored candidate the
    reference's main() took on the bundled faces (filter_faces_using_reference.py:85-99, :186-189) are reproduced on the GPU."""
    g = np.load(os.path.join(golden_dir, name))
    for c in range(int(g["n_classes"])):
        ref_feat = torch.from_numpy(g[f"c{c}_ref_feat"]).cuda()
        mean, thres = ops.ref_mean_and_thres(ref_feat)
        np.testing.assert_allclose(mean.cpu().numpy(), g[f"c{c}_mu"], rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(float(thres), float(g[f"c{c}_thres"]), rtol=1e-6)
        # decisions with the reference's own (mu, thres)
        cand = g[f"c{c}_cand"]
        want = g[f"c{c}_keep"][g[f"c{c}_cand_rows"]] if f"c{c}_cand_rows" in g.files else g[f"c{c}_keep"]
        res = ops.face_filter(torch.from_numpy(g[f"c{c}_mu"]).cuda(), torch.from_numpy(cand).cuda(),
                              float(g[f"c{c}_thres"]), metric="euclid")
        keep = res.keep.cpu().numpy()
        d64 = np.linalg.norm(cand.astype(np.float64) - g[f"c{c}_mu"].astype(np.float64), axis=1)
        noise = np.abs(d64 - float(g[f"c{c}_thres"])) < 1e-6 * max(1.0, float(g[f"c{c}_thres"]))
        assert np.array_equal(keep[~noise], want[~noise]), np.flatnonzero(keep != want)
        assert noise.sum() <= 2
        np.testing.assert_allclose(res.best_val.cpu().numpy(), d64, rtol=2e-6, atol=1e-6)
        assert np.all(res.best_idx.cpu().numpy() == 0)
        # and end to end with the GPU's own (mu, thres)
        res2 = ops.face_filter(mean, torch.from_numpy(cand).cuda(), float(thres), metric="euclid")
        k2 = res2.keep.cpu().numpy()
        assert np.array_equal(k2[~noise], want[~noise])


# ---------------------------------------------------------------- K2s (exact fp32 CUDA-core path)
@pytest.mark.parametrize("n_ref,n_cand,dim,metric", [
    (1, 1000, 128, "euclid"), (1, 777, 512, "euclid"), (1, 50, 100, "euclid"), (3, 500, 128, "euclid"),
    (8, 300, 128, "cosine"), (2, 301, 512, "cosine"), (5, 64, 256, "cosine"), (40, 200, 128, "euclid"),
    (33, 100, 36, "cosine"), (4, 129, 1024, "euclid"), (6, 10, 2048, "cosine"),
    # dim 128 / 256 with <= 2 references: the sub-warp-per-row kernel (ragged row counts, both metrics)
    (1, 1001, 256, "euclid"), (2, 515, 128, "cosine"), (2, 77, 256, "cosine"), (1, 3, 128, "cosine"), (2, 4099, 128, "euclid")])
def test_filter_fp32_small(ops, n_ref, n_cand, dim, metric):
    ref, cand = oracle.make_synthetic(n_ref, n_cand, dim, seed=n_ref + n_cand + dim, unit_norm=(metric == "cosine"))
    from face_detection_and_recognition_b200.ops import FLAG_FORCE_FP32
    if metric == "euclid":
        thr = float(np.median(oracle.filter_euclid(ref, cand, 0)[2]))
        ko, io, so = oracle.filter_euclid(ref, cand, thr)
    else:
        thr = 0.5
        ko, io, so = oracle.filter_cosine(ref, cand, thr)
    res = ops.face_filter(torch.from_numpy(ref).cuda(), torch.from_numpy(cand).cuda(), thr, metric=metric,
                          flags=FLAG_FORCE_FP32, want_stats=True)
    assert res.stats["path"] == "fp32"
    keep, idx, val = res.keep.cpu().numpy(), res.best_idx.cpu().numpy(), res.best_val.cpu().numpy()
    np.testing.assert_allclose(val, so, rtol=3e-6, atol=3e-6)
    near = np.abs(so - thr) < 1e-5 * max(1.0, abs(thr))
    assert np.array_equal(keep[~near], ko[~near])
    assert np.mean(idx == io) > 0.995            # fp32 near-ties only
    assert np.all(np.abs(val - so)[idx != io] < 1e-5)


def test_filter_fp32_index_base_and_empty(ops):
    ref, cand = oracle.make_synthetic(4, 10, 128, seed=1)
    r = ops.face_filter(torch.from_numpy(ref).cuda(), torch.from_numpy(cand).cuda(), 0.5, ref_index_base=1000)
    _, io, _ = oracle.filter_cosine(ref, cand, 0.5)
    assert np.array_equal(r.best_idx.cpu().numpy(), io + 1000)
    e = ops.face_filter(torch.from_numpy(ref).cuda(), torch.empty((0, 128), device="cuda"), 0.5)
    assert e.keep.numel() == 0 and e.best_idx.numel() == 0


# ---------------------------------------------------------------- K2 raw scores (validates TMA/UMMA descriptors)
@pytest.mark.parametrize("n_ref,n_cand,dim", [(256, 128, 64), (256, 128, 128), (512, 256, 512), (100, 77, 128),
                                              (300, 130, 256), (1000, 333, 192), (17, 5, 64)])
def test_mma_raw_scores(ffr_lib, ops, n_ref, n_cand, dim):
    """Every accumulator element the tcgen05 kernel produces == fp32 dot of the same fp16-rounded rows."""
    ref, cand = oracle.make_synthetic(n_ref, n_cand, dim, seed=11)
    r16 = ops.l2norm_rows(torch.from_numpy(ref).cuda(), want_f16=True, want_f32=False)["f16"]
    c16 = ops.l2norm_rows(torch.from_numpy(cand).cuda(), want_f16=True, want_f32=False)["f16"]
    ld = r16.shape[1]
    scores = torch.full((n_cand, n_ref), float("nan"), device="cuda")
    keep = torch.empty(n_cand, dtype=torch.uint8, device="cuda")
    idx = torch.empty(n_cand, dtype=torch.int32, device="cuda")
    val = torch.empty(n_cand, dtype=torch.float32, device="cuda")
    ws = torch.zeros(4096 + 64 * n_cand, dtype=torch.uint8, device="cuda")
    from face_detection_and_recognition_b200._lib import check
    check(ffr_lib.ffr_debug_mma_scores(r16.data_ptr(), n_ref, c16.data_ptr(), n_cand, ld, 0.5, keep.data_ptr(),
                                       idx.data_ptr(), val.data_ptr(), scores.data_ptr(), ws.data_ptr(), ws.numel(),
                                       torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    want = (c16.float() @ r16.float().T).cpu().numpy()
    got = scores.cpu().numpy()
    assert not np.isnan(got).any(), f"{np.isnan(got).sum()} score elements never written"
    err = np.abs(got - want)
    assert err.max() < 2e-5, (f"max err {err.max()} at {np.unravel_index(err.argmax(), err.shape)}; "
                              f"per-column-block max {[float(err[:, i:i + 32].max()) for i in range(0, min(n_ref, 256), 32)]}")
    np.testing.assert_allclose(val.cpu().numpy(), want.max(axis=1), atol=2e-5)
    assert np.mean(idx.cpu().numpy() == want.argmax(axis=1)) > 0.99


# ---------------------------------------------------------------- K1+K2+K3 end to end
@pytest.mark.parametrize("n_ref,n_cand,dim", [
    (9, 100, 128), (255, 1000, 128), (256, 1000, 128), (257, 1000, 128), (1000, 5000, 128), (300, 129, 512),
    (2000, 3000, 512), (513, 1, 256), (64, 4000, 64), (700, 900, 200), (1111, 2049, 384), (300, 500, 50), (100, 257, 3),
    (40, 1000, 510),
    (9000, 600, 128)])          # > 8192 references: the sequential update path (update_chunk), not the batched one
def test_filter_mma_vs_oracle(ops, n_ref, n_cand, dim):
    ref, cand = oracle.make_synthetic(n_ref, n_cand, dim, seed=n_ref * 7 + dim, n_adversarial=min(200, n_cand // 4),
                                      n_dup_refs=min(32, n_ref // 4))
    res = _check_cosine(ops, ref, cand, 0.5)
    assert res.stats["path"] == "tcgen05"


def test_filter_mma_unnormalised_inputs(ops):
    """Raw (un-normalised) embeddings: cosine is scale invariant, K1 normalises internally."""
    ref, cand = oracle.make_synthetic(600, 2500, 128, seed=77, unit_norm=False, n_adversarial=100, n_dup_refs=8)
    _check_cosine(ops, ref, cand, 0.5)


@pytest.mark.parametrize("copies", [2, 3, 4, 6, 12])
def test_filter_mma_exact_ties_pick_first(ops, copies):
    """Duplicated references give exactly equal scores: best_idx must be the FIRST occurrence (np.argmax).  Up to three
    equal leaders are resolved by the three-candidate fp32 check (K3a); four or more force the full fp32 rescan (K3b)."""
    rng = np.random.default_rng(5)
    base = rng.standard_normal((40, 128)).astype(np.float32)
    ref = np.concatenate([base] * copies, axis=0)
    cand = (base[rng.integers(0, 40, 900)] + 0.3 * rng.standard_normal((900, 128))).astype(np.float32)
    dev = torch.device("cuda:0")
    from face_detection_and_recognition_b200.ops import FLAG_FORCE_MMA
    res = ops.face_filter(torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev), 0.5, flags=FLAG_FORCE_MMA,
                          want_stats=True)
    idx = res.best_idx.cpu().numpy()
    assert np.all(idx < 40), f"{np.sum(idx >= 40)} rows picked a later duplicate"
    _, io, _ = oracle.filter_cosine(base, cand, 0.5)
    gap, _ = _top2_gap64(base, cand)
    assert np.array_equal(idx[gap > TIE_EPS], io[gap > TIE_EPS])
    if copies >= 4:
        # every row has >= 4 scores inside the window: the copies inside ONE 128-column part -- or two ADJACENT parts (6
        # copies = 240 references), joined when the column halves are merged -- are resolved by K3's part rescan; copies
        # spread over three or more parts (12 copies = 480 references) need every reference
        assert res.stats["part_rescans"] + res.stats["full_rescans"] >= 900
        if copies >= 10:
            assert res.stats["full_rescans"] >= 700
        elif copies >= 6:
            assert res.stats["part_rescans"] >= 700 and res.stats["full_rescans"] == 0
    else:
        assert res.stats["rechecked"] + res.stats["part_rescans"] >= 900


@pytest.mark.parametrize("n_ref,n_cand,dim", [(300, 5000, 128), (1000, 3001, 256), (64, 700, 64), (500, 129, 192),
                                              (300, 60_000, 128), (700, 45_000, 512), (257, 40_001, 320),
                                              (90, 38_000 + 100, 260), (33, 19_000 + 129, 64), (64, 512 * 74 + 77, 128),
                                              (500, 40_000, 100), (1100, 20_001, 72), (260, 57_000, 124)])
def test_fused_normalisation_path(ops, ffr_env, n_ref, n_cand, dim):
    """K2 with in-kernel normalisation of the candidates (two normaliser warps write the fp16 rows of the CTA's next tile
    into the workspace while the tensor core works; default for large reference sets, forced here with FFR_FUSE_K1=1):
    same parity bar as K1 + K2, and the same decisions as the K1 + K2 schedule.  Rows of 68..128 floats take the stage32
    form (fp32 rows staged through shared memory by TMA, fp16 A tile written in place, no global scratch)."""
    ref, cand = oracle.make_synthetic(n_ref, n_cand, dim, seed=dim + n_ref, n_adversarial=100, n_dup_refs=8, unit_norm=False)
    ffr_env.setenv("FFR_FUSE_K1", "1")
    res = _check_cosine(ops, ref, cand, 0.5)
    assert res.stats["launches"] == 3                      # K1(references only) + K2 + K3: no K1 pass over the candidates
    ffr_env.setenv("FFR_FUSE_K1", "0")
    import torch
    r2 = ops.face_filter(torch.from_numpy(ref).cuda(), torch.from_numpy(cand).cuda(), 0.5, band_tol=1e-3)
    # the two schedules differ by <= 1 fp16 ulp in rare operand elements (x * (1/|x|) vs x / |x|): same decisions
    assert (res.best_idx != r2.best_idx).float().mean().item() < 1e-3
    assert (res.keep != r2.keep).float().mean().item() < 1e-3
    assert (res.best_val - r2.best_val).abs().max().item() < 1e-3


def test_filter_mma_config2_full(ops):
    """BASELINE configs[1] in full: 1k references x 100k candidates x 128-d, threshold 0.5."""
    ref, cand = oracle.make_synthetic(1000, 100_000, 128, seed=42, n_adversarial=1000, n_dup_refs=100)
    res = _check_cosine(ops, ref, cand, 0.5)
    assert 0.3 < res.keep.float().mean().item() < 0.7


def test_filter_mma_f16_inputs(ops):
    """Pre-normalised fp16 rows in (FFR_DTYPE_F16): no fp32 re-check possible, values still within 1e-3."""
    ref, cand = oracle.make_synthetic(500, 2000, 256, seed=8)
    r16 = ops.l2norm_rows(torch.from_numpy(ref).cuda(), want_f16=True, want_f32=False)["f16"]
    c16 = ops.l2norm_rows(torch.from_numpy(cand).cuda(), want_f16=True, want_f32=False)["f16"]
    res = ops.face_filter(r16, c16, 0.5)
    ko, io, so = oracle.filter_cosine(ref, cand, 0.5)
    assert np.max(np.abs(res.best_val.cpu().numpy() - so)) < VAL_TOL
    assert np.mean(res.best_idx.cpu().numpy() == io) > 0.99
    far = np.abs(so - 0.5) > VAL_TOL
    assert np.array_equal(res.keep.cpu().numpy()[far], ko[far])


def test_host_filter_matches_device_path(ops):
    ref, cand = oracle.make_synthetic(300, 10_000, 128, seed=21)
    hf = ops.HostFilter(device=0, max_ref=1024, chunk_cand=3000, max_dim=128)
    keep, idx, val = hf(ref, cand, 0.5)
    res = ops.face_filter(torch.from_numpy(ref).cuda(), torch.from_numpy(cand).cuda(), 0.5)
    assert np.array_equal(keep, res.keep.cpu().numpy())
    assert np.array_equal(idx, res.best_idx.cpu().numpy())
    np.testing.assert_allclose(val, res.best_val.cpu().numpy(), atol=1e-6)
    assert hf.launches > 0
    # euclid, one mean vector (the reference's literal mode) through the host entry point
    mu = ref[:1] * 3.0
    keep_e, idx_e, val_e = hf(mu, cand * 3.0, 4.0, metric="euclid")
    ko, io, so = oracle.filter_euclid(mu, cand * 3.0, 4.0)
    near = np.abs(so - 4.0) < 1e-5
    assert np.array_equal(keep_e[~near], ko[~near])
    hf.close()


def test_errors_are_loud(ffr_lib, ops):
    from face_detection_and_recognition_b200._lib import FfrError
    ref = torch.randn(16, 128, device="cuda")
    cand = torch.randn(32, 128, device="cuda")
    with pytest.raises(TypeError):
        ops.face_filter(ref.cpu(), cand, 0.5)
    with pytest.raises(ValueError):
        ops.face_filter(ref, cand[:, :64], 0.5)
    with pytest.raises(FfrError):                                  # workspace too small is reported, not ignored
        from face_detection_and_recognition_b200._lib import check
        keep = torch.empty(32, dtype=torch.uint8, device="cuda")
        idx = torch.empty(32, dtype=torch.int32, device="cuda")
        check(ffr_lib.ffr_filter(ref.data_ptr(), 16, cand.data_ptr(), 32, 128, 0, None, None, 0, 0.5, 0,
                                 keep.data_ptr(), idx.data_ptr(), None, None, 0, None))


def test_fused_normalisation_is_the_default_for_large_reference_sets(ops):
    """Above 24 reference tiles and ~76 k candidates ffr_filter drops the K1 pass over the candidates on its own (two
    launches besides K3: K1 over the references + K2): checked on a ragged shape against the oracle."""
    n_ref, n_cand, dim = 6500, 75_777 + 300, 128
    ref, cand = oracle.make_synthetic(n_ref, n_cand, dim, seed=11, n_adversarial=500, n_dup_refs=50, unit_norm=False)
    res = _check_cosine(ops, ref, cand, 0.5)
    assert res.stats["launches"] == 3 and res.stats["path"] == "tcgen05"


# ---------------------------------------------------------------- K2 epilogue variants (round-1d)
def _near_tie_refs(n_ref, dim, seed, n_pairs):
    """References with planted near-duplicates (cos gap ~1e-4..1e-3 after fp16 rounding), both inside one 128-column part
    (offset 3, 9, 40) and across parts / tiles (offset 130, 300): every branch of update_grid sees traffic."""
    rng = np.random.default_rng(seed)
    ref = rng.standard_normal((n_ref, dim)).astype(np.float32)
    offs = [o for o in (3, 9, 40, 130, 300) if o < n_ref - 2]
    for k in range(n_pairs):
        off = offs[k % len(offs)]
        i = int(rng.integers(0, n_ref - off - 1))
        ref[i + off] = ref[i] + rng.standard_normal(dim).astype(np.float32) * 0.004
    return ref


@pytest.mark.parametrize("n_ref,n_cand,dim", [(700, 6000, 128), (1500, 3000, 256), (9000, 2500, 128), (300, 40_000, 64)])
@pytest.mark.parametrize("mode", ["default", "exact", "gated", "gated_flag_only"])
def test_update_grid_variants(ops, ffr_env, n_ref, n_cand, dim, mode):
    """update_grid (unconditional / gated), its two fall-backs for several in-window columns in one part (exact per-column
    masks, or flag-the-row-for-the-full-rescan) all meet the same parity bar -- on references with planted near-duplicates,
    so that the fall-backs actually run."""
    env = {"default": {}, "exact": {"FFR_GRID_EXACT": "1"},
           "gated": {"FFR_GRID_UPDATE_REFS": "0", "FFR_GRID_EXACT": "1"},
           "gated_flag_only": {"FFR_GRID_UPDATE_REFS": "0", "FFR_GRID_EXACT": "0"}}[mode]
    for k, v in env.items():
        ffr_env.setenv(k, v)
    ref = _near_tie_refs(n_ref, dim, seed=n_ref + dim, n_pairs=40)
    rng = np.random.default_rng(n_cand)
    cand = rng.standard_normal((n_cand, dim)).astype(np.float32)
    src = rng.integers(0, n_ref, n_cand // 2)
    cand[::2][: len(src)] = ref[src] + 0.25 * rng.standard_normal((len(src), dim)).astype(np.float32)
    from face_detection_and_recognition_b200.ops import FLAG_FORCE_MMA
    res = _check_cosine(ops, ref, cand, 0.5, flags=FLAG_FORCE_MMA)
    assert res.stats["path"] == "tcgen05"
    assert res.stats["rechecked"] + res.stats["part_rescans"] + res.stats["full_rescans"] > 0
    if mode in ("default", "gated_flag_only"):
        assert res.stats["k2"]["grid_exact"] == 0 and res.stats["part_rescans"] > 0      # same-part near ties -> K3's part rescan


def test_update_grid_variants_agree_bitwise(ops, ffr_env):
    """Every epilogue variant hands K3 what it needs: after the fp32 re-check the outputs are IDENTICAL, bit for bit."""
    ref = _near_tie_refs(2000, 128, seed=11, n_pairs=60)
    rng = np.random.default_rng(12)
    cand = rng.standard_normal((30_000, 128)).astype(np.float32)
    cand[::3] = ref[rng.integers(0, 2000, 10_000)] + 0.2 * rng.standard_normal((10_000, 128)).astype(np.float32)
    dev = torch.device("cuda:0")
    r_t, c_t = torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev)
    outs = []
    for env in ({}, {"FFR_GRID_EXACT": "1"}, {"FFR_GRID_UPDATE_REFS": "0"}, {"FFR_GRID_UPDATE_REFS": "0", "FFR_GRID_EXACT": "1"},
                {"FFR_CTA_GROUP": "1"}, {"FFR_CTA_GROUP": "1", "FFR_GRID_EXACT": "1"}):
        for k, v in env.items():
            ffr_env.setenv(k, v)
        res = ops.face_filter(r_t, c_t, 0.5, want_stats=True)
        torch.cuda.synchronize()
        outs.append((res.keep.cpu().numpy().copy(), res.best_idx.cpu().numpy().copy(), res.best_val.cpu().numpy().copy()))
        ffr_env.restore()
    gap, _ = _top2_gap64(ref, cand)
    unamb = gap > TIE_EPS
    for k, i, v in outs[1:]:
        assert np.array_equal(k, outs[0][0])
        assert np.array_equal(i[unamb], outs[0][1][unamb])
        np.testing.assert_allclose(v, outs[0][2], atol=2e-4)          # un-flagged rows carry the fp16-operand score


@pytest.mark.parametrize("tiles_per_cta,dim,n_ref", [(1, 128, 200), (2, 128, 777), (3, 128, 200), (5, 128, 300), (1, 384, 777),
                                                     (2, 384, 200), (3, 512, 200), (2, 512, 520)])
def test_candidate_tile_sequences(ops, tiles_per_cta, dim, n_ref):
    """Odd and even numbers of candidate tiles per CTA (the column halves take turns at the merge + emit tail; the A ring is
    handed over K-block by K-block, one stage at dim >= 320), with ONE reference tile (first = last) and several."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n_cand = 128 * sms * tiles_per_cta - 37
    ref, cand = oracle.make_synthetic(n_ref, n_cand, dim, seed=dim + tiles_per_cta + n_ref, n_adversarial=50, n_dup_refs=8)
    _check_cosine(ops, ref, cand, 0.5)


@pytest.mark.parametrize("stage32", ["1", "0"])
def test_fused_forms_agree(ops, ffr_env, stage32):
    """stage32 and the global-scratch form of the in-kernel normalisation do the same arithmetic per row (one float4 per
    lane, warp-shuffle sum, one division, multiplies): identical fp16 operands, hence identical outputs as the direct form
    with FFR_STAGE32=0.  Also covers cta_group::1 (five staging buffers instead of six)."""
    ref, cand = oracle.make_synthetic(900, 128 * 148 * 2 + 55, 128, seed=3, n_adversarial=200, n_dup_refs=16, unit_norm=False)
    ffr_env.setenv("FFR_FUSE_K1", "1")
    ffr_env.setenv("FFR_STAGE32", stage32)
    res = _check_cosine(ops, ref, cand, 0.5)
    ffr_env.setenv("FFR_CTA_GROUP", "1")
    r1 = _check_cosine(ops, ref, cand, 0.5)
    assert torch.equal(res.keep, r1.keep) and torch.equal(res.best_idx, r1.best_idx)


# ---------------------------------------------------------------- BASELINE configs[4]'s own reference count (round 2)
def _large_gallery(n_ref, n_cand, dim, seed):
    """100 k-reference gallery with the hard rows planted: near-duplicate references inside one 128-column part and
    across parts / tiles, exact duplicates, candidates within +-2e-3 of the threshold, and candidates sitting on the
    near-duplicate pairs (so the near ties are actually leading)."""
    ref, cand = oracle.make_synthetic(n_ref, n_cand, dim, seed=seed, n_adversarial=1000, n_dup_refs=1000)
    rng = np.random.default_rng(seed + 1)
    offs = (3, 9, 40, 130, 300, (n_ref * 7) // 10)
    src = rng.integers(0, n_ref // 4, 600)
    for k, i in enumerate(src):
        j = int(i) + offs[k % len(offs)]
        ref[j] = ref[i] + rng.standard_normal(dim).astype(np.float32) * 0.0004      # cos ~ 1 - 1e-5: inside delta
        ref[j] /= np.linalg.norm(ref[j])
    rows = rng.choice(n_cand, 3000, replace=False)
    tgt = src[rng.integers(0, len(src), len(rows))]
    noise = rng.standard_normal((len(rows), dim)).astype(np.float32)
    noise /= np.linalg.norm(noise, axis=1, keepdims=True)
    cand[rows] = 0.8 * ref[tgt] + 0.6 * noise
    return ref, cand, rows


def test_filter_mma_config4_gallery_size(ops):
    """n_ref = 100 000 x 128-d, default knobs: 391 reference tiles per candidate tile, indices > 65 535, the gated
    update_grid with the FLAG-ONLY fall-back (grid_exact = 0) and K3's full rescan over 100 k rows; >= 2 candidate tiles
    per CTA.  Oracle (fp32 + fp64 shadow) on a 3 k-row sample that contains every planted near-tie row."""
    n_ref, n_cand, dim = 100_000, 40_000, 128
    ref, cand, hard = _large_gallery(n_ref, n_cand, dim, seed=4)
    rng = np.random.default_rng(0)
    sample = np.unique(np.concatenate([hard[:1500], rng.choice(n_cand, 1500, replace=False)]))
    res = _check_cosine(ops, ref, cand, 0.5, sample=sample)
    assert res.stats["path"] == "tcgen05"
    assert res.stats["k2"]["grid_exact"] == 0 and res.stats["k2"]["grid_updates"] == 0, res.stats
    assert res.stats["part_rescans"] > 0 and res.stats["rechecked"] > 0
    assert int(res.best_idx.max()) > 65_535


def test_filter_mma_large_gallery_without_recheck_is_exact_in_fp16_space(ops, ffr_env):
    """fp16 input / FFR_FLAG_NO_RECHECK have no K3 behind them: the flag-only fall-back (placeholder column + 'rescan
    me') must not be taken, whatever FFR_GRID_EXACT says.  Every returned index must carry the row's best fp16-space
    score (ties -> first), also on rows with several in-window columns in one 128-column part."""
    from face_detection_and_recognition_b200.ops import FLAG_NO_RECHECK
    n_ref, n_cand, dim = 40_000, 6_000, 128
    ref, cand, hard = _large_gallery(n_ref, n_cand, dim, seed=9)
    ffr_env.setenv("FFR_GRID_EXACT", "0")
    r16 = ops.l2norm_rows(torch.from_numpy(ref).cuda(), want_f16=True, want_f32=False)["f16"]
    c16 = ops.l2norm_rows(torch.from_numpy(cand).cuda(), want_f16=True, want_f32=False)["f16"]
    want = (c16.float() @ r16.float().T)
    best, arg = want.max(dim=1)
    for res in (ops.face_filter(r16, c16, 0.5, want_stats=True, band_tol=1e-3),
                ops.face_filter(torch.from_numpy(ref).cuda(), torch.from_numpy(cand).cuda(), 0.5, flags=FLAG_NO_RECHECK,
                                want_stats=True, band_tol=1e-3)):
        assert res.stats["k2"]["grid_exact"] == 1, res.stats
        got = want.gather(1, res.best_idx.long()[:, None])[:, 0]
        # the accumulation order inside the tensor core differs from torch's: equal up to fp32 summation noise
        assert (got - best).abs().max().item() < 2e-6
        assert (res.best_val - best).abs().max().item() < 2e-5
        clear = (best - torch.topk(want, 2, dim=1).values[:, 1]) > 2e-6
        assert torch.equal(res.best_idx.long()[clear], arg[clear])
        # the tolerance band is listed on this path too (by K2's tail, from the fp16-operand score)
        listed = set(res.band_rows.cpu().numpy().tolist())
        must = set(torch.nonzero((best - 0.5).abs() <= 1e-3 - 3e-5)[:, 0].cpu().numpy().tolist())
        may = set(torch.nonzero((best - 0.5).abs() <= 1e-3 + 3e-5)[:, 0].cpu().numpy().tolist())
        assert must <= listed <= may and len(must) > 0


def test_two_devices_in_one_process(ops):
    """The > 48 KB shared-memory opt-in is a per-device function attribute: the first filter on a SECOND GPU of the same
    process must launch too (K2 and K3)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ref, cand = oracle.make_synthetic(700, 3000, 128, seed=5, n_adversarial=100, n_dup_refs=8)
    ko, io, _ = oracle.filter_cosine(ref, cand, 0.5)
    for d in (1, 0, 1):
        dev = torch.device("cuda", d)
        res = ops.face_filter(torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev), 0.5, want_stats=True)
        torch.cuda.synchronize(dev)
        assert res.stats["path"] == "tcgen05"
        assert np.mean(res.best_idx.cpu().numpy() == io) > 0.999


# ---------------------------------------------------------------- exact-duplicate references are folded before K2 (round 2)
@pytest.mark.parametrize("n_ref,n_cand,dim,copies", [(6000, 400_000, 128, 8), (4096, 500_000, 256, 3), (10_000, 210_000, 512, 5)])
def test_duplicate_heavy_gallery_is_folded(ops, ffr_env, n_ref, n_cand, dim, copies):
    """A gallery that enrols the same embedding several times (exact copies, scattered over the whole index range): the
    bit-identical rows are dropped before the tensor-core scan, K2 reports the unique row count, the answers are those of the
    oracle on the FULL gallery (first occurrence of the maximum), and nothing is left for K3's full rescan -- while the same
    call with FFR_DEDUP_REFS=0 sends every such row there (the cliff this removes) and gives the same answers."""
    rng = np.random.default_rng(n_ref + copies)
    n_id = n_ref // copies
    base = rng.standard_normal((n_id, dim)).astype(np.float32)
    ref = np.concatenate([base] * copies + [rng.standard_normal((n_ref - n_id * copies, dim)).astype(np.float32)])
    perm = rng.permutation(n_ref)
    ref = ref[perm]                                              # copies land anywhere; first occurrence = smallest index
    cand = rng.standard_normal((n_cand, dim)).astype(np.float32)
    hit = rng.integers(0, n_id, n_cand // 2)
    cand[::2][: len(hit)] = base[hit] + 0.35 * rng.standard_normal((len(hit), dim)).astype(np.float32)
    sample = rng.choice(n_cand, 3000, replace=False)
    res = _check_cosine(ops, ref, cand, 0.5, sample=sample)
    n_unique = len(np.unique(ref, axis=0))
    assert res.stats["refs_scanned"] == n_unique < n_ref, res.stats
    assert res.stats["full_rescans"] < n_cand // 200, res.stats
    ffr_env.setenv("FFR_DEDUP_REFS", "0")
    dev = torch.device("cuda:0")
    small = slice(0, 20_000)
    r0 = ops.face_filter(torch.from_numpy(ref).to(dev), torch.from_numpy(cand[small]).to(dev), 0.5, want_stats=True)
    ffr_env.setenv("FFR_DEDUP_REFS", "1")
    assert r0.stats["refs_scanned"] == n_ref
    if copies >= 4:
        assert r0.stats["full_rescans"] + r0.stats["part_rescans"] > 5000          # every planted row has >= 4 equal leaders
    r1 = ops.face_filter(torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev), 0.5)
    gap, _ = _top2_gap64(np.unique(ref, axis=0), cand[small][:2000])
    ok = torch.from_numpy(gap > TIE_EPS).to(dev)
    assert torch.equal(r0.best_idx[:2000][ok], r1.best_idx[:2000][ok]) and torch.equal(r0.keep[:2000], r1.keep[:2000])


@pytest.mark.parametrize("n_id,n_cand,dim", [(800, 80_000, 128), (1200, 40_000, 512), (7000, 30_000, 128)])
def test_near_duplicate_groups_across_part_boundaries(ops, n_id, n_cand, dim):
    """Five near-identical (cos 0.99995, NOT bit-equal) enrolments per identity, consecutive rows: every candidate of an
    identity has five scores inside the fp16 window, all in one 128-column part -- or, for the groups that straddle a part
    boundary (5 does not divide 128), in two ADJACENT parts, which the two column halves of the epilogue see separately.
    The merge of the halves joins adjacent parts into one record, so those rows get a two-part rescan instead of the fp32
    walk over every reference.  Parity with the oracle as everywhere; the full-rescan list stays (nearly) empty."""
    rng = np.random.default_rng(n_id + dim)
    base = rng.standard_normal((n_id, dim)).astype(np.float32)
    base /= np.linalg.norm(base, axis=1, keepdims=True)
    sib = np.repeat(base, 5, axis=0)
    jit = rng.standard_normal(sib.shape).astype(np.float32)
    jit -= (jit * sib).sum(1, keepdims=True) * sib
    jit /= np.linalg.norm(jit, axis=1, keepdims=True)
    c = 0.99995
    ref = (c * sib + np.sqrt(1 - c * c) * jit).astype(np.float32)
    ref[::5] = base                                              # the first enrolment is the clean one
    cand = rng.standard_normal((n_cand, dim)).astype(np.float32)
    hit = rng.integers(0, n_id, n_cand // 2)
    noise = rng.standard_normal((len(hit), dim)).astype(np.float32)
    cand[::2][: len(hit)] = base[hit] + np.float32(0.6 / np.sqrt(dim)) * noise      # cos ~ 0.86 to its identity
    sample = rng.choice(n_cand, 3000, replace=False)
    res = _check_cosine(ops, ref, cand, 0.5, sample=sample)
    st = res.stats
    assert st["part_rescans"] > n_cand // 4, st                  # every planted row has several leaders inside the window
    assert st["full_rescans"] < n_cand // 100, st                # ... and (nearly) none of them needs every reference


# ---------------------------------------------------------------- small galleries through the fused stage32 schedule (round 2)
@pytest.mark.parametrize("n_ref,n_cand,dim,offload", [
    (128, 75_776 + 77, 128, "auto"), (128, 113_704, 128, "1"), (64, 76_000, 72, "auto"), (32, 80_000, 128, "1"),
    (300, 80_000, 100, "auto"), (384, 77_000, 128, "auto"), (384, 77_000, 128, "0"), (129, 76_001, 96, "1"), (200, 151_552 + 129, 128, "auto")])
def test_small_galleries_fused(ops, ffr_env, n_ref, n_cand, dim, offload):
    """<= 128 live references in a tile leave the peer CTA's half of the B tile (and, for ragged candidate counts, of the A /
    staging boxes) entirely past the end of its tensor.  Such TMA boxes are never issued as they stand (measured: 4-5 x the
    tile time, and a launch failure with the offloaded tail): the last in-bounds rows are loaded instead, dead column groups
    (rows of 68..96 floats) are zeroed once.  Both forms of the stage32 tail, exact parity bar."""
    if offload != "auto":
        ffr_env.setenv("FFR_TAIL_OFFLOAD", offload)
    ref, cand = oracle.make_synthetic(n_ref, n_cand, dim, seed=n_ref + dim, n_adversarial=300, n_dup_refs=min(8, n_ref // 4),
                                      unit_norm=False)
    rng = np.random.default_rng(1)
    sample = rng.choice(n_cand, 6000, replace=False)
    sample = np.unique(np.concatenate([sample, np.arange(n_cand - 300, n_cand)]))          # the ragged tail in full
    res = _check_cosine(ops, ref, cand, 0.5, sample=sample)
    assert res.stats["k2"]["normalise"].startswith("stage32"), res.stats


def test_host_pipeline_folds_duplicates_once_per_call(ops):
    """ffr_ctx_filter_host with a duplicate-heavy gallery: the fold runs once per call (not per chunk), every chunk's K2 scans
    the unique rows, and the answers equal the device path's (which equal the oracle's, test above)."""
    rng = np.random.default_rng(17)
    n_id, copies, dim, n_cand = 750, 8, 128, 340_000
    base = rng.standard_normal((n_id, dim)).astype(np.float32)
    ref = np.concatenate([base] * copies)[rng.permutation(n_id * copies)]
    cand = rng.standard_normal((n_cand, dim)).astype(np.float32)
    hit = rng.integers(0, n_id, n_cand // 2)
    cand[::2] = base[hit] + 0.35 * rng.standard_normal((n_cand // 2, dim)).astype(np.float32)
    hf = ops.HostFilter(device=0, max_ref=len(ref), chunk_cand=100_000, max_dim=dim)
    keep, idx, val = hf(ref, cand, 0.5)
    hf.close()
    res = ops.face_filter(torch.from_numpy(ref).cuda(), torch.from_numpy(cand).cuda(), 0.5, want_stats=True)
    assert res.stats["refs_scanned"] == n_id
    gap, _ = _top2_gap64(np.unique(ref, axis=0), cand[:3000])
    ok = gap > TIE_EPS
    assert np.array_equal(idx[:3000][ok], res.best_idx.cpu().numpy()[:3000][ok])
    assert np.array_equal(keep, res.keep.cpu().numpy())
    first = {}
    for i, r in enumerate(ref):
        first.setdefault(r.tobytes(), i)
    assert all(first[ref[j].tobytes()] == j for j in idx[:20_000:7])          # every reported index is a FIRST occurrence


def test_graphed_filter_replays_the_eager_result(ops):
    """GraphedFilter.capture: K1 -> K2 -> K3 (programmatic dependent launch edges included) replayed as one CUDA graph over the
    caller's tensors gives the eager call's outputs, also after the inputs changed in place."""
    ref, cand = oracle.make_synthetic(1000, 100_000, 128, seed=5, n_adversarial=500, n_dup_refs=10)
    r_t, c_t = torch.from_numpy(ref).cuda(), torch.from_numpy(cand).cuda()
    out = (torch.empty(len(cand), dtype=torch.uint8, device="cuda"), torch.empty(len(cand), dtype=torch.int32, device="cuda"),
           torch.empty(len(cand), dtype=torch.float32, device="cuda"))
    g = ops.GraphedFilter.capture(r_t, c_t, 0.5, out=out)
    assert g.launches == 3
    for trial in range(3):
        if trial:
            c_t.copy_(c_t.roll(trial * 12_345, dims=0))
        g.replay()
        torch.cuda.synchronize()
        got = [t.clone() for t in out]
        eager = ops.face_filter(r_t, c_t, 0.5)
        torch.cuda.synchronize()
        assert torch.equal(got[0], eager.keep) and torch.equal(got[1], eager.best_idx) and torch.equal(got[2], eager.best_val)


@pytest.mark.parametrize("n_cand", [200, 9_000, 18_944, 19_201, 37_889, 40_000, 75_776, 80_001])
def test_offloaded_tail_last_tile_both_forms(ops, ffr_env, n_cand):
    """stage32 with the offloaded tail (> 256 references, 128-d) has two forms of the end-of-tile work: the CTA's last
    candidate tile is merged + emitted by the epilogue warps themselves, every other tile by the helper warps.  Sizes (148
    SMs = 74 CTA pairs of 256-row tiles): one ragged tile for the whole grid, at most one tile per CTA pair (the helper warps
    then merge nothing at all), exactly one full tile per pair, a ragged last tile, two tiles per pair plus one row, two to
    three tiles, and the smallest size the dispatcher picks this schedule for by itself and one just above it (the smaller
    ones force it: FFR_FUSE_K1)."""
    if n_cand < 75_776:
        ffr_env.setenv("FFR_FUSE_K1", "1")
    ref, cand = oracle.make_synthetic(1000, n_cand, 128, seed=n_cand, n_adversarial=300, n_dup_refs=8, unit_norm=False)
    res = _check_cosine(ops, ref, cand, 0.5)
    assert res.stats["k2"]["normalise"] == "stage32+tail_offload", res.stats
    assert res.stats["refs_scanned"] == 1000, res.stats
