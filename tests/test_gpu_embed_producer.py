"""SURVEY §8f row 3 / §8a row a3 on the GPU: the device-side embedding producer (batched nvJPEG decode, GPU resize +
standardisation, embeddings handed to the filter without leaving the device) behind the drop-in entry point, driven by a
small torch module with the ``embed`` contract of ``MobileFaceNetModel`` (the reference's own MobileFaceNet class is not
part of this repository; its adapter is covered in tests/test_cabi_and_host.py).

Replaces, for models that accept CUDA tensors, the reference's per-image host pipeline
(similar_face_filtering/filter_faces_using_reference.py:60-68), its batch-1 reference embedding (:77-84) and the
NumPy hand-over of every batch (:168-184)."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import oracle

pytestmark = pytest.mark.gpu


class TinyEmbedNet(torch.nn.Module):
    """[b, H, W, 3] standardised float32 -> [b, 128] float32; ``embed`` keeps everything on the device,
    ``predict`` is the reference's NumPy contract (:84,184)."""
    inputs, outputs = "[b,160,160,3]", "[b,128]"

    def __init__(self, device):
        super().__init__()
        g = torch.Generator().manual_seed(7)
        self.conv = torch.nn.Conv2d(3, 8, 5, stride=4, padding=2)
        self.fc = torch.nn.Linear(8 * 10 * 10, 128)
        with torch.no_grad():
            for p in self.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * 0.05)
        self.dev = torch.device(device)
        self.to(self.dev).eval()
        self.embed_calls, self.predict_calls, self.batch_sizes = 0, 0, []

    @torch.no_grad()
    def embed(self, batch):
        assert isinstance(batch, torch.Tensor) and batch.is_cuda, "the device branch must hand over CUDA tensors"
        self.embed_calls += 1
        self.batch_sizes.append(batch.shape[0])
        x = torch.relu(self.conv(batch.permute(0, 3, 1, 2)))
        x = torch.nn.functional.adaptive_avg_pool2d(x, (10, 10)).flatten(1)
        return self.fc(x)

    def predict(self, batch, verbose=0):
        self.predict_calls += 1
        x = torch.as_tensor(np.asarray(batch), dtype=torch.float32, device=self.dev)
        calls, sizes = self.embed_calls, list(self.batch_sizes)
        out = self.embed(x).cpu().numpy()
        self.embed_calls, self.batch_sizes = calls, sizes
        return out


def _make_dataset(root, rng, classes=("alice", "bob", "carol"), n_ref=12, n_cand=40):
    from PIL import Image
    sizes = [(24, 20), (30, 30), (20, 28)]
    for cls_i, cls in enumerate(classes):
        base = rng.integers(0, 255, (24, 20, 3))
        for kind, n in (("ref", n_ref), ("unf", n_cand)):
            d = os.path.join(root, kind, cls)
            os.makedirs(d)
            for i in range(n):
                pattern = base if (kind == "ref" or i % 3) else rng.integers(0, 255, (24, 20, 3))
                img = np.clip(pattern + rng.normal(0, 25, pattern.shape), 0, 255).astype(np.uint8)
                hh, ww = sizes[i % 3]                                            # variable image sizes, like the bundled faces
                img = np.kron(img[:hh, :ww] if hh <= 24 and ww <= 20 else np.resize(img, (hh, ww, 3)), np.ones((8, 8, 1), dtype=np.uint8))
                # 4:4:4 (no chroma subsampling): the two decoders then differ by IDCT rounding only; with 4:2:0 their
                # chroma UPSAMPLING filters differ too (libjpeg's "fancy" triangle filter vs nvJPEG's), which on these
                # random 8 x 8 colour blocks is a few per cent of the dynamic range at every block edge
                Image.fromarray(img).save(os.path.join(d, f"{i:03d}.jpg"), quality=95, subsampling=0)
    return os.path.join(root, "unf"), os.path.join(root, "ref")


def test_device_preprocess_matches_host(tmp_path, cuda_dev):
    """nvJPEG decode + GPU resize / standardise == PIL decode + read_and_preprocess_img up to the two decoders' IDCT
    rounding (a level or two of 255 on a few pixels)."""
    from face_detection_and_recognition_b200.filter_faces_using_reference import (read_and_preprocess_batch_device,
                                                                                  read_and_preprocess_img)
    rng = np.random.default_rng(3)
    ud, _ = _make_dataset(str(tmp_path), rng, classes=("x",), n_ref=1, n_cand=9)
    paths = sorted(glob.glob(os.path.join(ud, "x", "*.jpg")))
    dev_batch = read_and_preprocess_batch_device(paths, cuda_dev).cpu()
    host = torch.stack([read_and_preprocess_img(p) for p in paths])
    assert dev_batch.shape == host.shape == (9, 160, 160, 3)
    diff = (dev_batch - host).abs()
    assert diff.mean().item() < 2e-2 and diff.max().item() < 0.25, (diff.mean().item(), diff.max().item())
    np.testing.assert_allclose(dev_batch.mean(dim=(1, 2, 3)).numpy(), 0, atol=1e-4)
    np.testing.assert_allclose(dev_batch.std(dim=(1, 2, 3), unbiased=False).numpy(), 1, atol=1e-3)


def test_embed_paths_device_branch(tmp_path, ffr_lib, cuda_dev):
    from face_detection_and_recognition_b200.filter_faces_using_reference import _embed_paths, _embed_paths_device
    rng = np.random.default_rng(4)
    ud, _ = _make_dataset(str(tmp_path), rng, classes=("x",), n_ref=1, n_cand=50)
    paths = sorted(glob.glob(os.path.join(ud, "x", "*.jpg")))
    model = TinyEmbedNet(cuda_dev)
    stats = {}
    emb = _embed_paths_device(model, paths, 16, cuda_dev, stats=stats)
    assert emb.is_cuda and emb.shape == (50, 128) and model.embed_calls == 4 and model.predict_calls == 0
    assert "nvJPEG" in stats["decoder"] and stats["images"] == 50
    host = _embed_paths(model, paths, 16)                    # PIL + NumPy hand-over (the reference's contract)
    cos = torch.nn.functional.cosine_similarity(emb.cpu(), torch.from_numpy(host), dim=1)
    assert cos.min().item() > 0.999, cos.min().item()


def test_main_device_resident_model(tmp_path, capsys, ffr_lib, cuda_dev):
    """The drop-in's main() with a model that offers ``embed``: batched reference embedding, device-side decode, the
    embeddings never leave the GPU -- and the clean / unclean tree equals the oracle's decisions on the same embeddings."""
    from face_detection_and_recognition_b200.filter_faces_using_reference import _embed_paths_device, main
    rng = np.random.default_rng(5)
    ud, rd = _make_dataset(str(tmp_path), rng)
    td = str(tmp_path / "out")
    model = TinyEmbedNet(cuda_dev)
    main(["--ud", ud, "--rd", rd, "--td", td, "-b", "16", "-r", "8"], model=model)
    out = capsys.readouterr().out
    assert model.predict_calls == 0 and model.embed_calls > 0
    assert model.batch_sizes[:3] == [8, 8, 8]                # references: ONE batch per class, not eight batch-1 calls
    for cls in ("alice", "bob", "carol"):
        refs = sorted(glob.glob(os.path.join(rd, cls, "*.jpg")))[:8]
        cands = sorted(glob.glob(os.path.join(ud, cls, "*.jpg")))
        r_emb = _embed_paths_device(model, refs, 8, cuda_dev).cpu().numpy()
        c_emb = _embed_paths_device(model, cands, 16, cuda_dev).cpu().numpy()
        mu, thres = oracle.ref_mean_vec_and_thres(r_emb[:, None, :], 8)
        keep = oracle.euclid_keep_literal(c_emb, mu, thres)
        d = np.linalg.norm(c_emb - mu, axis=1)
        n_clean = 0
        for p, k, dist in zip(cands, keep, d):
            name = os.path.basename(p)
            in_clean = os.path.exists(os.path.join(td, "clean", cls, name))
            assert in_clean != os.path.exists(os.path.join(td, "unclean", cls, name))
            n_clean += in_clean
            if abs(dist - thres) > 1e-4 * max(1.0, thres):
                assert in_clean == bool(k), f"{cls}/{name}: dist {dist} thres {thres}"
        assert f"positive={n_clean}, total={len(cands)}" in out


def test_gallery_mode_device_resident_model(tmp_path, ffr_lib, cuda_dev):
    from face_detection_and_recognition_b200.filter_faces_using_reference import _embed_paths_device, main
    rng = np.random.default_rng(6)
    ud, rd = _make_dataset(str(tmp_path), rng, classes=("dave",), n_ref=12, n_cand=30)
    td = str(tmp_path / "out")
    model = TinyEmbedNet(cuda_dev)
    main(["--ud", ud, "--rd", rd, "--td", td, "--gallery", "--threshold", "0.6", "-r", "12"], model=model)
    refs = sorted(glob.glob(os.path.join(rd, "dave", "*.jpg")))
    cands = sorted(glob.glob(os.path.join(ud, "dave", "*.jpg")))
    r_emb = _embed_paths_device(model, refs, 32, cuda_dev).cpu().numpy()
    c_emb = _embed_paths_device(model, cands, 32, cuda_dev).cpu().numpy()
    ko, io, so = oracle.filter_cosine(r_emb, c_emb, 0.6)
    for p, k, s in zip(cands, ko, so):
        if abs(s - 0.6) > 1e-3:
            assert os.path.exists(os.path.join(td, "clean" if k else "unclean", "dave", os.path.basename(p)))


def test_main_classes_over_two_gpus(tmp_path, capsys, ffr_lib, cuda_dev):
    """--ngpus 2: the reference's per-class loop (:161) is the embarrassingly parallel axis -- class i runs on GPU i mod 2
    with its own model replica; tree and summary lines equal the single-GPU run's."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from face_detection_and_recognition_b200.filter_faces_using_reference import main
    rng = np.random.default_rng(8)
    ud, rd = _make_dataset(str(tmp_path), rng, classes=("a", "b", "c", "d", "e"))
    outs = []
    for n, td in ((1, str(tmp_path / "o1")), (2, str(tmp_path / "o2"))):
        main(["--ud", ud, "--rd", rd, "--td", td, "-b", "16", "-r", "8", "--ngpus", str(n)], model_factory=lambda d: TinyEmbedNet(d))
        text = capsys.readouterr().out
        outs.append((sorted(l for l in text.splitlines() if l.startswith("Similar images")),
                     sorted(os.path.relpath(p, td) for p in glob.glob(os.path.join(td, "*", "*", "*.jpg")))))
    assert outs[0] == outs[1] and len(outs[0][0]) == 5
