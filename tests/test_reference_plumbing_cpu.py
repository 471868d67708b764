"""BASELINE.json configs[0] — "ViT-B/32 clip_inference on 100 synthetic 224^2 images + captions, CPU ref
(plumbing)" — bench.run_reference_runner's replay of what the ORIGINAL project's own reader, runner and
writer did with this dataset (tests/golden/reference_runner_trace.json, recorded by
tests/golden/make_reference_golden.py), with the oracle's ViT-B/32 encoders (seeded weights) behind the mapper
glue that tests/test_oracle_cpu.py pins on the original `ClipMapper.__call__`.  What it pins:
  * the `preprocess` object `clip_retrieval_b200.load_clip` returns builds the batches the original `FilesReader`
    yielded (fields, dtypes, shapes);
  * the batch dict is the one the mapper contract (SURVEY §8b B1) describes;
  * the writer's shard layout (`img_emb/img_emb_{i}.npy`, fp16, partition order) is what
    `clip_retrieval_b200.load_index` enumerates, row for row.
The GPU mapper itself is tested against the same oracle in tests/test_embed_gpu.py."""
import os

import numpy as np
import torch

import bench


def _synthetic_tokenizer(texts):
    """Stands in for the BPE tokenizer (its vocabulary file is not available offline): SOT, hashed ids, EOT."""
    out = torch.zeros(len(texts), 77, dtype=torch.int64)
    for i, t in enumerate(texts):
        ids = [1 + (hash_ % 49000) for hash_ in (sum(w.encode()) * 31 + j for j, w in enumerate(t.split()))][:75]
        out[i, 0] = 49406
        out[i, 1:1 + len(ids)] = torch.tensor(ids, dtype=torch.int64)
        out[i, 1 + len(ids)] = 49407
    return out


def test_config0_plumbing_reference_reader_runner_writer(tmp_path):
    from PIL import Image
    from oracle import clip_ref
    from clip_retrieval_b200.index import list_embedding_shards
    from clip_retrieval_b200.model import make_preprocess

    n = 100
    rng = np.random.default_rng(0)
    src = tmp_path / "images"
    src.mkdir()
    for i in range(n):
        h, w = (224, 224) if i % 3 == 0 else (200 + i, 260 + (i * 7) % 90)
        Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).save(src / f"{i:04d}.png")
        (src / f"{i:04d}.txt").write_text(f"a photo of object {i}")

    cfg = clip_ref.CONFIGS["ViT-B/32"]
    sd = clip_ref.make_state_dict(cfg, seed=0)
    seen = {"image": 0, "text": 0}

    def mapper(batch, img, txt):
        if img:
            assert batch["image_tensor"].dtype == torch.float32 and tuple(batch["image_tensor"].shape[1:]) == (3, 224, 224)
            assert len(batch["image_filename"]) == batch["image_tensor"].shape[0]
            seen["image"] += batch["image_tensor"].shape[0]
        else:
            assert batch["text_tokens"].shape[1] == 77 and len(batch["text"]) == batch["text_tokens"].shape[0]
            seen["text"] += batch["text_tokens"].shape[0]
        return {"image_embs": clip_ref.mapper_image(sd, cfg, batch["image_tensor"]) if img else None,
                "text_embs": clip_ref.mapper_text(sd, cfg, batch["text_tokens"]) if txt else None,
                "image_filename": batch["image_filename"] if img else None, "text": batch["text"] if txt else None,
                "metadata": None}

    # The original FilesReader keys files by relative path INCLUDING the extension (reader.py:17-32), so image and
    # caption keys never intersect; its own tests read images only (test_reader.py:39).  The recorded job is one pass
    # over the images and one over the captions, two output partitions each.
    parts = 2
    bench.run_reference_runner(str(src), str(tmp_path), mapper, make_preprocess(224), _synthetic_tokenizer, parts, 32)
    assert seen == {"image": n, "text": n}

    shards = list_embedding_shards(str(tmp_path / "out_image" / "img_emb"))
    assert [os.path.basename(f) for f in shards] == ["img_emb_0.npy", "img_emb_1.npy"]
    rows = [np.load(f) for f in shards]
    assert all(r.dtype == np.float16 and r.shape == (50, 512) for r in rows)
    texts = [np.load(f) for f in list_embedding_shards(str(tmp_path / "out_text" / "text_emb"))]
    assert all(t.dtype == np.float16 and t.shape == (50, 512) for t in texts)
    # partition p holds samples p, p+2, ... of the sorted key list (runner.Sampler): check against the oracle mapper
    pre = make_preprocess(224)
    for p in range(parts):
        keys = [f"{i:04d}" for i in range(n)][p::parts]
        px = torch.stack([pre(Image.open(src / f"{k}.png")) for k in keys[:4]])
        # (batch of 32 in the run vs 4 here: the CPU GEMM blocks differently, so fp16-ulp differences are allowed)
        np.testing.assert_allclose(rows[p][:4].astype(np.float32), clip_ref.mapper_image(sd, cfg, px).astype(np.float32), atol=3e-4)
        tk = _synthetic_tokenizer([(src / f"{k}.txt").read_text() for k in keys[:4]])
        np.testing.assert_allclose(texts[p][:4].astype(np.float32), clip_ref.mapper_text(sd, cfg, tk).astype(np.float32), atol=3e-4)
    norms = np.linalg.norm(np.concatenate(rows + texts).astype(np.float32), axis=1)
    assert np.all(np.abs(norms - 1) < 2e-3)
