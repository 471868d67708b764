"""BASELINE.json configs[0] on the GPU: the CUDA `ClipMapper` fed the batches the original project's own FilesReader,
Runner and NumpyWriter formed over bench.py's dataset, its output written to the files that writer left — bench's
replay of tests/golden/reference_runner_trace.json (clip_retrieval/clip_inference/runner.py:27-62 calls `mapper(batch)` and hands
the dict to `writer`; worker.py:52-117 builds exactly these objects).  The written shards are compared row for row with
the fp32 oracle mapper applied to the same files in the partition order `runner.Sampler` defines, and loaded back
through `load_index`."""
import os

import numpy as np
import pytest

import bench
from oracle import clip_ref

pytestmark = pytest.mark.gpu


@pytest.mark.timeout(600)
def test_config0_reference_runner_drives_cuda_mapper(tmp_path):
    import torch
    from PIL import Image
    import clip_retrieval_b200 as m
    from clip_retrieval_b200.model import make_preprocess

    n, parts, bs = 100, 2, 32
    src = str(tmp_path / "images")
    bench.make_plumbing_dataset(src, n)
    mapper = m.ClipMapper(enable_image=True, enable_text=True, enable_metadata=False, use_mclip=False,
                          clip_model="synthetic:ViT-B/32", use_jit=True, mclip_model="", warmup_batch_size=bs)
    arch = mapper.model.arch
    pre = make_preprocess(arch.image_size)
    seen = {"image": 0, "text": 0}

    def cuda_mapper(batch, img, txt):
        mapper.enable_image, mapper.enable_text = img, txt
        if img:
            assert batch["image_tensor"].dtype == torch.float32 and tuple(batch["image_tensor"].shape[1:]) == (3, 224, 224)
            seen["image"] += batch["image_tensor"].shape[0]
        else:
            assert batch["text_tokens"].shape[1] == 77
            seen["text"] += batch["text_tokens"].shape[0]
        return mapper(batch)

    out = str(tmp_path / "out")
    bench.run_reference_runner(src, out, cuda_mapper, pre, bench.hashed_tokenizer, parts, bs)
    assert seen == {"image": n, "text": n}          # 100 = 32 + 18 per partition: short last batches included
    img, txt = bench.read_plumbing_output(out)
    assert len(img) == parts and len(txt) == parts
    assert all(a.dtype == np.float16 and a.shape == (n // parts, arch.embed_dim) for a in img + txt)

    cfg = clip_ref.CONFIGS["ViT-B/32"]
    sd = m.synthetic_state_dict(arch, seed=0)
    for p in range(parts):
        keys = ["%04d" % i for i in range(n)][p::parts]       # runner.Sampler over the sorted key list
        px = torch.stack([pre(Image.open(os.path.join(src, k + ".png"))) for k in keys])
        tk = bench.hashed_tokenizer([open(os.path.join(src, k + ".txt")).read() for k in keys])
        ci = 1 - clip_ref.cosine(img[p], clip_ref.mapper_image(sd, cfg, px))
        ct = 1 - clip_ref.cosine(txt[p], clip_ref.mapper_text(sd, cfg, tk))
        assert ci.max() <= 1e-3 and ct.max() <= 1e-3, (p, ci.max(), ct.max())
    norms = np.linalg.norm(np.concatenate(img + txt).astype(np.float32), axis=1)
    assert np.all(np.abs(norms - 1) < 2e-3)

    # the writer's output folder is what clip_back's load_index serves (a10): search it with its own rows
    idx = m.load_index(os.path.join(out, "out_image", "img_emb"))
    assert idx.ntotal == n
    allrows = np.concatenate(img).astype(np.float32)
    D, I = idx.search(allrows[:5], 3)
    assert list(I[:, 0]) == [0, 1, 2, 3, 4]
