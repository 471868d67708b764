"""Generate tests/golden/reference_calls.npz + reference_runner_trace.json: what the original clip-retrieval code
returns for the inputs of the tests that compare against it, so that those tests run without a checkout of it.

    python tests/golden/make_reference_golden.py <clip-retrieval checkout>

The original's functions are loaded from the checkout and run unmodified; only their results are stored:
  * clip_back.py `KnnService.connected_components` / `get_violent_items` on seeded random graphs and embeddings
    (tests/test_oracle_cpu.py::test_postfilter_oracle_matches_reference_functions);
  * clip_inference/mapper.py `ClipMapper.__call__` with the oracle's tiny encoders standing in for the model: the fp32
    features it was handed and the dict it returned (::test_mapper_glue_matches_reference_call);
  * clip_back.py `KnnService.knn_search` + `post_filter` + `normalized` over the oracle's flat index
    (::test_index_contract_through_reference_knn_search);
  * clip_inference reader.py / runner.py / writer.py (`FilesReader`, `Runner`, `NumpyWriter`) over bench.py's plumbing
    dataset: the batches the reader hands the mapper (keys, tensor shapes and dtypes, sample files in order) and the
    files the writer leaves (path, dtype, shape, which sample each row holds), for the (samples, partitions, batch)
    shapes bench.py and the plumbing tests run (reference_runner_trace.json; replayed by bench.run_reference_runner).
"""
import ast
import contextlib
import importlib.util
import json
import os
import sys
import tempfile
import textwrap
import types
from collections import defaultdict

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from oracle import clip_ref, knn_ref, postfilter_ref, synth_ref  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
RUNNER_SHAPES = [(100, 2, 32), (10, 2, 4)]   # (samples, output partitions, batch size)


def _functions(path, cls_name, names, ns):
    src = open(path).read()
    tree = ast.parse(src)
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in names:
            exec(ast.get_source_segment(src, node), ns)
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == cls_name)
    for node in cls.body:
        if isinstance(node, ast.FunctionDef) and node.name in names:
            exec(textwrap.dedent(ast.get_source_segment(src, node)), ns)
    return ns


def postfilter_calls(back, out):
    fns = _functions(back, "KnnService", ("connected_components", "get_violent_items"), {"np": np})
    rng = np.random.default_rng(0)
    for trial in range(20):
        k = int(rng.integers(2, 60))
        A = rng.random((k, k)) < 0.05
        A = A | A.T | np.eye(k, dtype=bool)
        neigh = defaultdict(list)
        for i in range(k):
            for j in np.nonzero(A[i])[0]:
                neigh[int(i)].append(int(j))
        groups = fns["connected_components"](None, neigh)
        out["cc_adjacency_%d" % trial] = A
        out["cc_groups_%d" % trial] = np.concatenate([np.asarray(g, np.int64) for g in groups])
        out["cc_group_sizes_%d" % trial] = np.array([len(g) for g in groups], np.int64)
    E = rng.standard_normal((200, 64)).astype(np.float32)
    P = rng.standard_normal((3, 64)).astype(np.float32)
    out["violent_embeddings"], out["violent_prompts"] = E, P
    out["violent_items"] = np.asarray(fns["get_violent_items"](None, P, E), np.int64)


def mapper_call(mapper_py, out):
    ns = _functions(mapper_py, "ClipMapper", ("__call__",), {"torch": torch, "np": np})
    cfg = clip_ref.CONFIGS["tiny"]
    sd = clip_ref.make_state_dict(cfg, seed=0)
    px = clip_ref.synth_images(5, cfg, seed=1)
    tk = clip_ref.synth_tokens(5, cfg, seed=1)
    fi, ft = clip_ref.encode_image(sd, cfg, px), clip_ref.encode_text(sd, cfg, tk)
    me = types.SimpleNamespace(enable_image=True, enable_text=True, enable_metadata=True, use_mclip=False, device="cpu",
                               model_img=lambda x: fi.clone(), model_txt=lambda x: ft.clone())
    item = {"image_tensor": px, "text_tokens": tk, "image_filename": list("abcde"), "text": list("vwxyz"), "metadata": list("12345")}
    r = ns["__call__"](me, item)
    out["mapper_image_features"], out["mapper_text_features"] = fi.numpy(), ft.numpy()
    out["mapper_image_embs"], out["mapper_text_embs"] = r["image_embs"], r["text_embs"]
    out["mapper_keys"] = np.array(list(r))
    out["mapper_passthrough"] = np.array([r["image_filename"], r["text"], r["metadata"]])


def knn_search_calls(back, out):
    timer = types.SimpleNamespace(time=lambda: contextlib.nullcontext())
    ns = _functions(back, "KnnService", ("normalized", "knn_search", "post_filter", "connected_components_dedup"),
                    {"np": np, "KNN_INDEX_TIME": timer, "DEDUP_TIME": timer, "SAFETY_TIME": timer})
    d, n = 64, 30
    X = synth_ref.rows_f16(n, d)
    X[7] = X[3]
    index = types.SimpleNamespace(search_and_reconstruct=lambda q, k: knn_ref.flat_search_and_reconstruct(X, q, k))
    svc = types.SimpleNamespace(get_non_uniques=lambda emb, threshold=0.94: postfilter_ref.get_non_uniques(emb, threshold))
    svc.connected_components_dedup = lambda emb: ns["connected_components_dedup"](svc, emb)
    svc.post_filter = lambda *a: ns["post_filter"](svc, *a)
    res = types.SimpleNamespace(image_index=index, text_index=index, metadata_is_ordered_by_ivf=False, safety_model=None,
                                violence_detector=None)
    q = X[3:4].astype(np.float32)
    for name, dedup in (("knn", False), ("knn_dedup", True)):
        dist, ind = ns["knn_search"](svc, q, "image", 40, res, dedup, False, False)
        out[name + "_distances"] = np.asarray(dist, np.float32)
        out[name + "_indices"] = np.asarray(ind, np.int64)


def runner_trace(inference, n, parts, bs):
    def load(name):
        spec = importlib.util.spec_from_file_location("ref_" + name, os.path.join(inference, name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    from clip_retrieval_b200.model import make_preprocess

    reader, runner, writer = load("reader"), load("runner"), load("writer")

    class Logger:
        def start(self): pass
        def end(self): pass
        def __call__(self, stats): pass

    with tempfile.TemporaryDirectory() as tmp:
        src, out_root = os.path.join(tmp, "images"), os.path.join(tmp, "out")
        bench.make_plumbing_dataset(src, n)
        runs = []
        for modality in ("image", "text"):
            img, txt = modality == "image", modality == "text"
            out = os.path.join(out_root, "out_" + modality)
            for p in range(parts):
                batches = []

                def mapper(batch, img=img, txt=txt, batches=batches):
                    files = batch["image_filename"] if img else None
                    ids = [int(os.path.basename(f).split(".")[0]) for f in files] if img else [int(t.split()[-1]) for t in batch["text"]]
                    batches.append({"fields": {k: ([str(v.dtype), list(v.shape)] if torch.is_tensor(v) else type(v).__name__)
                                               for k, v in sorted(batch.items())},
                                    "samples": ids,
                                    "image_filename": [os.path.relpath(f, src) for f in files] if img else None,
                                    "text": list(batch["text"]) if txt else None})
                    e = np.repeat(np.asarray(ids, dtype=np.float16)[:, None], 16, axis=1)
                    return {"image_embs": e if img else None, "text_embs": e if txt else None,
                            "image_filename": files, "text": batch["text"] if txt else None, "metadata": None}

                run = runner.Runner(
                    reader_builder=lambda sampler, img=img, txt=txt: reader.FilesReader(
                        sampler, make_preprocess(224), bench.hashed_tokenizer, src, bs, 0, enable_text=txt, enable_image=img,
                        enable_metadata=False),
                    mapper_builder=lambda mapper=mapper: mapper,
                    writer_builder=lambda i, out=out, img=img, txt=txt: writer.NumpyWriter(
                        partition_id=i, output_folder=out, enable_text=txt, enable_image=img, enable_metadata=False,
                        output_partition_count=parts),
                    logger_builder=lambda i: Logger(),
                    output_partition_count=parts)
                run(p)
                runs.append({"modality": modality, "partition": p, "batches": batches})
        files = []
        for dirpath, _, names in os.walk(out_root):
            for f in sorted(names):
                path = os.path.join(dirpath, f)
                rel = os.path.relpath(path, out_root)
                entry = {"path": rel}
                if f.endswith(".npy"):
                    a = np.load(path)
                    entry.update(dtype=str(a.dtype), shape=list(a.shape), samples=[int(v) for v in a[:, 0]])
                files.append(entry)
        files.sort(key=lambda e: e["path"])
    return {"samples": n, "partitions": parts, "batch_size": bs, "runs": runs, "files": files}


def main():
    ref = os.path.abspath(sys.argv[1])
    back = os.path.join(ref, "clip_retrieval", "clip_back.py")
    inference = os.path.join(ref, "clip_retrieval", "clip_inference")
    out = {}
    postfilter_calls(back, out)
    mapper_call(os.path.join(inference, "mapper.py"), out)
    knn_search_calls(back, out)
    path = os.path.join(GOLDEN, "reference_calls.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")
    trace = [runner_trace(inference, *shape) for shape in RUNNER_SHAPES]
    path = os.path.join(GOLDEN, "reference_runner_trace.json")
    with open(path, "w") as f:
        json.dump(trace, f, indent=0, sort_keys=True)
        f.write("\n")
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
