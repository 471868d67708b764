"""bench.py contract on the CPU: the reference arm prints exactly one JSON line on stdout with the keys
the driver reads, and library chatter cannot reach stdout."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, WORLD_SIZE="1", RANK="0")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-sample", "2"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["unit"] == "pairs/s" and j["higher_is_better"] is True
    assert j["value"] > 0 and j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0
    for key in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config"):
        assert key in j
    assert j["steps"] == 1


def test_steps_below_one_are_rejected():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps" in r.stderr and r.stdout.strip() == ""


def test_dump_outputs_stays_within_its_budget(tmp_path):
    """--dump-outputs: float32 / float64 files, a seeded row sample (with its row numbers) of an array over the
    per-array cap, 1-D arrays included, and never more bytes on disk than the budget it is given."""
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench

    big = np.random.default_rng(1).standard_normal((4096, 1024)).astype(np.float16)
    ids = np.arange(3_000_000, dtype=np.int64)
    used = bench.dump_outputs(str(tmp_path), "w", {"embs": big, "I": ids}, 6 << 20)
    files = {f: os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)}
    assert used == sum(files.values()) <= 6 << 20
    e, rows = np.load(tmp_path / "w_embs.npy"), np.load(tmp_path / "w_embs_rows.npy")
    assert e.dtype == np.float32 and rows.dtype == np.float64 and np.array_equal(e, big[rows.astype(np.int64)].astype(np.float32))
    i, irows = np.load(tmp_path / "w_I.npy"), np.load(tmp_path / "w_I_rows.npy")
    assert i.dtype == np.float64 and np.array_equal(i, irows)
    again = tmp_path / "again"
    bench.dump_outputs(str(again), "w", {"embs": big}, 6 << 20)
    assert np.array_equal(np.load(again / "w_embs_rows.npy"), rows)      # the same rows from run to run


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, WORLD_SIZE="2", RANK="1", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_plumbing_helpers_drive_the_reference_runner(tmp_path):
    """configs[0] helpers of bench.py on the CPU: the synthetic tokenizer ends every caption with the largest id (the
    text tower pools at argmax), and a ClipMapper-contract callable driven through bench's replay of the original
    project's own Runner job (tests/golden/reference_runner_trace.json) produces the writer's shard layout in the
    sampler's order."""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    tok = bench.hashed_tokenizer(["a photo of object 3", "", "x " * 200])
    assert tok.shape == (3, 77) and tok.dtype == torch.int64
    assert all(int(row.argmax()) == int((row != 0).sum()) - 1 and int(row.max()) == 49407 and int(row[0]) == 49406 for row in tok)
    from clip_retrieval_b200.model import make_preprocess

    n, parts, bs, d = 10, 2, 4, 16
    src = str(tmp_path / "images")
    bench.make_plumbing_dataset(src, n)
    calls = []

    def fake_mapper(batch, img, txt):
        b = batch["image_tensor"].shape[0] if img else batch["text_tokens"].shape[0]
        calls.append((img, b))
        # embedding = the sample's number taken from its file name / caption, so the order can be checked in the shards
        keys = batch["image_filename"] if img else batch["text"]
        ids = [int(os.path.basename(k).split(".")[0]) if img else int(k.split()[-1]) for k in keys]
        e = np.repeat(np.asarray(ids, dtype=np.float16)[:, None], d, axis=1)
        return {"image_embs": e if img else None, "text_embs": e if txt else None,
                "image_filename": batch["image_filename"] if img else None, "text": batch["text"] if txt else None, "metadata": None}

    sec = bench.run_reference_runner(src, str(tmp_path / "out"), fake_mapper, make_preprocess(224), bench.hashed_tokenizer, parts, bs)
    assert sec >= 0 and sum(b for img, b in calls if img) == n and sum(b for img, b in calls if not img) == n
    img, txt = bench.read_plumbing_output(str(tmp_path / "out"))
    for shards in (img, txt):
        assert len(shards) == parts and all(s.dtype == np.float16 and s.shape == (n // parts, d) for s in shards)
        for p in range(parts):   # runner.Sampler: partition p holds samples p, p + parts, ...
            assert list(shards[p][:, 0].astype(int)) == list(range(n))[p::parts]
