"""bench.py's reference arm runs on CPU: check the JSON contract of the line it prints (one line on stdout, the keys
the driver reads).  The GPU arm prints the same keys plus roofline / clocks / gpu_launches (checked on the GPU box by
the round-end run itself)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--entities", "3000", "--edges", "50000", "--relations", "8"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1                                   # exactly one JSON line on stdout
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["unit"] == "edges/s" and j["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data",
                "config", "cpu_baseline", "e2e"):
        assert key in j, key
    assert j["value"] > 0 and j["vs_baseline"] is None and j["data"] == "synthetic" and "workload" in j["config"]
    cb, e2e = j["cpu_baseline"], j["e2e"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == j["value"] and "sample" in cb
    assert e2e["value"] == j["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_rejects_zero_steps_and_dump_of_the_reference_arm(tmp_path):
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "out")]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args],
                             capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", args
    assert not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_dump_outputs_match_the_pass_and_repeat_across_runs(tmp_path):
    """Two runs with 1 and 3 timed steps: the timed region issues 3x the launches of the one-step run, both dumps hold
    the same sample of the same inputs' outputs, and that sample equals what the drop-in computes in this process for
    the inputs bench.py builds (update_att + gat_embeddings), so the dump is neither a stale A_in nor another tensor."""
    import argparse
    import torch
    import bench
    import literalkg_b200 as L
    n, e, n_rel = 60000, 1500000, 8
    small = ["--entities", str(n), "--edges", str(e), "--relations", str(n_rel), "--warmup", "1", "--no-cpu-baseline",
             "--no-scoring", "--no-training"]
    runs = []
    for steps in (1, 3):
        d = tmp_path / f"steps{steps}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), *small,
                              "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        j = json.loads(out.stdout)
        assert j["steps"] == steps
        runs.append((j, {p.stem: np.load(p) for p in d.glob("*.npy")}))
    (j1, a), (j3, b) = runs
    assert j1["gpu_launches"] > 0 and j3["gpu_launches"] == 3 * j1["gpu_launches"]
    assert sorted(a) == ["attention_indices", "attention_values", "embedding_rows", "embeddings"]
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    rows, idx, vals = a["embedding_rows"], a["attention_indices"], a["attention_values"]
    nnz = j1["config"]["unique_pairs"]
    assert 0 < len(rows) < n and len(vals) < nnz                    # this graph is larger than the sample
    assert np.array_equal(rows, np.unique(rows)) and rows[0] >= 0 and rows[-1] < n
    assert a["embeddings"].shape[0] == len(rows) and idx.shape == (2, len(vals))
    for k in ("embedding_rows", "attention_indices"):
        assert np.array_equal(a[k], b[k]), k
    for k in ("embeddings", "attention_values"):
        np.testing.assert_allclose(a[k], b[k], rtol=1e-5, atol=1e-6, err_msg=k)

    # the same pass in this process, on the inputs run_ours builds
    dev = torch.device("cuda:0")
    cfg = bench.oracle_config(argparse.Namespace(layers=3, aggregator="bi-interaction"))
    kg = L.synthetic.make_kg(n, e, n_rel)
    num, txt = L.synthetic.make_literals(n, device=dev)
    args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    args.device = str(dev)
    torch.manual_seed(2022)
    m = L.LiteralKG(args, n, n_rel, None, num, txt).to(dev).eval()
    h, t, r = (torch.from_numpy(x.astype(np.int32)).to(dev) for x in (kg.h, kg.t, kg.r))
    with torch.no_grad():
        m(h, t, r, list(range(n_rel)), device=dev, mode="update_att")
        emb = m.gat_embeddings(gather=False)
    assert m.A_in.data._nnz() == nnz
    np.testing.assert_allclose(a["embeddings"], emb[torch.from_numpy(rows.astype(np.int64)).to(dev)].cpu().numpy(),
                               rtol=1e-5, atol=1e-6)
    ai = m.A_in.data._indices().cpu().numpy()
    keys = ai[0] * n + ai[1]                                        # coalesced: sorted by (head, tail)
    want = idx[0].astype(np.int64) * n + idx[1].astype(np.int64)
    pos = np.searchsorted(keys, want)
    assert np.array_equal(keys[pos], want)
    np.testing.assert_allclose(vals, m.A_in.data._values().cpu().numpy()[pos], rtol=1e-5, atol=1e-9)
