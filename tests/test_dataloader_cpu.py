"""Host side of the data layer (SURVEY.md 8(a) rows a1, a3): file readers against the oracle's restatement of the
reference loader, on synthetic files and -- where the reference checkout is mounted -- on its bundled data/Test."""
import os

import numpy as np
import pytest

import literalkg_oracle as O
from literalkg_b200 import dataloader as D

REF = os.environ.get("LKG_REFERENCE", "")         # a checkout of the original NSLab-CUK/LiteralKG, where available
REF_DATA = os.path.join(REF, "data", "Test")
NO_REF = "LKG_REFERENCE names no checkout of the original LiteralKG"


def _write(tmp_path, name, text):
    p = tmp_path / name
    p.write_text(text)
    return str(p)


def test_read_triples_dedup_keeps_first_occurrence_and_order(tmp_path):
    rng = np.random.default_rng(0)
    trip = rng.integers(0, 40, size=(500, 3))
    trip[:, 1] %= 5
    trip = np.concatenate([trip, trip[rng.integers(0, 500, 80)]])       # exact duplicate rows
    rng.shuffle(trip)
    text = "\n".join(f"{h} {r} {t}" for h, r, t in trip) + "\n"
    got = D.read_triples(_write(tmp_path, "kg.txt", text))
    h, t, r = O.parse_triples(text)
    assert np.array_equal(got[:, 0], h) and np.array_equal(got[:, 1], r) and np.array_equal(got[:, 2], t)
    assert D.relation_order(got[:, 1]) == O.relation_order(r)
    # ids too wide for one packed key take the row-wise path: same result
    big = trip.astype(np.int64)
    big[:, 0] += 1 << 40
    big[:, 2] += 1 << 41
    textb = "\n".join(f"{h} {r} {t}" for h, r, t in big) + "\n"
    gotb = D.read_triples(_write(tmp_path, "kg_big.txt", textb))
    hb, tb, rb = O.parse_triples(textb)
    assert np.array_equal(gotb[:, 0], hb) and np.array_equal(gotb[:, 2], tb) and np.array_equal(gotb[:, 1], rb)


def test_numeric_literals_match_the_oracle(tmp_path):
    age = "3\n0\t4.0\n2\t9.0\n7\t1.5\n2\t3.0\n"           # leading count line, a repeated id keeps its last value
    weight = "2\n2\t10.0\n5\t40.0\n"
    paths = [_write(tmp_path, "age_dict.txt", age), _write(tmp_path, "weight_dict.txt", weight)]
    table, max_id = D.read_numeric_literals(paths, 9, 2)
    assert max_id == 7 and table.shape == (9, 2)
    assert np.array_equal(table, O.numeric_literal_table([age, weight], 9, 2))
    assert table[2, 0] == 0 and table[2, 1] == np.float32(11.0 / 40.0)     # the later file resets the whole row


@pytest.mark.skipif(not REF or not os.path.exists(os.path.join(REF_DATA, "pre_training_train.txt")), reason=NO_REF)
def test_bundled_reference_data_dir():
    path = os.path.join(REF_DATA, "pre_training_train.txt")
    got = D.read_triples(path)
    h, t, r = O.parse_triples(open(path).read())
    assert np.array_equal(got[:, 0], h) and np.array_equal(got[:, 1], r) and np.array_equal(got[:, 2], t)
    import pandas as pd                                      # the reference's own load_graph (dataloader.py:186-190)
    ref = pd.read_csv(path, sep=" ", names=["h", "r", "t"], engine="python").drop_duplicates()
    assert np.array_equal(got, ref[["h", "r", "t"]].to_numpy())
    files = [os.path.join(REF_DATA, f) for f in ("age_dict.txt", "weight_dict.txt")]
    n = int(max(got[:, 0].max(), got[:, 2].max()) + 1)
    table, max_id = D.read_numeric_literals(files, n, 2)
    want = O.numeric_literal_table([open(f).read() for f in files], max(n, max_id + 1), 2)
    assert np.array_equal(table, want)


# ---- text-literal pickles + the whole data directory (dataloader.py:111-152, 405-438) ---------------------------------
def _make_dir(tmp_path, rng, text_dim=6):
    import pickle
    trip = np.unique(np.stack([rng.integers(0, 30, 200), rng.integers(0, 4, 200), rng.integers(0, 30, 200)], 1), axis=0)
    rng.shuffle(trip)
    (tmp_path / "pre_training_train.txt").write_text("\n".join(f"{h} {r} {t}" for h, r, t in trip) + "\n")
    (tmp_path / "age_dict.txt").write_text("4\n0\t4.0\n2\t9.0\n7\t1.5\n33\t2.0\n")          # id 33 is beyond the KG ids
    (tmp_path / "weight_dict.txt").write_text("2\n2\t10.0\n5\t40.0\n")
    cc = {3: rng.normal(size=text_dim), 2: rng.normal(size=text_dim), 40: rng.normal(size=text_dim)}   # 40: largest id
    memo = {3: rng.normal(size=text_dim), 9: rng.normal(size=text_dim)}                     # overrides entity 3
    for name, d in (("cc_dict.pickle", cc), ("memo_dict.pickle", memo)):
        with open(tmp_path / name, "wb") as fh:
            pickle.dump(d, fh)
    return trip, cc, memo


def test_data_dir_with_text_pickles(tmp_path):
    rng = np.random.default_rng(4)
    trip, cc, memo = _make_dir(tmp_path, rng)
    got_trip, num, txt = D.read_data_dir(str(tmp_path), numeric_dim=2, text_dim=6)
    assert np.array_equal(got_trip, trip)
    assert num.shape == (41, 2) and txt.shape == (41, 6)                      # n = largest literal id + 1
    assert np.allclose(txt[3], memo[3]) and np.allclose(txt[2], cc[2]) and np.allclose(txt[40], cc[40])
    assert np.allclose(txt[9], memo[9]) and not txt[0].any() and not txt[33].any()      # numeric-only entities: zero text
    assert not num[2].any() and not num[3].any()                              # entities of a pickle: numeric row zeroed
    assert num[0, 0] == np.float32(5.0 / 9.0) and num[5, 1] == np.float32(41.0 / 40.0) and num[33, 0] == np.float32(3.0 / 9.0)
    # single-literal configurations
    _, num_only, none_txt = D.read_data_dir(str(tmp_path), numeric_dim=2, text_dim=6, use_txt_lit=False)
    assert none_txt is None and num_only[2, 1] == np.float32(11.0 / 40.0)     # pickles are not read: row 2 survives
    _, none_num, txt_only = D.read_data_dir(str(tmp_path), numeric_dim=2, text_dim=6, use_num_lit=False)
    assert none_num is None and txt_only.shape == (41, 6) and np.allclose(txt_only[40], cc[40])


@pytest.mark.skipif(not REF or not os.path.exists(os.path.join(REF, "dataloader.py")), reason=NO_REF)
@pytest.mark.parametrize("use_num,use_txt", [(True, True), (True, False), (False, True)])
def test_data_dir_matches_the_reference_loader(tmp_path, use_num, use_txt):
    """The reference's own load_attributes / construct_data / embed_*_literal (dataloader.py:111-152, 369-438) run on a
    stub object over the same directory."""
    import argparse
    import sys
    import torch
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import dataloader as ref_dl
    rng = np.random.default_rng(7)
    _make_dir(tmp_path, rng)
    stub = ref_dl.DataLoader.__new__(ref_dl.DataLoader)
    stub.args = argparse.Namespace(use_num_lit=use_num, use_txt_lit=use_txt)
    stub.data_dir, stub.device = str(tmp_path), "cpu"
    stub.numeric_literal_files = ["age_dict.txt", "weight_dict.txt"]
    stub.text_literal_files = ["cc_dict.pickle", "memo_dict.pickle"]
    stub.numeric_dim, stub.text_dim = 2, 6
    stub.numeric_embed, stub.text_embed = {}, {}
    stub.n_heads = stub.n_tails = 0
    stub.num_embedding_table = stub.text_embedding_table = None
    stub.load_attributes()
    stub.construct_data(stub.load_graph(os.path.join(str(tmp_path), "pre_training_train.txt")))
    stub.embed_num_literal()
    stub.embed_txt_literal()
    trip, num, txt = D.read_data_dir(str(tmp_path), numeric_dim=2, text_dim=6, text_files=("cc_dict.pickle", "memo_dict.pickle"),
                                     use_num_lit=use_num, use_txt_lit=use_txt)
    assert np.array_equal(trip[:, 0], stub.h_list.numpy()) and np.array_equal(trip[:, 2], stub.t_list.numpy())
    for ours, theirs in ((num, stub.num_embedding_table), (txt, stub.text_embedding_table)):
        assert (ours is None) == (theirs is None)
        if ours is not None:
            assert ours.shape[0] == stub.n_entities
            assert np.array_equal(ours, theirs.numpy())


def test_result_writers_and_checkpoint_layout(tmp_path):
    import torch
    from literalkg_b200 import results as R
    metrics = {"accuracy": 0.73264, "precision": 0.5, "recall": 0.25, "f1": 1 / 3}
    scores = torch.arange(12, dtype=torch.float32).reshape(3, 4)
    out = R.write_test_results(str(tmp_path / "run"), 12.34, metrics, scores)
    import pandas as pd                                         # what a reader of test.py:40-42's file does
    df = pd.read_csv(out["tsv"], sep="\t")
    assert list(df.columns) == ["metrics"] and df["metrics"][0] == R.metrics_line(12.34, metrics)
    assert "Accuracy [0.7326]" in df["metrics"][0] and "F1 [0.3333]" in df["metrics"][0]
    assert out["npy"].endswith("runprediction_scores.npy")      # upstream concatenates without a separator (test.py:44)
    assert np.array_equal(np.load(out["npy"]), scores.numpy())
    lin = torch.nn.Linear(3, 2)
    p = R.save_model(lin, str(tmp_path / "ck"), 5, name="fine-tuning")
    assert os.path.basename(p) == "fine-tuning_model_epoch5.pth"
    ck = torch.load(p, weights_only=False)
    assert set(ck) == {"model_state_dict", "epoch"} and ck["epoch"] == 5
    p2 = R.save_model(lin, str(tmp_path / "ck"), 7, last_best_epoch=5, name="fine-tuning")
    assert not os.path.exists(p) and os.path.exists(p2)
    lin2 = R.load_model(torch.nn.Linear(3, 2), p2)
    assert torch.equal(lin2.weight, lin.weight) and not lin2.training
