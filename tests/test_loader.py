"""Loader mirror (multimodaltopicsegmentation_b200/load_datasets_precomputed.py) against outputs of the unmodified
reference loader (tests/golden/loader_split.npz, made by tests/golden/make_golden_loader.py) and, in k-fold and
sentence-masking mode, against the reference itself where it is present and against tests/golden/loader_kfold.npz."""
import json
import os
import pickle
import sys

import numpy as np
import pytest
import torch


def _rebuild(fx, root):
    names = sorted({k.split(":")[1] for k in fx.files if k.startswith("in:ep")})
    os.makedirs(os.path.join(root, "text"))
    os.makedirs(os.path.join(root, "audio"))
    labs, times = {}, {}
    for n in names:
        np.save(os.path.join(root, "text", n + ".npy"), fx[f"in:{n}:text"])
        np.save(os.path.join(root, "audio", n + ".npy"), fx[f"in:{n}:audio"])
        labs[n] = fx[f"in:{n}:labs"].tolist()
        times[n] = fx[f"in:{n}:times"].tolist()
    with open(os.path.join(root, "labs_dict.pkl"), "wb") as f:
        pickle.dump(labs, f)
    with open(os.path.join(root, "times.pkl"), "wb") as f:
        pickle.dump(times, f)
    with open(os.path.join(root, "split.json"), "w") as f:
        f.write(str(fx["in:split"]))
    return names


@pytest.mark.parametrize("tag", ["plain", "timed"])
def test_standard_split_matches_reference_golden(golden, tmp_path, tag):
    from multimodaltopicsegmentation_b200 import load_dataset_from_precomputed

    fx = golden("loader_split")
    root = str(tmp_path)
    _rebuild(fx, root)
    res = load_dataset_from_precomputed(os.path.join(root, "text") + "+" + os.path.join(root, "audio"),
                                        os.path.join(root, "labs_dict.pkl"), split=os.path.join(root, "split.json"),
                                        timing_info=os.path.join(root, "times.pkl") if tag == "timed" else None)
    assert len(res) == 1 and len(res[0]) == 3
    for part, eps in zip(("train", "test", "validation"), res[0]):   # the reference's order: train, TEST, validation
        assert [e[2] for e in eps] == fx[f"{tag}:{part}:names"].tolist()
        for e in eps:
            np.testing.assert_array_equal(e[0].numpy(), fx[f"{tag}:{part}:{e[2]}:x"])   # bit-exact: pure data movement
            assert list(e[1]) == fx[f"{tag}:{part}:{e[2]}:y"].tolist()
            assert e[1][-1] == 0                                                       # last label forced to 0


def test_keep_modalities_is_the_unconcatenated_view(golden, tmp_path):
    from multimodaltopicsegmentation_b200 import load_dataset_from_precomputed

    fx = golden("loader_split")
    root = str(tmp_path)
    _rebuild(fx, root)
    args = (os.path.join(root, "text") + "+" + os.path.join(root, "audio"), os.path.join(root, "labs_dict.pkl"))
    cat = load_dataset_from_precomputed(*args, split=os.path.join(root, "split.json"))
    sep = load_dataset_from_precomputed(*args, split=os.path.join(root, "split.json"), keep_modalities=True)
    for a_part, b_part in zip(cat[0], sep[0]):
        for a, b in zip(a_part, b_part):
            assert isinstance(b[0], tuple) and len(b[0]) == 2 and a[2] == b[2]
            assert torch.equal(a[0], torch.cat(b[0], dim=-1))


def test_cross_validation_split_partitions():
    from multimodaltopicsegmentation_b200 import cross_validation_split

    data = [(torch.zeros(2, 1), [0, 0], f"f{i}") for i in range(13)]
    folds = cross_validation_split(data, num_folds=5, inverse_augmentation=False)
    assert len(folds) == 5
    for i, (train, test) in enumerate(folds):
        assert [e[2] for e in test] == [f"f{j}" for j in range(2 * i, 2 * i + 2)]
        assert sorted(e[2] for e in train + test) == sorted(e[2] for e in data)
    with pytest.raises(NotImplementedError):
        cross_validation_split(data, inverse_augmentation=True)


@pytest.mark.skipif(not os.path.isdir("/root/reference/utils"), reason="the reference exists in the build container only")
def test_kfold_and_masking_match_reference_live(golden, tmp_path):
    sys.path.insert(0, "/root/reference")
    try:
        from utils import load_datasets_precomputed as ref
    finally:
        sys.path.pop(0)
    from multimodaltopicsegmentation_b200 import load_dataset_from_precomputed

    fx = golden("loader_split")
    root = str(tmp_path)
    _rebuild(fx, root)
    emb = os.path.join(root, "text") + "+" + os.path.join(root, "audio")
    lab = os.path.join(root, "labs_dict.pkl")
    for kwargs in ({"k_folds": 3}, {"k_folds": 2, "mask_inner_sentences": True, "mask_probability": 0.5}):
        a = ref.load_dataset_from_precomputed(emb, lab, **kwargs)      # same process, same directory listing order
        b = load_dataset_from_precomputed(emb, lab, **kwargs)
        assert len(a) == len(b)
        for fa, fb in zip(a, b):
            for pa, pb in zip(fa, fb):
                assert [e[2] for e in pa] == [e[2] for e in pb]
                for ea, eb in zip(pa, pb):
                    assert torch.equal(ea[0], eb[0]) and list(ea[1]) == list(eb[1])


def test_kfold_and_masking_match_golden(golden, tmp_path, monkeypatch):
    """k-fold and sentence-masking modes against tests/golden/loader_kfold.npz (made by
    tests/golden/make_golden_loader_kfold.py), with the directory listing sorted as it was when the file was written.
    Its `source` entry names the loader that wrote it: this package's, as a regression pin, until it is re-recorded
    from a reference checkout."""
    from multimodaltopicsegmentation_b200 import load_dataset_from_precomputed

    fx = golden("loader_kfold")
    root = str(tmp_path)
    _rebuild(golden("loader_split"), root)
    listdir = os.listdir
    monkeypatch.setattr(os, "listdir", lambda p: sorted(listdir(p)))
    emb = os.path.join(root, "text") + "+" + os.path.join(root, "audio")
    lab = os.path.join(root, "labs_dict.pkl")
    tags = sorted({k.split(":")[0] for k in fx.files if k.endswith(":kwargs")})
    assert tags == ["kfold2_masked", "kfold3"]
    for tag in tags:
        folds = load_dataset_from_precomputed(emb, lab, **json.loads(str(fx[f"{tag}:kwargs"])))
        assert len(folds) == int(fx[f"{tag}:folds"])
        for i, fold in enumerate(folds):
            assert len(fold) == 2
            for part, eps in zip(("train", "test"), fold):
                assert [e[2] for e in eps] == fx[f"{tag}:{i}:{part}:names"].tolist()
                for e in eps:
                    x = fx[f"{tag}:{i}:{part}:{e[2]}:x"]
                    assert e[0].numpy().dtype == x.dtype
                    np.testing.assert_array_equal(e[0].numpy(), x)
                    assert list(e[1]) == fx[f"{tag}:{i}:{part}:{e[2]}:y"].tolist()


@pytest.mark.gpu
def test_resident_dataset_batches_equal_the_host_collater(golden, tmp_path):
    """Device-side collater (mts_gather_pad) == the reference-shaped host collater, bit for bit, and the pair input of
    the early-fusion model gives the same scores as the concatenated one."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from multimodaltopicsegmentation_b200 import (AudioPortionDataset, BiLSTM, ResidentDataset,
                                                  load_dataset_from_precomputed)

    dev = torch.device("cuda:0")
    fx = golden("loader_split")
    root = str(tmp_path)
    _rebuild(fx, root)
    args = (os.path.join(root, "text") + "+" + os.path.join(root, "audio"), os.path.join(root, "labs_dict.pkl"))
    cat = load_dataset_from_precomputed(*args, split=os.path.join(root, "split.json"))[0][0]
    sep = load_dataset_from_precomputed(*args, split=os.path.join(root, "split.json"), keep_modalities=True)[0][0]
    host_ds = AudioPortionDataset(cat, {"0": 0, "1": 1}, CRF=False, truncate=False)
    ids = [2, 0, 3]
    host = host_ds.collater([host_ds[i] for i in ids])
    res_cat = ResidentDataset(cat, dev).batch(ids)
    res_sep = ResidentDataset(sep, dev).batch(ids)
    assert torch.equal(res_cat["src_tokens"].cpu(), host["src_tokens"])
    assert torch.equal(res_cat["tgt_tokens"].cpu(), host["tgt_tokens"])
    assert res_cat["src_lengths"].tolist() == host["src_lengths"].tolist()
    assert torch.equal(torch.cat([t.cpu() for t in res_sep["src_tokens"]], dim=-1), host["src_tokens"])
    torch.manual_seed(0)
    m = BiLSTM(2, 10, 256, num_layers=1, loss_fn="FocalLoss").to(dev)
    m.th = 0.5
    s1, t1 = m(res_cat["src_tokens"], res_cat["src_lengths"])
    s2, t2 = m(res_sep["src_tokens"], res_sep["src_lengths"])
    assert torch.equal(s1, s2) and t1 == t2
