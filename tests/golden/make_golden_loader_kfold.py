"""Golden fixture for the k-fold and sentence-masking modes of the loader: the dataset stored in loader_split.npz, written
to a folder and loaded with each keyword set in CASES, directory listings sorted (the fold layout follows the listing
order).  Stores, per case and fold, the episode names and the x / y of every episode in tests/golden/loader_kfold.npz.

    MTS_REFERENCE=<checkout of the reference> python tests/golden/make_golden_loader_kfold.py

records the reference's utils/load_datasets_precomputed.py; without MTS_REFERENCE it records the loader of this package
(a regression pin).  The `source` entry of the file says which one wrote it."""
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from test_loader import _rebuild  # noqa: E402

CASES = {"kfold3": {"k_folds": 3},
         "kfold2_masked": {"k_folds": 2, "mask_inner_sentences": True, "mask_probability": 0.5}}


def main():
    ref = os.environ.get("MTS_REFERENCE")
    if ref:
        sys.path.insert(0, ref)
        from utils.load_datasets_precomputed import load_dataset_from_precomputed
        source = "reference utils/load_datasets_precomputed.py"
    else:
        from multimodaltopicsegmentation_b200 import load_dataset_from_precomputed
        source = "multimodaltopicsegmentation_b200.load_datasets_precomputed"
    listdir = os.listdir
    os.listdir = lambda p: sorted(listdir(p))
    fx = np.load(os.path.join(HERE, "loader_split.npz"))
    out = {"source": np.array(source)}
    with tempfile.TemporaryDirectory() as root:
        _rebuild(fx, root)
        emb = os.path.join(root, "text") + "+" + os.path.join(root, "audio")
        for tag, kwargs in CASES.items():
            folds = load_dataset_from_precomputed(emb, os.path.join(root, "labs_dict.pkl"), **kwargs)
            out[f"{tag}:kwargs"] = np.array(json.dumps(kwargs))
            out[f"{tag}:folds"] = np.array(len(folds))
            for i, fold in enumerate(folds):
                assert len(fold) == 2
                for part, eps in zip(("train", "test"), fold):
                    out[f"{tag}:{i}:{part}:names"] = np.array([e[2] for e in eps])
                    for e in eps:
                        out[f"{tag}:{i}:{part}:{e[2]}:x"] = e[0].numpy()
                        out[f"{tag}:{i}:{part}:{e[2]}:y"] = np.array(e[1])
    np.savez_compressed(os.path.join(HERE, "loader_kfold.npz"), **out)
    print("written", os.path.join(HERE, "loader_kfold.npz"), len(out), "arrays from", source)


if __name__ == "__main__":
    main()
