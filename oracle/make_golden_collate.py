"""Generate tests/golden/collate.npz by running the reference's UNMODIFIED ``collate_fn`` (src/tasks.py:138-158) on CPU.

Needs a checkout of the original project:   python oracle/make_golden_collate.py <checkout>/src

``tasks.py`` imports ``h5py`` and ``scipy.misc.imread/imresize`` (absent / removed, SURVEY.md Q9) without using them in
``collate_fn``; the three names are stubbed in ``sys.modules`` so that the module imports.  Only numeric outputs are
committed: the ragged token lists fed in (flat + offsets) and the padded captions / lengths / max length that came out.
"""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_collate(src):
    for name in ("h5py", "torchtext"):
        sys.modules.setdefault(name, types.ModuleType(name))
    import scipy
    misc = types.ModuleType("scipy.misc")
    misc.imread = misc.imresize = lambda *a, **k: None
    sys.modules["scipy.misc"] = misc
    scipy.misc = misc
    sys.path.insert(0, src)
    import tasks
    return tasks.collate_fn


def cases():
    rng = np.random.RandomState(1008)
    out = {}
    out["ragged"] = [list(rng.randint(4, 1000, size=n)) for n in (5, 1, 14, 7, 14, 2, 9, 3)]
    out["single"] = [list(rng.randint(4, 50, size=6))]
    out["empty_caption"] = [[], list(rng.randint(4, 50, size=3)), []]            # a caption with no tokens: <S> <E> only
    out["all_empty"] = [[], []]
    out["long"] = [list(rng.randint(4, 30000, size=n)) for n in rng.randint(1, 49, size=64)]
    return out


def main():
    if len(sys.argv) != 2:
        sys.exit("usage: python oracle/make_golden_collate.py <checkout of the original project>/src")
    collate = load_collate(sys.argv[1])
    blob = {}
    for name, lists in cases().items():
        batch = [(torch.zeros(3, 4, 4), [int(t) for t in toks]) for toks in lists]
        images, captions, lengths, max_len = collate(batch)
        flat = np.array([t for toks in lists for t in toks], dtype=np.int64)
        offs = np.cumsum([0] + [len(t) for t in lists]).astype(np.int64)
        blob[name + "/tokens"] = flat
        blob[name + "/offsets"] = offs
        blob[name + "/captions"] = captions.numpy()
        blob[name + "/lengths"] = lengths.numpy()
        blob[name + "/max_caption_len"] = np.int64(max_len)
        assert captions.dtype == torch.int64 and lengths.dtype == torch.int32
    path = os.path.join(ROOT, "tests", "golden", "collate.npz")
    np.savez_compressed(path, **blob)
    print("wrote", path, "%.1f KB" % (os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
