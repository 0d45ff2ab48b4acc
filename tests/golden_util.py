"""Shared loaders of tests/golden/tfidf_golden.json (made by tests/golden/make_tfidf_golden.py) and of
tests/golden/rtflann_knn2.npz (made by tests/golden/make_rtflann_golden.py)."""
import functools
import hashlib
import json
from pathlib import Path

import numpy as np

GOLD = json.loads((Path(__file__).parent / "golden" / "tfidf_golden.json").read_text())
RTFLANN = Path(__file__).parent / "golden" / "rtflann_knn2.npz"


def load_golden_into(d, remap):
    """Feed the golden inverted index into a dictionary-like object (oracle or engine)."""
    word_ids = sorted(int(w) for w in GOLD["words"])
    desc = np.zeros((len(word_ids), 32), np.uint8)
    desc[:, :4] = np.asarray(word_ids, dtype=np.uint32).view(np.uint8).reshape(-1, 4)
    d.add_words(word_ids, desc)
    d.update()
    rp = [0]
    sig, cnt = [], []
    for w in word_ids:
        for s, c in GOLD["words"][str(w)]:
            sig.append(remap(s))
            cnt.append(c)
        rp.append(len(sig))
    d.load_csr(word_ids, rp, sig, cnt)
    d.set_ni([remap(s) for s in GOLD["sig_ids"]], GOLD["ni"])


def knn2_digest(data, queries) -> str:
    """SHA-256 of a 2-NN problem (dtype, shape and bytes of the rows and of the queries)."""
    h = hashlib.sha256()
    for a in (data, queries):
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.data)
    return h.hexdigest()


@functools.cache
def _rtflann():
    with np.load(RTFLANN) as z:
        return {k: z[k] for k in z.files}


def rtflann_knn2(name, data, queries):
    """The 2-NN of `queries` over the rows of `data` as the reference's own rtflann LinearIndex answered it, stored under `name`:
    (idx[nq, 2] int64, -1 where there is no neighbour; dist[nq, 2] float32).  The answer is only returned for the very inputs it was
    computed for."""
    g = _rtflann()
    if f"{name}.digest" not in g:
        raise KeyError(f"no stored rtflann answer named {name!r}; tests/golden/make_rtflann_golden.py makes them")
    assert str(g[f"{name}.digest"]) == knn2_digest(data, queries), f"{name}: the inputs differ from those of the stored rtflann answer"
    return g[f"{name}.idx"].astype(np.int64), g[f"{name}.dist"]
