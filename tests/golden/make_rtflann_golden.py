"""Make tests/golden/rtflann_knn2.npz: every 2-NN answer of the reference's own rtflann LinearIndex (FlannIndex::knnSearch at
Kp/NNStrategy=0, compiled from the reference sources into oracle/_ref/libref_flann.so by oracle/Makefile) that the tests compare with:

  tests/test_oracle_ref.py        run here with the live library, so its assertions check the oracle against it on the way;
  tests/test_gpu_configs.py C3    the grown 720p dictionary, rebuilt on the CPU (cv2 ORB, which the test pins the CUDA ORB to bit
                                  for bit, and the oracle's quantiser, which the test pins the engine to);
  tests/test_gpu_configs.py C4    the 1 100 000-row float dictionary.

Each answer is stored with the digest of its inputs (golden_util.knn2_digest); the tests refuse an answer for other inputs.

Run where the reference sources are readable:  python tests/golden/make_rtflann_golden.py
"""
import sys
from pathlib import Path

import numpy as np

TESTS = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(TESTS.parent), str(TESTS)]

import golden_util  # noqa: E402
import test_gpu_configs as C  # noqa: E402
import test_oracle_ref as T  # noqa: E402
from oracle import feature2d_py as f2d  # noqa: E402
from oracle import oracle_py as orc  # noqa: E402

OUT = golden_util.RTFLANN
answers = {}


def live_knn2(name, data, queries):
    assert orc.ref_lib() is not None, "oracle/_ref/libref_flann.so is not built and the reference sources are not readable"
    assert f"{name}.digest" not in answers, f"two searches named {name}"
    idx, dist = orc.ref_knn2(data, queries)
    answers[f"{name}.digest"] = np.array(golden_util.knn2_digest(data, queries))
    answers[f"{name}.idx"] = idx.astype(np.int32)
    answers[f"{name}.dist"] = dist
    return idx, dist


def c3_grown_dictionary():
    """test_c3's dictionary after its stream, in the engine's row order (initial rows, then each update's new words by id)."""
    vocab, imgs, deps, rng = C.c3_stream()
    ids = np.arange(1, C.C3_W0 + 1, dtype=np.int32)
    o = orc.OracleDictionary(0, 32, True, 0.8, True)
    o.add_words(ids, vocab)
    o.last_word_id = C.C3_W0
    o.update()
    rows, row_ids = [vocab], [ids]
    frame2 = None
    for t in range(len(imgs)):
        _, desc, _ = f2d.detect_describe(imgs[t], deps[t], C.C3_K4, f2d.OrbParams(n_features=1000))
        frame2 = desc if t == 2 else frame2
        last = o.last_word_id
        o.update()
        w = o.add_new_words(desc, 1 + t)
        new_ids, first = np.unique(w[w > last], return_index=True)   # a new word's descriptor is that of the query that made it
        rows.append(desc[np.flatnonzero(w > last)[first]])
        row_ids.append(new_ids.astype(np.int32))
    o.update()
    gi, gv = np.concatenate(row_ids), np.concatenate(rows)
    assert np.array_equal(gi, o.indexed_ids()) and len(gi) > 262144
    return gv, C.c3_queries(vocab, frame2, rng)


def main():
    T.rtflann_knn2 = live_knn2
    for rows, dim in T.HAMMING_CASES:
        T.test_hamming_matches_rtflann(rows, dim)
    for rows, dim in T.L2_CASES:
        T.test_l2_matches_rtflann_bit_exact(rows, dim)
    for kind in T.KINDS:
        T.test_quantiser_loop_against_reference_primitives(kind)
        T.test_find_nn_against_reference_primitives(kind)
    live_knn2("c3_grown_dictionary", *c3_grown_dictionary())
    vocab, _, q = C.c4_problem()
    live_knn2("c4_million_rows", vocab, q)
    np.savez_compressed(OUT, **answers)
    print(f"wrote {OUT}: {len(answers) // 3} searches, {OUT.stat().st_size} bytes")


if __name__ == "__main__":
    main()
