"""Pin the restated linear 2-NN scan (oracle/oracle.cpp) against the REFERENCE'S OWN rtflann: the answers of its LinearIndex,
compiled from the reference sources by oracle/Makefile, are stored in tests/golden/rtflann_knn2.npz (make_rtflann_golden.py).
Covers Hamming (ORB) and squared-L2 (SURF) incl. exact ties and fewer than two rows."""
import numpy as np
import pytest

from golden_util import rtflann_knn2
from oracle import oracle_py as orc

HAMMING_CASES = [(1, 32), (2, 32), (3, 32), (777, 32), (4096, 32), (1000, 16), (500, 64)]
L2_CASES = [(2, 64), (1500, 64), (800, 128)]
KINDS = ["hamming", "l2"]


@pytest.mark.parametrize("rows,dim", HAMMING_CASES)
def test_hamming_matches_rtflann(rows, dim):
    rng = np.random.default_rng(rows * 7 + dim)
    data = rng.integers(0, 256, (rows, dim), dtype=np.uint8)
    q = rng.integers(0, 256, (64, dim), dtype=np.uint8)
    if rows > 10:
        data[5] = data[1]
        data[9] = data[1]          # three identical rows -> ties resolved to the lowest row
        q[0] = data[1]
        q[1] = data[rows - 1]
        q[2] = np.bitwise_xor(data[3], 1)
    i_ref, d_ref = rtflann_knn2(f"hamming_{rows}x{dim}", data, q)
    i_orc, d_orc = orc.knn2_raw(data, q)
    assert np.array_equal(i_ref, i_orc)
    valid = i_ref >= 0
    assert np.array_equal(d_ref[valid], d_orc[valid])


@pytest.mark.parametrize("rows,dim", L2_CASES)
def test_l2_matches_rtflann_bit_exact(rows, dim):
    rng = np.random.default_rng(rows + dim)
    data = rng.standard_normal((rows, dim)).astype(np.float32)
    data /= np.linalg.norm(data, axis=1, keepdims=True)
    q = (data[rng.integers(0, rows, 48)] + 0.02 * rng.standard_normal((48, dim))).astype(np.float32)
    if rows > 10:
        data[7] = data[2]
        q[0] = data[2]
    i_ref, d_ref = rtflann_knn2(f"l2_{rows}x{dim}", data, q)
    i_orc, d_orc = orc.knn2_raw(data, q)
    assert np.array_equal(i_ref, i_orc)
    # same float summation order as rtflann::L2 (dist.h:158-166): identical bits
    assert np.array_equal(d_ref.view(np.uint32), d_orc.view(np.uint32))


# ---- the quantiser loop, replayed on the reference's own primitives ---------------------------------------------------
def _replay_add_new_words(name, index_ids, index_desc, frame, nndr, last_id, incremental=True, cmp_new=True):
    """VWDictionary::addNewWords "Process results" loop (VWDictionary.cpp:1088-1219) written a second time, independently of
    oracle/oracle.cpp, on the primitives the reference itself calls: its own rtflann LinearIndex (its stored answer `name`)
    for the index search and cv::BFMatcher::knnMatch (OpenCV, the installed cv2) for the words created by the same frame.
    fullResults is a std::multimap<float,int>: a stable sort by distance of the insertion sequence."""
    import cv2

    binary = frame.dtype == np.uint8
    bf = cv2.BFMatcher(cv2.NORM_HAMMING if binary else cv2.NORM_L2SQR)
    idx_all, dist_all = (rtflann_knn2(name, index_desc, frame) if len(index_desc) else (None, None))
    new_desc, new_ids, out = [], [], []
    for i in range(len(frame)):
        full = []
        if idx_all is not None:
            for j in range(2):
                if idx_all[i, j] < 0:
                    break
                full.append((np.float32(dist_all[i, j]), int(index_ids[idx_all[i, j]])))
        if cmp_new and new_desc:
            for mt in bf.knnMatch(frame[i:i + 1], np.stack(new_desc), k=2 if len(new_desc) > 1 else 1)[0]:
                full.append((np.float32(mt.distance), new_ids[mt.trainIdx]))
        full.sort(key=lambda t: t[0])                     # stable: equal distances keep insertion order, like the multimap
        if incremental:
            bad = len(full) < 2 or full[0][0] > np.float32(nndr) * full[1][0]
            if bad:
                last_id += 1
                new_desc.append(frame[i])
                new_ids.append(last_id)
                out.append(last_id)
            else:
                out.append(full[0][1])
        elif full:
            out.append(full[0][1])
    return np.array(out, np.int32), last_id


@pytest.mark.parametrize("kind", KINDS)
def test_quantiser_loop_against_reference_primitives(kind):
    """Pins the NNDR / new-word loop of the oracle (the part of the quantiser the reference has no golden vector for) to an
    independent replay that gets every distance from the reference's rtflann and from cv::BFMatcher."""
    rng = np.random.default_rng(31)
    if kind == "hamming":
        vocab = rng.integers(0, 256, (1200, 32), dtype=np.uint8)

        def near(rows, k):
            out = rows.copy()
            for r in out:
                for b in rng.integers(0, 256, k):
                    r[b >> 3] ^= np.uint8(1 << (b & 7))
            return out
        o = orc.OracleDictionary(0, 32, True, 0.8, True)
    else:
        vocab = rng.standard_normal((1200, 64)).astype(np.float32)
        vocab /= np.linalg.norm(vocab, axis=1, keepdims=True)

        def near(rows, k):
            q = rows + 0.004 * k * rng.standard_normal(rows.shape).astype(np.float32)
            return (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
        o = orc.OracleDictionary(1, 64, True, 0.8, True)
    ids = np.arange(1, 1201, dtype=np.int32) * 3
    o.add_words(ids, vocab)
    o.last_word_id = int(ids.max())
    o.update()
    index_ids, index_desc = ids.copy(), vocab.copy()
    last = int(ids.max())
    for t in range(1, 5):
        fresh = rng.integers(0, 256, (120, 32), dtype=np.uint8) if kind == "hamming" else near(rng.standard_normal((120, 64)).astype(np.float32), 0)
        frame = np.concatenate([near(vocab[rng.integers(0, 1200, 50)], 6), fresh, near(fresh[:40], 4), fresh[5:8]])
        want, last = _replay_add_new_words(f"quantiser_{kind}_frame{t}", index_ids, index_desc, frame, 0.8, last)
        got = o.add_new_words(frame, t)
        assert np.array_equal(got, want), f"{kind} frame {t}"
        assert o.last_word_id == last
        # update(): the frame's new words join the index in ascending id order (first occurrence of every new id)
        new_ids, first = np.unique(want[want > index_ids.max()], return_index=True)
        pos = np.flatnonzero(want > index_ids.max())[first]
        index_ids = np.concatenate([index_ids, new_ids.astype(np.int32)])
        index_desc = np.concatenate([index_desc, frame[pos]])
        o.update()


@pytest.mark.parametrize("kind", KINDS)
def test_find_nn_against_reference_primitives(kind):
    """VWDictionary::findNN (VWDictionary.cpp:1273-1552): index hits from the reference's rtflann, hits among the words that are
    not indexed yet from cv::BFMatcher::knnMatch, multimap order, NNDR — replayed independently and compared with the oracle."""
    import cv2

    rng = np.random.default_rng(41)
    if kind == "hamming":
        vocab = rng.integers(0, 256, (900, 32), dtype=np.uint8)
        pend = rng.integers(0, 256, (60, 32), dtype=np.uint8)
        o = orc.OracleDictionary(0, 32, True, 0.8, True)
        q = np.concatenate([vocab[:40] ^ np.uint8(1), pend[:20] ^ np.uint8(2), rng.integers(0, 256, (30, 32), dtype=np.uint8), pend[3:5]])
        bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    else:
        vocab = rng.standard_normal((900, 64)).astype(np.float32)
        pend = rng.standard_normal((60, 64)).astype(np.float32)
        o = orc.OracleDictionary(1, 64, True, 0.8, True)
        q = np.concatenate([vocab[:40] + np.float32(0.01), pend[:20] - np.float32(0.02), rng.standard_normal((30, 64)).astype(np.float32), pend[3:5]])
        bf = cv2.BFMatcher(cv2.NORM_L2SQR)
    ids = np.arange(1, 901, dtype=np.int32) * 2
    pend_ids = np.arange(2001, 2061, dtype=np.int32)
    o.add_words(ids, vocab)
    o.update()
    o.add_words(pend_ids, pend)            # not indexed: no update()
    o.last_word_id = 2060
    idx, dist = rtflann_knn2(f"find_nn_{kind}", vocab, q)
    mni = bf.knnMatch(q, pend, k=2)
    want = np.zeros(len(q), np.int32)
    for i in range(len(q)):
        full = [(np.float32(dist[i, j]), int(ids[idx[i, j]])) for j in range(2) if idx[i, j] >= 0]
        full += [(np.float32(m.distance), int(pend_ids[m.trainIdx])) for m in mni[i]]
        full.sort(key=lambda t: t[0])
        if len(full) >= 2 and not (full[0][0] > np.float32(0.8) * full[1][0]):
            want[i] = full[0][1]
    got = o.find_nn(q)
    assert np.array_equal(got, want)
    assert (want > 2000).any() and (want == 0).any() and ((want > 0) & (want <= 1800)).any()
