"""Parity at the sizes BASELINE.json's configs name (VERDICT r1, item 1) — every check goes through the C ABI and compares with
the CPU oracle (rtflann-pinned restatement) or with the reference's own compiled rtflann (its answers stored in
tests/golden/rtflann_knn2.npz) / cv2 where that is the reference:

  C1  the reference's own data/samples images (tests/golden/samples_c1.npz): CUDA ORB vs cv::ORB bit for bit on REAL images, then
      the incremental dictionary + raw likelihood of every frame vs the oracle, and the loop-closure recall against samples_GT.bmp
      (tools/ConsoleApp/main.cpp:321,401);
  C2  49 152 words / 10 000 signatures / 1000 keypoints per 640x480 frame through lcd_process_frames, revisits, rotated views and
      never-seen places;
  C3  1280x720 mapping-mode stream whose dictionary grows PAST 262 144 words (the cv::BFMatcher ceiling, VWDictionary.cpp:576-583);
  C4  float descriptors against >= 1 048 576 dictionary rows (row field of the packed keys, 64-bit keys).
"""
from pathlib import Path

import numpy as np
import pytest

from golden_util import rtflann_knn2
from oracle import feature2d_py as f2d
from oracle import oracle_py as orc
from rtabmap_b200 import Engine, synth

pytestmark = pytest.mark.gpu
GOLDEN = Path(__file__).parent / "golden"


# --------------------------------------------------------------------------------------- C1 ---
def _samples():
    import cv2

    z = np.load(GOLDEN / "samples_c1.npz")
    off = z["offsets"]
    imgs = [cv2.imdecode(z["jpeg"][off[i]:off[i + 1]], cv2.IMREAD_COLOR) for i in range(len(off) - 1)]
    return imgs, z["gt"]


def test_c1_sample_images_orb_bit_exact():
    """Every data/samples image through the CUDA ORB (BGR -> gray, FAST, Harris, retainBest order, IC angle, rBRIEF) against cv::ORB."""
    imgs, _ = _samples()
    eng = Engine()
    K4 = (400.0, 400.0, 256.0, 192.0)
    total = 0
    for nf in (1000, 150):  # 150: retainBest / limitKeypoints actually cut on these low-texture frames
        op = Engine.orb_params(K4, n_features=nf)
        out = eng.orb_detect_describe(np.stack(imgs), None, op)
        for i, im in enumerate(imgs):
            kp_o, d_o, _ = f2d.detect_describe(im, None, K4, f2d.OrbParams(n_features=nf))
            kp, d, _ = out[i]
            assert len(kp) == len(kp_o), f"image {i + 1}: {len(kp)} vs {len(kp_o)} keypoints"
            assert np.array_equal(kp, kp_o), f"image {i + 1}: keypoints differ"
            assert np.array_equal(d, d_o), f"image {i + 1}: descriptors differ"
            total += len(kp)
    assert total > 84 * 150


def test_c1_sample_stream_incremental_dictionary_likelihood_and_recall():
    """ConsoleApp's loop on data/samples (config #1): per frame update() -> addNewWords() -> computeLikelihood() over the signatures
    outside the short-term memory (Mem/STMSize = 10).  Word ids bit-exact, raw likelihood 1e-4; the arg-max hypotheses are scored
    against the reference's ground-truth matrix."""
    imgs, gt = _samples()
    eng = Engine()
    o = orc.OracleDictionary(0, 32, True, 0.8, True)
    op = Engine.orb_params((400.0, 400.0, 256.0, 192.0), n_features=1000)
    feats = eng.orb_detect_describe(np.stack(imgs), None, op)
    stm = 10
    hits = misses = 0
    for t, (kp, desc, _) in enumerate(feats, start=1):
        eng.update()
        o.update()
        if len(desc) == 0:  # a textureless frame: VWDictionary::addNewWords returns an empty list (VWDictionary.cpp:920-925)
            continue
        g, n_new = eng.quantize(desc, t)
        w = o.add_new_words(desc, t)
        assert np.array_equal(g, w), f"frame {t}: word ids differ"
        ids = np.arange(1, t - stm + 1, dtype=np.int32)  # working memory: everything older than the STM
        if len(ids) == 0:
            continue
        like_g = eng.score(g, ids, t)
        like_o = o.likelihood(w, ids, t)
        assert np.allclose(like_g, like_o, rtol=1e-4, atol=1e-6), f"frame {t}: likelihood differs"
        best = int(np.argmax(like_g))
        assert best == int(np.argmax(like_o))
        row = gt[t - 1]
        if (row[:len(ids)] == 255).any() and like_g[best] > 0:
            if row[best] == 255:
                hits += 1
            else:
                misses += 1
    assert eng.last_word_id == o.last_word_id and eng.size() == o.size()
    assert hits + misses >= 40
    # the raw TF-IDF arg-max (no Bayes filter) already finds the true revisit for the large majority of the revisited frames
    assert hits / (hits + misses) >= 0.8, (hits, misses)


# --------------------------------------------------------------------------------------- C2 ---
@pytest.fixture(scope="module")
def c2_world():
    eng = Engine(max_words=49152, max_signatures=10002, max_queries=1000, max_batch=16)
    op = Engine.orb_params(synth.CAMERA_K4, n_features=1000)
    world = synth.make_place_world(lambda im, dp: eng.orb_detect_describe(im[None], dp[None], op, cap=1000)[0], 50, 49152, 10000, 1000)
    sm = world.smap
    eng.add_words(world.word_ids, world.vocab)
    eng.last_word_id = int(world.word_ids.max())
    eng.update()
    eng.load_csr(sm.word_ids, sm.row_ptr, sm.sig, sm.cnt)
    eng.set_ni(sm.sig_ids, sm.ni)
    for s0 in range(0, 10000, 1000):
        eng.sig_add_batch(sm.sig_ids[s0:s0 + 1000], world.store.desc[s0:s0 + 1000], world.store.xyz[s0:s0 + 1000], sm.ni[s0:s0 + 1000])
    o = orc.OracleDictionary(0, 32, True, 0.8, True)
    o.add_words(world.word_ids, world.vocab)
    o.last_word_id = int(world.word_ids.max())
    o.update()
    o.load_csr(sm.word_ids, sm.row_ptr, sm.sig, sm.cnt)
    o.set_ni(sm.sig_ids, sm.ni)
    return eng, o, world, op


def test_c2_full_size_whole_path_matches_oracle(c2_world):
    """BASELINE configs[1] at FULL size (49 152 words, 10 000 signatures, ~1000 keypoints per 640x480 frame): 12 frames — plain revisits,
    rotated / scaled revisits and never-seen places — through lcd_process_frames against cv::ORB + the oracle, stage by stage."""
    eng, o, world, op = c2_world
    assert len(world.vocab) == 49152
    sm = world.smap
    imgs, deps, places = synth.make_view_frames(world, 12, seed=11, mode="mixed")
    vp = Engine.verify_params(synth.CAMERA_K4, image_size=(640, 480))
    nkp, words, like, hyp, res = eng.process_frames(imgs, deps, op, sm.sig_ids, 10001, vp, True, 0.8, True)
    n_ok = 0
    for b in range(len(imgs)):
        kp, d, x = f2d.detect_describe(imgs[b], deps[b], synth.CAMERA_K4, f2d.OrbParams(n_features=1000))
        assert nkp[b] == len(kp), f"frame {b}"
        w_o, l_o = o.localize_ro(d, sm.sig_ids, 10001)
        assert np.array_equal(words[b][:len(w_o)], w_o), f"frame {b}: word ids"
        assert np.allclose(like[b], l_o, rtol=1e-4, atol=1e-6), f"frame {b}: likelihood"
        h = int(np.argmax(l_o))
        if l_o[h] <= 0:
            assert hyp[b] == 0
            continue
        assert hyp[b] == int(sm.sig_ids[h])
        n = int(sm.ni[h])
        v = orc.verify_pair_cov(world.store.desc[h][:n], world.store.xyz[h][:n], d, kp[:, :2], synth.CAMERA_K4, xyz_to=x, image_size=(640, 480))
        r = res[b]
        assert r["ok"] == v["ok"] and r["n_matches"] == len(v["matches"]) and r["n_inliers"] == len(v["inliers"]), f"frame {b}: verification"
        if v["ok"]:
            n_ok += 1
            assert np.allclose(r["rvec"], v["rvec"], atol=1e-4) and np.allclose(r["tvec"], v["tvec"], atol=1e-4)
            assert np.allclose(r["covariance"], v["covariance"], rtol=1e-4, atol=1e-9)
    assert 3 <= n_ok < len(imgs)  # revisits verify, never-seen places do not


def test_c2_full_size_localisation_batch_of_synthetic_queries(c2_world):
    """The quantise -> score half at full size on descriptor-level queries with heavy intra-frame duplication (new-word chains)."""
    eng, o, world, op = c2_world
    sm = world.smap
    rng = np.random.default_rng(5)
    B, F = 6, 1000
    q = np.empty((B, F, 32), np.uint8)
    for b in range(B):
        q[b] = synth.flip_bits(world.vocab[rng.integers(0, 49152, F)], 0.06, rng)
        q[b, ::9] = rng.integers(0, 256, (len(q[b, ::9]), 32), dtype=np.uint8)
        q[b, 1::9] = synth.flip_bits(q[b, 0::9][: len(q[b, 1::9])], 0.01, rng)  # near copies of brand-new descriptors
    words, like = eng.localize_batch(q.reshape(-1, 32), B, sm.sig_ids, 10001)
    for b in range(B):
        w_o, l_o = o.localize_ro(q[b], sm.sig_ids, 10001)
        assert np.array_equal(words[b], w_o)
        assert np.allclose(like[b], l_o, rtol=1e-4, atol=1e-6)


# --------------------------------------------------------------------------------------- C3 ---
C3_W0 = 261000
C3_K4 = (910.0, 910.0, 640.0, 360.0)


def c3_stream():
    """The initial vocabulary and the 720p frames of test_c3, and the generator that then draws its queries."""
    rng = np.random.default_rng(12)
    vocab = synth.make_binary_vocabulary(C3_W0, 32, 5)
    n_frames = 8
    imgs = np.stack([synth.make_image(720, 1280, 300 + (k % 5), n_rects=3000) for k in range(n_frames)])
    for k in range(n_frames):  # later frames re-observe earlier ones with noise: their words must be found among the NEW rows
        if k >= 5:
            imgs[k] = np.clip(imgs[k - 5].astype(np.int16) + rng.integers(-3, 4, imgs[k].shape), 0, 255).astype(np.uint8)
    deps = np.stack([synth.make_depth(720, 1280, 400 + k) for k in range(n_frames)])
    return vocab, imgs, deps, rng


def c3_queries(vocab, frame2_desc, rng):
    """Noisy copies of initial words and of words the stream created (frame 2's descriptors)."""
    return synth.flip_bits(np.concatenate([vocab[rng.integers(0, C3_W0, 100)], frame2_desc[:100]]), 0.05, rng)


def test_c3_mapping_stream_720p_grows_past_262144_words():
    """configs[2]: 1280x720 frames in mapping mode.  The dictionary starts at 261 000 words (as after a long run / a database load)
    and every frame adds its unmatched descriptors, so the stream crosses 262 144 rows — where the reference's BF strategies stop
    (VWDictionary.cpp:576-583) and only the FLANN-linear order (the rtflann-pinned oracle) is defined."""
    W0 = C3_W0
    vocab, imgs, deps, rng = c3_stream()
    ids = np.arange(1, W0 + 1, dtype=np.int32)
    eng = Engine(max_words=300000, max_queries=1000)
    o = orc.OracleDictionary(0, 32, True, 0.8, True)
    for d in (eng, o):
        d.add_words(ids, vocab)
        d.last_word_id = W0
        d.update()
    K4 = C3_K4
    op = Engine.orb_params(K4, n_features=1000)
    n_frames = len(imgs)
    feats = eng.orb_detect_describe(imgs, deps, op)
    crossed = False
    for t in range(n_frames):
        kp, desc, xyz = feats[t]
        kp_o, d_o, x_o = f2d.detect_describe(imgs[t], deps[t], K4, f2d.OrbParams(n_features=1000))
        assert np.array_equal(kp, kp_o) and np.array_equal(desc, d_o) and np.array_equal(xyz, x_o, equal_nan=True), f"frame {t}: ORB at 720p"
        eng.update()
        o.update()
        g, n_new = eng.quantize(desc, 1 + t)
        w = o.add_new_words(desc, 1 + t)
        assert np.array_equal(g, w), f"frame {t}: word ids"
        crossed = crossed or eng.size() > 262144
    assert crossed and eng.size() == o.size() and eng.last_word_id == o.last_word_id
    eng.update()
    o.update()
    assert eng.indexed_size() > 262144
    # the re-observed frames found words created by this stream (ids above the initial vocabulary)
    assert (g > W0).sum() > 100
    # exact 2-NN over the grown dictionary against the reference's own compiled rtflann
    q = c3_queries(vocab, feats[2][1], rng)
    gi, gv = eng.get_indexed()
    r_idx, r_dist = rtflann_knn2("c3_grown_dictionary", gv, q)
    i1, d1, i2, d2 = eng.knn2(q)
    assert np.array_equal(i1, gi[r_idx[:, 0]]) and np.array_equal(i2, gi[r_idx[:, 1]])
    assert np.array_equal(d1, r_dist[:, 0].astype(np.float32)) and np.array_equal(d2, r_dist[:, 1].astype(np.float32))


# --------------------------------------------------------------------------------------- C4 ---
C4_W = 1_100_000


def c4_problem():
    """The dictionary rows of test_c4, the rows its queries start from, and the queries."""
    W = C4_W
    vocab = synth.make_float_vocabulary(W, 64, 21)
    rng = np.random.default_rng(22)
    nq = 96
    src = rng.integers(0, W, nq)
    src[:8] = np.array([0, 1, W - 1, W - 2, 1 << 20, (1 << 20) - 1, (1 << 20) + 1, 524288])  # rows at the ends and around 2^20
    q = vocab[src] + rng.normal(0, 0.02, (nq, 64)).astype(np.float32)
    q[-16:] = synth.make_float_vocabulary(16, 64, 99)  # unrelated descriptors: NNDR rejects, new words
    q[-8:-4] = q[-16:-12] + np.float32(1e-3)            # near copies of new descriptors inside the frame
    return vocab, src, np.ascontiguousarray(q, np.float32)


def test_c4_float_quantiser_over_a_million_rows():
    """configs[3] size: SURF-like 64-D float descriptors against 1 100 000 dictionary rows (beyond 2^20): exact squared-L2 2-NN ids and
    distances bit for bit against the reference's compiled rtflann (its stored answer), then the NNDR / new-word pass against the oracle."""
    W = C4_W
    vocab, src, q = c4_problem()
    ids = np.arange(1, W + 1, dtype=np.int32)
    eng = Engine(desc_type=1, desc_dim=64, max_words=W + 4096, max_queries=1000)
    eng.add_words(ids, vocab)
    eng.last_word_id = W
    eng.update()
    i1, d1, i2, d2 = eng.knn2(q)
    r_idx, r_dist = rtflann_knn2("c4_million_rows", vocab, q)
    assert np.array_equal(i1, ids[r_idx[:, 0]]) and np.array_equal(i2, ids[r_idx[:, 1]])
    assert np.array_equal(d1, r_dist[:, 0]) and np.array_equal(d2, r_dist[:, 1])
    assert (i1[:8] == ids[src[:8]]).all()
    o = orc.OracleDictionary(1, 64, True, 0.8, True)
    o.add_words(ids, vocab)
    o.last_word_id = W
    o.update()
    g, n_new = eng.quantize(q, 7)
    w = o.add_new_words(q, 7)
    assert np.array_equal(g, w) and n_new >= 8
