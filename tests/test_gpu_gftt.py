"""Parity of the CUDA GFTT/ORB detector (Kp/DetectorStrategy=8: cv::GFTTDetector corners described by cv::ORB::compute) against
opencv-python through the oracle's restated RTAB-Map wrapper (oracle/feature2d_py.py).  Same bar as tests/test_gpu_orb.py: keypoints
in the same order (pt, size, octave exact; response and angle bit for bit), descriptor bytes and 3-D points bit for bit."""
import numpy as np
import pytest

from oracle import feature2d_py as f2d
from oracle import gftt_py
from rtabmap_b200 import Engine, LcdError, synth
from rtabmap_b200.capi import LCD_DETECTOR_GFTT_ORB, LCD_DETECTOR_ORB

pytestmark = pytest.mark.gpu
K4 = synth.CAMERA_K4
LCD_ERR_CAPACITY = -3


def check_frame(got, want):
    kp_g, d_g, x_g = got
    kp_w, d_w, x_w = want
    assert len(kp_g) == len(kp_w), (len(kp_g), len(kp_w))
    assert np.array_equal(kp_g[:, [0, 1, 2, 5]], kp_w[:, [0, 1, 2, 5]]), "keypoint set / order differs"
    assert np.array_equal(kp_g[:, 4].view(np.uint32), kp_w[:, 4].view(np.uint32)), "responses differ"
    assert np.array_equal(kp_g[:, 3].view(np.uint32), kp_w[:, 3].view(np.uint32)), "angles differ"
    assert np.array_equal(d_g, d_w), f"{int(np.unpackbits(d_g ^ d_w).sum())} descriptor bits differ"
    assert np.array_equal(np.isnan(x_g), np.isnan(x_w))
    assert np.array_equal(np.nan_to_num(x_g).view(np.uint32), np.nan_to_num(x_w).view(np.uint32)), "3-D points differ"


def gftt_engine(gp: gftt_py.GfttParams = gftt_py.GfttParams()) -> Engine:
    eng = Engine()
    eng.set_detector(LCD_DETECTOR_GFTT_ORB, Engine.gftt_params(gp.quality_level, gp.min_distance, gp.block_size))
    return eng


@pytest.mark.parametrize("hw", [(480, 640), (720, 1280), (252, 332), (244, 324), (241, 333)])
@pytest.mark.parametrize("block", [3, 5, 7])
def test_min_eigenvalue_map_is_cv2s(hw, block):
    import cv2

    h, w = hw
    imgs = np.stack([synth.make_image(h, w, 70 + i) for i in range(2)])
    eng = gftt_engine(gftt_py.GfttParams(block_size=block))
    eng.orb_detect_describe(imgs, None, Engine.orb_params(K4, n_features=500, depth_as_mask=False))
    lam = eng.debug_orb_buffer(10, 2 * h * w * 4, np.float32).reshape(2, h, w)
    for i in range(2):
        want = cv2.cornerMinEigenVal(imgs[i], block, 3)
        assert np.array_equal(lam[i].view(np.uint32), want.view(np.uint32)), f"frame {i}: {int((lam[i] != want).sum())} pixels differ"


@pytest.mark.parametrize("seed", [5, 6])
@pytest.mark.parametrize("gp", [gftt_py.GfttParams(), gftt_py.GfttParams(0.01, 4.5, 5), gftt_py.GfttParams(0.001, 1.0, 3), gftt_py.GfttParams(0.001, 0.0, 7)],
                         ids=["default", "q01_d4.5_b5", "d1", "d0_b7"])
def test_gftt_gray_with_u16_depth(seed, gp):
    img = synth.make_image(480, 640, seed)
    depth = synth.make_depth(480, 640, seed + 10)
    eng = gftt_engine(gp)
    got = eng.orb_detect_describe(img[None], depth[None], Engine.orb_params(K4))[0]
    want = gftt_py.detect_describe(img, depth, K4, f2d.OrbParams(), gp)
    assert len(want[0]) > 500
    check_frame(got, want)


def test_gftt_bgr_float_depth_batch_min_max_depth():
    imgs = np.stack([synth.make_image(480, 640, 20 + i, bgr=True) for i in range(3)])
    depth = np.stack([synth.make_depth(480, 640, 30 + i, as_float=True) for i in range(3)])
    eng = gftt_engine()
    got = eng.orb_detect_describe(imgs, depth, Engine.orb_params(K4, min_depth=0.5, max_depth=3.5))
    for i in range(3):
        check_frame(got[i], gftt_py.detect_describe(imgs[i], depth[i], K4, f2d.OrbParams(min_depth=0.5, max_depth=3.5)))


def test_gftt_no_depth_low_texture_and_textureless():
    imgs = np.stack([synth.make_image(240, 320, 3, n_rects=40), np.full((240, 320), 7, np.uint8)])
    eng = gftt_engine()
    op = Engine.orb_params(K4, n_features=400, depth_as_mask=False)
    got = eng.orb_detect_describe(imgs, None, op)
    p = f2d.OrbParams(n_features=400, depth_as_mask=False)
    for i in range(2):
        check_frame(got[i], gftt_py.detect_describe(imgs[i], None, K4, p))
    assert len(got[1][0]) == 0 and np.isnan(got[0][2]).all()


@pytest.mark.parametrize("nf", [100, 1000, 4000])
def test_gftt_max_corners_and_edge_threshold_31(nf):
    img = synth.make_image(480, 640, 12)
    eng = gftt_engine()
    # GFTT never returns more than maxCorners keypoints: cap = nf holds them (4000 + 256 would pass the 4096 rows per frame)
    got = eng.orb_detect_describe(img[None], None, Engine.orb_params(K4, n_features=nf, edge_threshold=31, depth_as_mask=False), cap=nf)[0]
    check_frame(got, gftt_py.detect_describe(img, None, K4, f2d.OrbParams(n_features=nf, edge_threshold=31, depth_as_mask=False)))


@pytest.mark.parametrize("hw", [(720, 1280), (252, 332), (241, 333), (121, 163)])
def test_gftt_sizes(hw):
    """1280x720 holds more candidates than one sorted chunk; the others are not multiples of 16 (the scalar tail of the Sobel row pass,
    no tensor map) or of 2 (general preparation kernel)."""
    h, w = hw
    img = synth.make_image(h, w, 61)
    depth = synth.make_depth(h, w, 62)
    k4 = (910.0, 910.0, w / 2, h / 2)
    eng = gftt_engine()
    got = eng.orb_detect_describe(img[None], depth[None], Engine.orb_params(k4))[0]
    want = gftt_py.detect_describe(img, depth, k4, f2d.OrbParams())
    assert len(want[0]) > 10
    check_frame(got, want)


def _samples():
    import cv2
    from pathlib import Path

    z = np.load(Path(__file__).resolve().parent / "golden" / "samples_c1.npz")
    off = z["offsets"]
    return [cv2.imdecode(z["jpeg"][off[i]:off[i + 1]], cv2.IMREAD_COLOR) for i in range(len(off) - 1)]


def test_gftt_c1_sample_images():
    imgs = _samples()
    eng = gftt_engine()
    K4s = (400.0, 400.0, 256.0, 192.0)
    for nf in (1000, 150):
        out = eng.orb_detect_describe(np.stack(imgs), None, Engine.orb_params(K4s, n_features=nf))
        for i, im in enumerate(imgs):
            check_frame(out[i], gftt_py.detect_describe(im, None, K4s, f2d.OrbParams(n_features=nf)))


def test_gftt_candidate_overflow_is_reported():
    rng = np.random.default_rng(1)
    noise = rng.integers(0, 256, (1, 1080, 1920), dtype=np.uint8)  # ~138k local maxima above the quality threshold
    eng = gftt_engine()
    with pytest.raises(LcdError) as ei:
        eng.orb_detect_describe(noise, None, Engine.orb_params(K4, depth_as_mask=False))
    assert ei.value.code == LCD_ERR_CAPACITY
    assert eng.orb_overflow()


def test_gftt_invalid_parameters_raise():
    eng = Engine()
    for gp in (Engine.gftt_params(quality_level=0.0), Engine.gftt_params(min_distance=-1.0), Engine.gftt_params(block_size=4),
               Engine.gftt_params(use_harris=True)):
        with pytest.raises(LcdError):
            eng.set_detector(LCD_DETECTOR_GFTT_ORB, gp)
    with pytest.raises(LcdError):
        eng.set_detector(LCD_DETECTOR_GFTT_ORB, None)
    with pytest.raises(LcdError):
        eng.set_detector(6, Engine.gftt_params())
    eng.set_detector(LCD_DETECTOR_GFTT_ORB, Engine.gftt_params())
    img = np.zeros((1, 240, 320), np.uint8)
    with pytest.raises(LcdError):
        eng.orb_detect_describe(img, None, Engine.orb_params(K4, patch_size=15))


def test_orb_after_switching_detectors_equals_a_fresh_engine():
    imgs = np.stack([synth.make_image(480, 640, 40 + i, bgr=True) for i in range(2)])
    depth = np.stack([synth.make_depth(480, 640, 50 + i) for i in range(2)])
    op = Engine.orb_params(K4)
    fresh = Engine().orb_detect_describe(imgs, depth, op)
    eng = Engine()
    eng.orb_detect_describe(imgs, depth, op)
    eng.set_detector(LCD_DETECTOR_GFTT_ORB, Engine.gftt_params())
    g = eng.orb_detect_describe(imgs, depth, op)
    check_frame(g[0], gftt_py.detect_describe(imgs[0], depth[0], K4, f2d.OrbParams()))
    eng.set_detector(LCD_DETECTOR_ORB)
    again = eng.orb_detect_describe(imgs, depth, op)
    for a, b in zip(fresh, again):
        for x, y in zip(a, b):
            assert np.array_equal(np.nan_to_num(x).view(np.uint8), np.nan_to_num(y).view(np.uint8))


def _gftt_world():
    p = f2d.OrbParams(n_features=600)
    gp = gftt_py.GfttParams()
    orb_fn = lambda img, dep: gftt_py.detect_describe(img, dep, K4, p, gp)
    return synth.make_place_world(orb_fn, n_places=5, n_words=2800, n_signatures=120, feats=600, height=240, width=320, seed=9)


def _load(d, world):
    d.add_words(world.word_ids, world.vocab)
    d.last_word_id = int(world.word_ids.max())
    d.update()
    d.load_csr(world.smap.word_ids, world.smap.row_ptr, world.smap.sig, world.smap.cnt)
    d.set_ni(world.smap.sig_ids, world.smap.ni)


def test_process_frames_gftt_orb_full_path_matches_oracle():
    from oracle import oracle_py as orc
    from rtabmap_b200.capi import VerifyResult

    world = _gftt_world()
    imgs, deps, places = synth.make_view_frames(world, 4, seed=5, max_shift=4)
    imgs[3] = 7
    eng = gftt_engine()
    o = orc.OracleDictionary()
    for d in (eng, o):
        _load(d, world)
    eng.sig_add_batch(world.smap.sig_ids, world.store.desc, world.store.xyz, world.smap.ni)
    K4s = (262.5, 262.5, 160.0, 120.0)
    op = Engine.orb_params(K4s, n_features=600)
    vp = Engine.verify_params(K4s)
    nkp, words, like, hyp, res = eng.process_frames(imgs, deps, op, world.smap.sig_ids, 121, vp)
    p2 = f2d.OrbParams(n_features=600)
    n_ok = 0
    for b in range(4):
        kp, d, x = gftt_py.detect_describe(imgs[b], deps[b], K4s, p2)
        assert nkp[b] == len(kp)
        if len(kp) == 0:
            assert not res[b]["ok"] and (words[b] == 0).all()
            continue
        w_o, l_o = o.localize_ro(d, world.smap.sig_ids, 121)
        assert np.array_equal(words[b][:len(w_o)], w_o) and (words[b][len(w_o):] == 0).all()
        assert np.allclose(like[b], l_o, atol=1e-4, rtol=1e-4)
        h = int(np.argmax(l_o))
        assert hyp[b] == world.smap.sig_ids[h]
        n = int(world.smap.ni[h])
        v = orc.verify_pair(world.store.desc[h][:n], world.store.xyz[h][:n], d, kp[:, :2], K4s)
        assert res[b]["ok"] == v["ok"] and res[b]["n_matches"] == len(v["matches"]) and res[b]["n_inliers"] == len(v["inliers"])
        n_ok += int(res[b]["ok"])
    assert n_ok >= 2
    # the pipelined pair computes the same
    n = len(imgs)
    o_nkp = np.zeros(n, np.int32)
    o_words = np.zeros_like(words)
    o_like = np.zeros_like(like)
    o_hyp = np.zeros(n, np.int32)
    o_res = (VerifyResult * n)()
    eng.process_frames_submit(imgs, deps, op, world.smap.sig_ids, 121, vp, o_nkp, o_words, o_like, o_hyp, o_res)
    eng.process_frames_wait()
    assert np.array_equal(o_nkp, nkp) and np.array_equal(o_words, words) and np.array_equal(o_like, like) and np.array_equal(o_hyp, hyp)


def test_gftt_mapping_stream_equals_per_call_sequence():
    rng = np.random.default_rng(3)
    op = Engine.orb_params(K4, n_features=500)
    base_img = [synth.make_image(240, 320, 900 + p, bgr=True) for p in range(3)]
    base_dep = [synth.make_depth(240, 320, 950 + p) for p in range(3)]
    frames = [synth.render_view(base_img[t % 3], base_dep[t % 3], int(rng.integers(-4, 5)), int(rng.integers(-4, 5)), 2.0, rng) for t in range(8)]
    pipe, seq = gftt_engine(), gftt_engine()
    pipe.map_detect_async(frames[0][0], frames[0][1], op)
    for t in range(len(frames)):
        sig = t + 1
        if t + 1 < len(frames):
            pipe.map_detect_async(frames[t + 1][0], frames[t + 1][1], op)
        wm = np.arange(1, max(sig - 2, 1), dtype=np.int32)
        n_kp, words, n_new, like, kp, desc, xyz = pipe.map_frame(sig, wm, sig, want_features=True)
        kp_s, desc_s, xyz_s = seq.orb_detect_describe(frames[t][0][None], frames[t][1][None], op, cap=500)[0]
        seq.update()
        w_s, n_new_s = seq.quantize(desc_s, sig)
        assert n_kp == len(kp_s) and np.array_equal(desc, desc_s) and np.array_equal(xyz, xyz_s, equal_nan=True)
        assert np.array_equal(words, w_s) and n_new == n_new_s, f"frame {t}"
        _, d_o, x_o = gftt_py.detect_describe(frames[t][0], frames[t][1], K4, f2d.OrbParams(n_features=500))
        assert np.array_equal(desc, d_o) and np.array_equal(xyz, x_o, equal_nan=True)


def test_gftt_single_rank_sharded_step_equals_the_unsharded_call():
    import torch

    eng = Engine(max_words=8192, max_signatures=400)
    eng.set_detector(LCD_DETECTOR_GFTT_ORB, Engine.gftt_params())
    op = Engine.orb_params(synth.CAMERA_K4, n_features=300)
    world = synth.make_place_world(lambda im, dp: eng.orb_detect_describe(im[None], dp[None], op, cap=300)[0], 6, 1500, 120, 300, 240, 320)
    sm = world.smap
    eng.add_words(world.word_ids, world.vocab)
    eng.last_word_id = int(world.word_ids.max())
    eng.update()
    eng.load_csr(sm.word_ids, sm.row_ptr, sm.sig, sm.cnt)
    eng.set_ni(sm.sig_ids, sm.ni)
    eng.sig_add_batch(sm.sig_ids, world.store.desc, world.store.xyz, sm.ni)
    imgs, deps, places = synth.make_view_frames(world, 3, seed=4)
    vp = Engine.verify_params(synth.CAMERA_K4, image_size=(320, 240))
    nf, ns = len(imgs), len(sm.sig_ids)
    d_img = torch.from_numpy(imgs).cuda()
    d_dep = torch.from_numpy(deps.view(np.int16)).cuda()
    d_sig = torch.from_numpy(sm.sig_ids).cuda()
    d_rowids = torch.from_numpy(world.word_ids).cuda()
    ext = torch.cuda.ExternalStream(eng.stream)
    with torch.cuda.stream(ext):
        w0 = torch.zeros(nf * 300, dtype=torch.int32, device="cuda")
        l0 = torch.zeros(nf * ns, dtype=torch.float32, device="cuda")
        eng.process_frames_dev(d_img.data_ptr(), nf, 320, 240, 3, d_dep.data_ptr(), 1, op, d_sig.data_ptr(), ns, ns + 1, vp, w0.data_ptr(), l0.data_ptr(),
                               True, 0.8, True)
        hyp0, res0 = eng.process_fetch(nf)
        eng.shard_comm_init(Engine.shard_unique_id(), 0, 1)
        w1 = torch.zeros(nf * 300, dtype=torch.int32, device="cuda")
        l1 = torch.zeros(nf * ns, dtype=torch.float32, device="cuda")
        eng.shard_process_frames_dev(d_img.data_ptr(), nf, 320, 240, 3, d_dep.data_ptr(), 1, op, d_sig.data_ptr(), ns, ns + 1, d_rowids.data_ptr(),
                                     int(world.word_ids.max()), vp, w1.data_ptr(), l1.data_ptr(), True, 0.8, True)
        hyp1, res1 = eng.process_fetch(nf)
        eng.shard_comm_destroy()
    assert torch.equal(w0, w1) and torch.equal(l0, l1)
    assert np.array_equal(hyp0, hyp1) and (hyp0 > 0).all()
    for a, b in zip(res0, res1):
        assert a["ok"] == b["ok"] and a["n_inliers"] == b["n_inliers"] and np.array_equal(a["rvec"], b["rvec"])


def test_gftt_shim_driver_equals_the_oracle(tmp_path):
    import subprocess
    from pathlib import Path

    root = Path(__file__).resolve().parent.parent
    lib = root / "rtabmap_b200" / "lib"
    exe = tmp_path / "gftt_shim_driver"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-I", str(root / "integration" / "stubs"), "-I", str(root / "include"),
                        str(root / "integration" / "gftt_shim_driver.cpp"), str(root / "integration" / "GFTT_ORB_B200.cpp"), "-o", str(exe),
                        "-L", str(lib), "-llcd_b200", f"-Wl,-rpath,{lib}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    img = synth.make_image(480, 640, 33)
    depth = synth.make_depth(480, 640, 34)
    mask = f2d.depth_mask(depth, f2d.OrbParams())
    img.tofile(tmp_path / "img.raw")
    mask.tofile(tmp_path / "mask.raw")
    out = tmp_path / "out.bin"
    r = subprocess.run([str(exe), str(tmp_path / "img.raw"), "640", "480", str(tmp_path / "mask.raw"), "800", str(out)], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0 and "gftt shim driver ok" in r.stdout, r.stdout + r.stderr
    raw = out.read_bytes()
    n = int(np.frombuffer(raw[:4], np.int32)[0])
    kp = np.frombuffer(raw[4:4 + n * 24], np.float32).reshape(n, 6)
    desc = np.frombuffer(raw[4 + n * 24:], np.uint8).reshape(n, 32)
    kp_o, d_o, _ = gftt_py.detect_describe(img, depth, K4, f2d.OrbParams(n_features=800))
    assert n == len(kp_o) > 300
    assert np.array_equal(kp.view(np.uint32), kp_o.view(np.uint32)) and np.array_equal(desc, d_o)
