"""oracle/gftt_py.py (the written spec of rtabmap_b200/csrc/gftt.cuh) against opencv-python: cv2.cornerMinEigenVal bit for bit, and
cv2.GFTTDetector's keypoints, order and response bits.  Plus the GFTT/ORB reference-side shim compiled and linked against the C ABI."""
import subprocess
from pathlib import Path

import cv2
import numpy as np
import pytest

from oracle import gftt_py
from rtabmap_b200 import synth

ROOT = Path(__file__).resolve().parent.parent


def _samples():
    z = np.load(ROOT / "tests" / "golden" / "samples_c1.npz")
    off = z["offsets"]
    return [cv2.cvtColor(cv2.imdecode(z["jpeg"][off[i]:off[i + 1]], cv2.IMREAD_COLOR), cv2.COLOR_BGR2GRAY) for i in range(len(off) - 1)]


def _cv_detect(gray, n, q, md, bs, mask):
    kps = cv2.GFTTDetector_create(n, q, md, bs).detect(gray, mask)
    return np.array([[k.pt[0], k.pt[1], k.size, k.angle, k.response, k.octave] for k in kps], np.float32).reshape(-1, 6)


@pytest.mark.parametrize("hw", [(480, 640), (720, 1280), (252, 332), (244, 324), (241, 333)])
@pytest.mark.parametrize("block", [3, 5, 7])
def test_min_eigenvalue_replay_is_bit_exact(hw, block):
    img = synth.make_image(*hw, 5)
    got = gftt_py.min_eigen_val(img, block)
    want = cv2.cornerMinEigenVal(img, block, 3)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), int((got != want).sum())


@pytest.mark.parametrize("block", [3, 5, 7])
def test_min_eigenvalue_replay_on_the_c1_samples(block):
    for i, g in enumerate(_samples()[::3]):
        got = gftt_py.min_eigen_val(g, block)
        assert np.array_equal(got.view(np.uint32), cv2.cornerMinEigenVal(g, block, 3).view(np.uint32)), f"sample {i}"


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("md", [7.0, 4.5, 1.0, 0.0])
@pytest.mark.parametrize("q", [0.001, 0.01])
@pytest.mark.parametrize("n", [100, 1000, 4000])
def test_selection_replay_equals_gftt_detector(masked, md, q, n):
    img = synth.make_image(480, 640, 8)
    mask = np.where(synth.make_depth(480, 640, 18) > 0, 255, 0).astype(np.uint8) if masked else None
    got = gftt_py.detect(img, n, q, md, 3, mask)
    want = _cv_detect(img, n, q, md, 3, mask)
    assert got.shape == want.shape and np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_selection_replay_on_the_c1_samples_and_other_block_sizes():
    for i, g in enumerate(_samples()[::4]):
        for bs, md in ((3, 7.0), (5, 4.5), (7, 2.5)):
            assert np.array_equal(gftt_py.detect(g, 1000, 0.001, md, bs).view(np.uint32), _cv_detect(g, 1000, 0.001, md, bs, None).view(np.uint32)), (i, bs)


def test_candidate_ties_are_ordered_by_address_descending():
    """Equal eigenvalues are common (about 470 ties among the candidates of a VGA frame): their order is the address order, reversed."""
    img = synth.make_image(480, 640, 5)
    eig = gftt_py.min_eigen_val(img, 3)
    idx = gftt_py.candidates(eig, 0.001)
    lam = eig.ravel()[idx]
    tie = lam[1:] == lam[:-1]
    assert tie.sum() > 50 and (idx[1:][tie] < idx[:-1][tie]).all()


def test_gftt_shim_compiles_and_links_against_the_c_abi(tmp_path):
    import rtabmap_b200

    rtabmap_b200.load_library()
    lib = ROOT / "rtabmap_b200" / "lib"
    objs = []
    for src in ("GFTT_ORB_B200.cpp", "ORB_B200.cpp"):
        obj = tmp_path / (src + ".o")
        r = subprocess.run(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-fPIC", "-I", str(ROOT / "integration" / "stubs"), "-I", str(ROOT / "include"),
                            "-c", str(ROOT / "integration" / src), "-o", str(obj)], capture_output=True, text=True)
        assert r.returncode == 0, f"{src}:\n{r.stderr}"
        objs.append(str(obj))
    exe = tmp_path / "gftt_shim_driver"
    r = subprocess.run(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", str(ROOT / "integration" / "stubs"), "-I", str(ROOT / "include"),
                        str(ROOT / "integration" / "gftt_shim_driver.cpp"), *objs, "-o", str(exe), "-L", str(lib), "-llcd_b200", "-Wl,--no-undefined",
                        f"-Wl,-rpath,{lib}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
