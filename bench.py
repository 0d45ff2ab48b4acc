#!/usr/bin/env python
"""bench.py — loop-closure queries/sec on B200 (BASELINE.json metric) + roofline + CPU baseline.

    python bench.py --gpus 1 --steps 30 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference          # the reference's CPU algorithm on the host cores
    python bench.py --dump-outputs DIR        # + what the last timed step returned, as DIR/<name>.npy

Workload = BASELINE.json configs[1]: 640x480 synthetic RGB-D stream, ORB 1000 kp/frame, 49 152-word binary
dictionary, 10 000 signatures.  One "step" = one batch of B independent loop-closure queries (frames); each
frame goes through the WHOLE hot path:
  detect   BGR->gray, depth mask, ORB detect + describe, 3-D lifting      (Memory::createSignature feature block)
  quantise exact 2-NN + NNDR + intra-frame new words against the dictionary (VWDictionary::addNewWords)
  score    TF-IDF over the inverted index of all signatures                (Memory::computeLikelihood)
  verify   top hypothesis: descriptor matching + PnP RANSAC + refinement   (Memory::computeTransform)
The map is built (untimed) from 50 textured places seen 200 times each; the vocabulary is made of the
places' own ORB descriptors, query frames are shifted, noisy re-observations of random places, so the
likelihood arg-max is a true loop closure and its verification succeeds.

`value`   frames/s with images + depth already resident in HBM (CUDA events on the engine stream).
`e2e`     frames/s through the host-buffer C-ABI call lcd_process_frames (pinned host images + depth in,
          word ids + likelihood + verified poses out; H2D/D2H inside the timed region).
`roofline` the dictionary-NN kernel (knn2_tensor_kernel; knn2_hamming_kernel with LCD_NN_TENSOR=0), timed live with CUDA events on its stream.
`cpu_baseline` / --impl reference: cv2.ORB + the oracle port of the reference algorithm on the host cores.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)

W_WORDS = 49152
S_SIGS = 10000
F_FEATS = 1000
N_PLACES = 50
IMG_W, IMG_H = 640, 480
DESC_BYTES = 32
NNDR = 0.8
KCAM = (525.0, 525.0, 320.0, 240.0)
METRIC = "loop-closure queries/sec"
UNIT = "queries/s"
STAGES = ["detect(bgr->gray, depth mask, orb detect+describe, 3-D lifting)", "quantise(knn2+nndr+new-words)", "score(tf-idf)",
          "verify(top-1 hypothesis: descriptor matching + pnp-ransac + refinement)"]


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


def tensor_peak_tops():
    """Dense s8 tensor peak in Tera-op/s: MEASURED_PEAKS.json holds the measured bf16 figure (burst: the kernel is timed
    alone); tcgen05 kind::i8 runs at twice the bf16 rate (K=32 per instruction against K=16), so the s8 roof is 2x it."""
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        if "bf16_tflops" in d:
            return 2.0 * float(d["bf16_tflops"]), "2 x measured bf16 dense (MEASURED_PEAKS.json bf16_tflops, burst)"
    return 2.0 * 2250.0, "2 x nominal bf16 dense (B200_PROFILING.md fallback)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(index)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.p:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


DUMP_LIMIT_BYTES = 64_000_000


def step_outputs(words, like, hyp=None, res=None) -> dict:
    """What a caller of the timed path receives for the frames of one step, one row per frame: word ids, likelihood rows and, where the
    step verifies, the hypotheses and the verification results.  Integers as float64 (exact), floats at their own precision."""
    out = {"words": np.asarray(words, np.float64), "likelihood": np.asarray(like, np.float32)}
    if hyp is not None:
        out["hypothesis"] = np.asarray(hyp, np.float64)
        for k in ("ok", "n_matches", "n_inliers", "iterations_run"):
            out["verify_" + k] = np.array([r[k] for r in res], np.float64)
        out["verify_rvec"] = np.stack([r["rvec"] for r in res]).astype(np.float64)
        out["verify_tvec"] = np.stack([r["tvec"] for r in res]).astype(np.float64)
        out["verify_transform"] = np.stack([r["transform"] for r in res]).astype(np.float32)
        out["verify_covariance"] = np.stack([r["covariance"] for r in res]).astype(np.float64)
    return out


def dump_outputs(out_dir: str, outputs: dict, prefix: str = "") -> None:
    """Write `outputs` (step_outputs) as out_dir/<prefix><name>.npy, and the frames they hold as <prefix>frame_index.npy.  Beyond
    DUMP_LIMIT_BYTES in all (.npy headers included), the same fixed, seeded sample of frames is kept from every array."""
    n = len(outputs["words"])
    per_frame = sum(a.nbytes for a in outputs.values()) // max(n, 1) + 8
    keep = min(n, (DUMP_LIMIT_BYTES - 1024 * (len(outputs) + 1)) // per_frame)
    if keep == 0:
        raise SystemExit(f"--dump-outputs: one frame's outputs ({per_frame} bytes) exceed {DUMP_LIMIT_BYTES} bytes")
    frames = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / f"{prefix}frame_index.npy", frames.astype(np.float64))
    for name, a in outputs.items():
        np.save(d / f"{prefix}{name}.npy", a[frames])
    log(f"wrote the outputs of the last timed step ({keep} of {n} frames) to {d}")


def parallelism_text(world_size: int, batch: int) -> str:
    if world_size == 1:
        return "single GPU"
    return (f"x{world_size}: every GPU detects and verifies its own {batch} frames per step, dictionary + inverted index sharded by word range; "
            "exchanges inside the C ABI (lcd_shard_process_frames): all-gather(descriptors, top-2 keys, word ids) + sparse score exchange over NCCL")


def job_config(args, world_size: int):
    """The `config` object of the JSON line: identical for the GPU arm and the reference arm of the same job (the CPU arm times a
    bounded sample of it, described in its cpu_baseline.sample)."""
    batch = args.batch * world_size
    return {
        "workload": "BASELINE configs[1]: 640x480 synthetic RGB-D stream, ORB 1000 kp/frame, 49k-word binary dictionary, 10k signatures",
        "frames": "every query a shifted, noisy revisit of a mapped place" if args.workload == "revisit" else
                  "mixed: 30 % never-seen places, 40 % rotated (+-12 deg) / scaled (0.85-1.15) / shifted revisits, 30 % plain revisits (SURVEY 8(d))",
        "words": W_WORDS, "signatures": S_SIGS, "features_per_frame": F_FEATS, "descriptor_bytes": DESC_BYTES, "image": f"{IMG_W}x{IMG_H} BGR8 + depth16",
        "places": N_PLACES, "frames_per_step": batch, "frames_per_gpu": args.batch,
        "mode": "localisation (frozen dictionary + map; per-frame insert/score/roll-back semantics, SURVEY App. C.5)",
        "stages": STAGES,
        "params": "Kp/DetectorStrategy=2 ORB(3 levels, scale 2, edge 19, FAST 20), Kp/MaxFeatures=1000, Mem/DepthAsMask, exact NN (Kp/NNStrategy=0 order), "
                  "Kp/NndrRatio=0.8, Kp/NewWordsComparedTogether, Kp/IncrementalDictionary, Vis/Iterations=300, Vis/PnPReprojError=2, Vis/MinInliers=20, "
                  "Vis/PnPRefineIterations=1, Vis/CorNNDR=0.8, Vis/PnPVarianceMedianRatio=4; hypothesis = raw-likelihood arg-max",
        "l2": "flushed between timed steps (256 MiB write, outside the timed events)",
        "parallelism": parallelism_text(world_size, args.batch),
    }


# ------------------------------------------------------------------------- CPU (reference) arm
def cv2_orb_fn():
    from oracle import feature2d_py as f2d
    from rtabmap_b200 import synth

    p = f2d.OrbParams(n_features=F_FEATS)
    return lambda img, dep: f2d.detect_describe(img, dep, synth.CAMERA_K4, p)


class CpuReference:
    """The reference's CPU algorithm for one frame: cv2.ORB (the OpenCV the reference calls), the index search by the REFERENCE'S OWN
    rtflann compiled from /root/reference (oracle/_ref/libref_flann.so: FlannIndex::knnSearch on the LinearIndex, Kp/NNStrategy=0) when that
    library travelled with the repo, and the oracle port for the rest (NNDR / new-word loop, TF-IDF over std::map, computeTransform)."""

    def __init__(self, world):
        from oracle import oracle_py as orc

        self.orc = orc
        self.world = world
        self.orb = cv2_orb_fn()
        o = orc.OracleDictionary(0, DESC_BYTES, True, NNDR, True)
        o.add_words(world.word_ids, world.vocab)
        o.last_word_id = int(world.word_ids.max())
        o.update()
        o.load_csr(world.smap.word_ids, world.smap.row_ptr, world.smap.sig, world.smap.cnt)
        o.set_ni(world.smap.sig_ids, world.smap.ni)
        self.o = o
        self.rtflann = orc.ref_lib() is not None
        self.vocab = np.ascontiguousarray(world.vocab)  # rows in search order (ascending word id)

    def legs(self):
        nn = "reference (rtflann LinearIndex compiled from /root/reference, 1 thread per frame)" if self.rtflann else "port (oracle scalar popcount scan)"
        return {"detect": "cv2.ORB 4.13 (the OpenCV the reference calls) + port of Feature2D's wrapper", "nn": nn,
                "nndr+new words+tf-idf": "port (std::multimap / std::map as in the reference)", "verify": "port (restated cv3::solvePnPRansac + refinement)"}

    def one(self, img, dep):
        w = self.world
        kp, d, x = self.orb(img, dep)
        if self.rtflann and len(d):
            ki, kd = self.orc.ref_knn2(self.vocab, d)
            words, like = self.o.localize_ro_knn(d, ki, kd, w.smap.sig_ids, S_SIGS + 1)
        else:
            words, like = self.o.localize_ro(d, w.smap.sig_ids, S_SIGS + 1)
        h = int(np.argmax(like))
        if like[h] <= 0:
            return kp, d, words, like, 0, {"ok": False, "inliers": [], "matches": [], "rvec": np.zeros(3), "tvec": np.zeros(3)}, x
        n = int(w.smap.ni[h])
        v = self.orc.verify_pair_cov(w.store.desc[h][:n], w.store.xyz[h][:n], d, kp[:, :2], KCAM, xyz_to=x, image_size=(IMG_W, IMG_H))
        return kp, d, words, like, int(w.smap.sig_ids[h]), v, x

    def rate(self, imgs, deps, n_frames: int, threads: int):
        import cv2

        cv2.setNumThreads(1)  # parallelism is over frames
        t0 = time.perf_counter()
        if threads <= 1:
            res = [self.one(imgs[b], deps[b]) for b in range(n_frames)]
        else:
            with ThreadPoolExecutor(threads) as ex:
                res = list(ex.map(lambda b: self.one(imgs[b], deps[b]), range(n_frames)))
        dt = time.perf_counter() - t0
        return n_frames / dt, dt, res


def run_reference(args):
    from rtabmap_b200 import synth

    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    if args.config == "c4":
        return run_reference_c4(args)
    threads = max(1, min(os.cpu_count() or 1, args.ref_threads or (os.cpu_count() or 1)))
    world = synth.make_place_world(cv2_orb_fn(), N_PLACES, W_WORDS, S_SIGS, F_FEATS, IMG_H, IMG_W)
    ref = CpuReference(world)
    # one step = a bounded sample of the workload: `per_step` frames spread over all host threads.  The sample is sized from one
    # probe step so that the --steps / --warmup the caller asked for finish in about two minutes.
    per_step = threads
    imgs, deps, places = synth.make_view_frames(world, per_step, mode=args.workload)
    _, probe_s, _ = ref.rate(imgs, deps, per_step, threads)
    budget_s = float(os.environ.get("LCD_REF_BUDGET_S", "120"))
    n_calls = args.steps + args.warmup
    if probe_s * n_calls > budget_s:
        per_step = int(max(min(threads, 8), per_step * budget_s / (probe_s * n_calls)))
        imgs, deps, places = imgs[:per_step], deps[:per_step], places[:per_step]
    for _ in range(args.warmup):
        ref.rate(imgs, deps, per_step, threads)
    total = 0.0
    for _ in range(args.steps):
        _, dt, res = ref.rate(imgs, deps, per_step, threads)
        total += dt
    value = per_step * args.steps / total
    known = places >= 0
    hit = float(np.mean([world.sig_place[r[4] - 1] == places[b] if r[4] > 0 else False for b, r in enumerate(res) if known[b]])) if known.any() else None
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "config": job_config(args, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "reference" if ref.rtflann else "port", "legs": ref.legs(),
                         "sample": f"{per_step} frames/step x {args.steps} steps (+{args.warmup} warm-up) of the same workload, frames spread over "
                                   f"{threads} host threads (one frame per thread at a time); probe step {probe_s:.1f} s"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "top1_place_hit_rate": hit, "verified_rate": float(np.mean([r[5]["ok"] for r in res])),
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------- GPU arm
def run_b200(args):
    import torch
    import torch.distributed as dist

    from rtabmap_b200 import Engine, sharding, synth

    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world_size != args.gpus:
        log(f"warning: --gpus {args.gpus} but WORLD_SIZE={world_size}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl b200) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    if world_size > 1:
        # NCCL's communicator lines (rank count, transport) go to stderr for the driver to read; stdout carries exactly one JSON line
        # (NCCL would print them to stdout; a file per process keeps stdout clean, rank 0 copies the lines to stderr at the end)
        if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
            os.environ["NCCL_DEBUG"] = "INFO"
            os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        os.environ["NCCL_DEBUG_FILE"] = os.path.join(tempfile.gettempdir(), f"lcd_nccl_{os.getpid()}.log")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    # weak scaling: every GPU brings its own --batch frames per step (a relocalisation service adds cameras with GPUs); the
    # dictionary and the inverted index are sharded by word range, so each rank still searches ALL frames' descriptors.
    BL = args.batch                # frames per step detected and verified by this rank
    B = BL * world_size            # frames per step of the whole job
    n_pool = 3

    # capacity hints with the headroom the mapping-mode extra needs (52 more signatures, ~30k more words): growing a 440 MB signature
    # store in the middle of a stream costs one cudaMalloc + copy (300 ms measured); a mapping session sizes its engine for the session
    eng = Engine(device=local, desc_dim=DESC_BYTES, max_words=W_WORDS + 65536, max_signatures=S_SIGS + 128, max_queries=F_FEATS, max_batch=B)
    op = Engine.orb_params(KCAM, n_features=F_FEATS)
    vp = Engine.verify_params(KCAM, image_size=(IMG_W, IMG_H))

    def gpu_orb_fn(img, dep):
        return eng.orb_detect_describe(img[None], dep[None], op, cap=F_FEATS)[0]

    t0 = time.time()
    world = synth.make_place_world(gpu_orb_fn, N_PLACES, W_WORDS, S_SIGS, F_FEATS, IMG_H, IMG_W)
    imgs_all, deps_all, places = synth.make_view_frames(world, BL * n_pool, seed=3 + rank, mode=args.workload)  # this rank's frames only
    log(f"[rank {rank}] world built in {time.time() - t0:.1f}s: {len(world.vocab)} words, {world.smap.nnz} postings")

    r0, r1 = sharding.shard_rows(W_WORDS, world_size, rank)
    ids, vocab, smap = world.word_ids, world.vocab, world.smap
    eng.add_words(ids[r0:r1], vocab[r0:r1])
    eng.last_word_id = W_WORDS
    eng.update()
    if world_size > 1:
        eng.shard_set_row_offset(r0)
        w_, p_, s_, c_ = sharding.shard_csr(smap.word_ids, smap.row_ptr, smap.sig, smap.cnt, ids[r0:r1])
        eng.load_csr(w_, p_, s_, c_)
    else:
        eng.load_csr(smap.word_ids, smap.row_ptr, smap.sig, smap.cnt)
    eng.set_ni(smap.sig_ids, smap.ni)
    for s0 in range(0, S_SIGS, 1000):  # signature store, replicated on every rank
        eng.sig_add_batch(smap.sig_ids[s0:s0 + 1000], world.store.desc[s0:s0 + 1000], world.store.xyz[s0:s0 + 1000], smap.ni[s0:s0 + 1000])

    ext = torch.cuda.ExternalStream(eng.stream, device=local)
    torch.cuda.set_stream(ext)
    nq = B * F_FEATS
    f0, f1 = rank * BL, (rank + 1) * BL  # this rank's rows in the job-wide (all-gathered) arrays
    nf = BL
    d_img = [torch.from_numpy(imgs_all[k * BL:(k + 1) * BL]).cuda() for k in range(n_pool)]
    d_dep = [torch.from_numpy(deps_all[k * BL:(k + 1) * BL].view(np.int16)).cuda() for k in range(n_pool)]
    h_img = [torch.from_numpy(imgs_all[k * BL:(k + 1) * BL]).pin_memory() for k in range(n_pool)]
    h_dep = [torch.from_numpy(deps_all[k * BL:(k + 1) * BL].view(np.int16)).pin_memory() for k in range(n_pool)]
    d_sig = torch.from_numpy(smap.sig_ids).cuda()
    h_sig = torch.from_numpy(smap.sig_ids).pin_memory()
    d_words = torch.zeros(nq, dtype=torch.int32, device="cuda")
    d_like = torch.zeros(B * S_SIGS, dtype=torch.float32, device="cuda")
    h_words = torch.zeros((B, F_FEATS), dtype=torch.int32).pin_memory()
    h_like = torch.zeros((B, S_SIGS), dtype=torch.float32).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    img_bytes = IMG_W * IMG_H * 3
    dep_bytes = IMG_W * IMG_H * 2
    if world_size > 1:
        # the exchanges live behind the C ABI (lcd_shard_process_frames_dev): the library's own NCCL communicator, bootstrapped like any
        # NCCL program — rank 0 creates the unique id, the host (here: torch.distributed) hands it to the other ranks
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(Engine.shard_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        eng.shard_comm_init(bytes(uid.cpu().numpy().tobytes()), rank, world_size)
        d_rowids = torch.from_numpy(ids).cuda()
        d_words = torch.zeros(nf * F_FEATS, dtype=torch.int32, device="cuda")   # this rank's frames only
        d_like = torch.zeros(nf * S_SIGS, dtype=torch.float32, device="cuda")
        h_words = torch.zeros((nf, F_FEATS), dtype=torch.int32).pin_memory()
        h_like = torch.zeros((nf, S_SIGS), dtype=torch.float32).pin_memory()

    def sharded_step(img_t, dep_t):
        # detect: frames sharded; quantise: words sharded; score: words sharded; verify: frames sharded — one library call per step
        eng.shard_process_frames_dev(img_t.data_ptr(), nf, IMG_W, IMG_H, 3, dep_t.data_ptr(), 1, op, d_sig.data_ptr(), S_SIGS, S_SIGS + 1,
                                     d_rowids.data_ptr(), W_WORDS, vp, d_words.data_ptr(), d_like.data_ptr(), True, NNDR, True)

    def step_dev(k):
        if world_size == 1:
            eng.process_frames_dev(d_img[k % n_pool].data_ptr(), B, IMG_W, IMG_H, 3, d_dep[k % n_pool].data_ptr(), 1, op, d_sig.data_ptr(), S_SIGS,
                                   S_SIGS + 1, vp, d_words.data_ptr(), d_like.data_ptr(), True, NNDR, True)
        else:
            sharded_step(d_img[k % n_pool], d_dep[k % n_pool])

    def step_host(k):
        hi, hd = h_img[k % n_pool], h_dep[k % n_pool]
        if world_size == 1:
            nkp, _, _, hyp, res = eng.process_frames(hi.numpy(), hd.numpy().view(np.uint16), op, h_sig.numpy(), S_SIGS + 1, vp, True, NNDR, True,
                                                     out_words=h_words.numpy(), out_like=h_like.numpy())
            return hyp, res
        di, dd = d_img[0], d_dep[0]
        di.copy_(hi, non_blocking=True)  # every rank uploads the frames it detects
        dd.copy_(hd, non_blocking=True)
        sharded_step(di, dd)
        h_words.view(-1).copy_(d_words, non_blocking=True)
        h_like.view(-1).copy_(d_like, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return eng.process_fetch(nf)

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing (value) -------------------------------------------------
    for k in range(args.warmup):
        step_dev(k)
    barrier()
    eng.profile_enable(True)
    eng.profile_reset()
    launches0 = eng.launch_count
    sampler = ClockSampler(local) if rank == 0 else None
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    torch.cuda.cudart().cudaProfilerStart()  # lets `ncu --profile-from-start off` see exactly the timed region
    t_wall0 = time.perf_counter()
    host_enqueue_s = 0.0
    for k in range(args.steps):
        flush.fill_(k & 0xFF)  # L2 flush, outside the timed events
        ev[k][0].record(ext)
        th = time.perf_counter()
        step_dev(k)
        host_enqueue_s += time.perf_counter() - th
        ev[k][1].record(ext)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    torch.cuda.cudart().cudaProfilerStop()
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    launches = eng.launch_count - launches0
    prof = {name: eng.profile_read(i) for i, name in enumerate(["nn", "resolve", "score", "match", "pnp", "orb"])}
    eng.profile_enable(False)
    if world_size > 1:
        t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms = float(t.item())
    value = B * args.steps / (dev_ms * 1e-3)

    # sanity inside the bench: the verified hypothesis must be a view of the revisited place
    last_pool = (args.steps - 1) % n_pool
    true_places = places[last_pool * BL:(last_pool + 1) * BL]
    hyp_d, res_d = eng.process_fetch(nf)
    # captured now: the measurements after the timed loop reuse d_words / d_like
    outputs = step_outputs(d_words.view(nf, F_FEATS).cpu(), d_like.view(nf, S_SIGS).cpu(), hyp_d, res_d) if args.dump_outputs else None
    def hit_rate(hyp):
        known = true_places >= 0
        return float(np.mean((world.sig_place[np.maximum(hyp, 1) - 1] == true_places)[known] & (hyp[known] > 0))) if known.any() else None

    hit = hit_rate(hyp_d)
    verified = float(np.mean([r["ok"] for r in res_d]))
    iters_hist = np.bincount(np.minimum(np.array([r["iterations_run"] for r in res_d]) // 50, 6), minlength=7).tolist()

    # ---- end-to-end timing through the host-buffer C ABI ------------------------------------
    for k in range(min(args.warmup, 3)):
        step_host(k)
    barrier()
    e2e_s = 0.0
    if world_size == 1:
        # the call a relocalisation service makes: lcd_process_frames_submit / _wait, two batches in flight, so the PCIe upload
        # of batch k+1 runs under the kernels of batch k.  Every step's images + depth come from pinned host memory and every
        # step's word ids, likelihood rows, hypotheses and verification results are copied back; all of it inside the timed
        # region, and so is the L2 flush between steps (queued on the engine stream).
        from rtabmap_b200.capi import VerifyResult
        sets = []
        for _ in range(2):
            sets.append(dict(nkp=torch.zeros(B, dtype=torch.int32).pin_memory(), words=torch.zeros((B, F_FEATS), dtype=torch.int32).pin_memory(),
                             like=torch.zeros((B, S_SIGS), dtype=torch.float32).pin_memory(), hyp=torch.zeros(B, dtype=torch.int32).pin_memory(),
                             res=(VerifyResult * B)()))
        sig_np = h_sig.numpy()

        def submit(k):
            o = sets[k & 1]
            eng.process_frames_submit(h_img[k % n_pool].numpy(), h_dep[k % n_pool].numpy().view(np.uint16), op, sig_np, S_SIGS + 1, vp,
                                      o["nkp"].numpy(), o["words"].numpy(), o["like"].numpy(), o["hyp"].numpy(), o["res"], True, NNDR, True)

        def collect(k):
            eng.process_frames_wait()
            o = sets[k & 1]
            return o["hyp"].numpy().copy(), [{"ok": int(r.ok)} for r in o["res"]]

        for k in range(2):  # warm-up of the pipelined path (allocates the two staging slots)
            submit(k)
        collect(0)
        collect(1)
        torch.cuda.synchronize()
        with torch.cuda.stream(ext):
            t0 = time.perf_counter()
            trace = [] if os.environ.get("LCD_BENCH_TRACE") else None
            submit(0)
            for k in range(1, args.steps):
                flush.fill_(k & 0xFF)
                ta = time.perf_counter()
                submit(k)
                tb = time.perf_counter()
                hyp_h, res_h = collect(k - 1)
                if trace is not None:
                    trace.append((round((ta - t0) * 1e3, 2), round((tb - ta) * 1e3, 2), round((time.perf_counter() - tb) * 1e3, 2)))
            hyp_h, res_h = collect(args.steps - 1)
            e2e_s = time.perf_counter() - t0
            if trace:
                print("e2e trace (t_submit_ms, submit_call_ms, collect_call_ms):", trace[:10], file=sys.stderr)
    else:
        up = torch.cuda.Stream()
        up_ev = [torch.cuda.Event(), torch.cuda.Event()]
        if os.environ.get("LCD_BENCH_PIPELINED_E2E", "0") != "1":
            # sharded job: the public calls are the *_dev entry points, so the caller owns the copies.  Double-buffered: the upload of
            # step k+1 (this rank's frames, pinned host memory) runs on a side stream under the kernels and collectives of step k;
            # every step's word ids, likelihood rows, hypotheses and verification results are copied back inside the timed region
            # (lcd_process_fetch: one device-wide synchronisation per step).  This is the loop every committed N>1 line was measured with.
            def prefetch(k):
                with torch.cuda.stream(up):
                    d_img[k & 1].copy_(h_img[k % n_pool], non_blocking=True)
                    d_dep[k & 1].copy_(h_dep[k % n_pool], non_blocking=True)
                    up_ev[k & 1].record(up)

            barrier()
            t0 = time.perf_counter()
            prefetch(0)
            for k in range(args.steps):
                flush.fill_(k & 0xFF)
                ext.wait_event(up_ev[k & 1])
                sharded_step(d_img[k & 1], d_dep[k & 1])
                h_words.view(-1).copy_(d_words, non_blocking=True)
                h_like.view(-1).copy_(d_like, non_blocking=True)
                if k + 1 < args.steps:
                    prefetch(k + 1)
                hyp_h, res_h = eng.process_fetch(nf)  # device-wide synchronisation + results of this rank's frames
            e2e_s = time.perf_counter() - t0
            e2e_api = "lcd_shard_process_frames_dev (exchanges inside the library), double-buffered pinned uploads on a side stream, results copied back every step"
        else:
            # sharded job: the public calls are the *_dev entry points, so the caller owns the copies.  Two steps in flight: the upload of
            # step k+1 (this rank's frames, pinned host memory) runs on a side stream under the kernels and collectives of step k, and
            # every step's word ids, likelihood rows, hypotheses and verification results are queued behind it (lcd_process_fetch_async)
            # into one of two pinned result sets; the host reads the set of step k-1 while step k runs.
            from rtabmap_b200.capi import VerifyResult
            done_ev = [torch.cuda.Event(), torch.cuda.Event()]
            res_bytes = ctypes.sizeof(VerifyResult) * nf
            sets = [dict(words=torch.zeros((nf, F_FEATS), dtype=torch.int32).pin_memory(), like=torch.zeros((nf, S_SIGS), dtype=torch.float32).pin_memory(),
                         hyp=torch.zeros(nf, dtype=torch.int32).pin_memory(), res=torch.zeros(res_bytes, dtype=torch.uint8).pin_memory()) for _ in range(2)]

            def prefetch(k):
                with torch.cuda.stream(up):
                    if k >= 2:
                        up.wait_event(done_ev[k & 1])  # step k-2 read this device buffer
                    d_img[k & 1].copy_(h_img[k % n_pool], non_blocking=True)
                    d_dep[k & 1].copy_(h_dep[k % n_pool], non_blocking=True)
                    up_ev[k & 1].record(up)

            def consume(k):
                done_ev[k & 1].synchronize()
                o = sets[k & 1]
                return o["hyp"].numpy().copy(), Engine.results_from_buffer(o["res"].numpy(), nf)

            barrier()
            t0 = time.perf_counter()
            prefetch(0)
            for k in range(args.steps):
                flush.fill_(k & 0xFF)
                ext.wait_event(up_ev[k & 1])
                sharded_step(d_img[k & 1], d_dep[k & 1])
                o = sets[k & 1]
                o["words"].view(-1).copy_(d_words, non_blocking=True)
                o["like"].view(-1).copy_(d_like, non_blocking=True)
                eng.process_fetch_async(nf, o["hyp"].data_ptr(), o["res"].data_ptr(), eng.stream)
                done_ev[k & 1].record(ext)
                if k + 1 < args.steps:
                    prefetch(k + 1)
                if k > 0:
                    hyp_h, res_h = consume(k - 1)
            hyp_h, res_h = consume(args.steps - 1)
            e2e_s = time.perf_counter() - t0
            h_words, h_like = sets[(args.steps - 1) & 1]["words"], sets[(args.steps - 1) & 1]["like"]  # what the oracle check below reads
            e2e_api = "lcd_shard_process_frames_dev (exchanges inside the library) + lcd_process_fetch_async: two steps in flight, pinned uploads on a side stream, every step's word ids / likelihood / hypotheses / results copied back"
    barrier()
    clocks = sampler.stop() if sampler else None
    if world_size > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = B * args.steps / e2e_s
    e2e_hit = hit_rate(np.asarray(hyp_h))
    e2e_verified = float(np.mean([r["ok"] for r in res_h]))
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs, f"rank{rank}_" if world_size > 1 else "")

    if rank != 0:
        if world_size > 1:
            dist.destroy_process_group()
        return 0

    hbm_peak, peak_src, sm_max = peaks()
    rows_local = r1 - r0
    alg_bytes = rows_local * DESC_BYTES + nq * DESC_BYTES + nq * 16  # SURVEY §8(d): W*D + Q*D + Q*16 per launch
    nn_ms, nn_launches = prof["nn"]
    nn_avg_s = (nn_ms / max(nn_launches, 1)) * 1e-3
    achieved = alg_bytes / nn_avg_s / 1e9 if nn_avg_s > 0 else 0.0
    pairs = float(rows_local) * nq
    popc_per_pair = 5  # LCD_NN_VARIANT=2: partial carry-save tree, 8 XOR words -> 5 POPC
    sm_clk = (clocks or {}).get("sm_mhz") or sm_max
    popc_peak = 16.0 * 148 * sm_clk * 1e6  # 16 POPC lanes / clk / SM, measured (profiles/r01_nn_sweep.json)
    traffic = None
    tp = ROOT / "profiles" / "roofline_traffic.json"
    if tp.exists():
        try:
            traffic = json.loads(tp.read_text()).get("knn2_hamming_kernel_dram_bytes_per_launch")
        except Exception:
            traffic = None
    share = dict({k + "_ms": v[0] / args.steps for k, v in prof.items()}, step_ms=dev_ms / args.steps)
    if os.environ.get("LCD_NN_TENSOR", "1") != "0":
        # dominant kernel: knn2_tensor_kernel (tcgen05 kind::i8).  Algorithmic work per launch = one s8 multiply-add per
        # (query, word, descriptor bit): 2 * Q * W * 256 operations (DESIGN.md §4).
        ops = 2.0 * pairs * DESC_BYTES * 8
        tpeak, tsrc = tensor_peak_tops()
        ach = ops / nn_avg_s / 1e12 if nn_avg_s > 0 else 0.0
        traffic_t = None
        if tp.exists():
            try:
                traffic_t = json.loads(tp.read_text()).get("knn2_tensor_kernel_dram_bytes_per_launch")
            except Exception:
                traffic_t = None
        roofline = {
            "kernel": "knn2_tensor_kernel (tcgen05.mma kind::i8, M128 N256 K32)", "bound": "tensor", "achieved": ach, "peak": tpeak,
            "unit": "TFLOP/s", "frac": ach / tpeak, "peak_source": tsrc, "traffic": traffic_t,
            "algorithmic_ops_per_launch": ops, "algorithmic_bytes_per_launch": alg_bytes,
            "avg_launch_ms": nn_avg_s * 1e3, "launches_timed": int(nn_launches),
            "note": "s8 operations counted as FLOPs of the +-1 encoded Hamming GEMM; results are exact integers (parity tests)",
            "pairs_per_s": pairs / nn_avg_s if nn_avg_s > 0 else 0.0, "step_share_ms": share,
        }
    else:
        roofline = {
            "kernel": "knn2_hamming_kernel<8,8,2>", "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
            "peak_source": peak_src, "traffic": traffic, "algorithmic_bytes_per_launch": alg_bytes,
            "avg_launch_ms": nn_avg_s * 1e3, "launches_timed": int(nn_launches),
            "binding_resource": "integer pipes (POPC 16 lanes/clk/SM on XU + LOP3 on ALU): the vocabulary is SMEM/L2 resident, see DESIGN.md §4",
            "pairs_per_s": pairs / nn_avg_s if nn_avg_s > 0 else 0.0,
            "popc_per_s": pairs * popc_per_pair / nn_avg_s if nn_avg_s > 0 else 0.0, "popc_peak_per_s": popc_peak,
            "popc_frac": (pairs * popc_per_pair / nn_avg_s) / popc_peak if nn_avg_s > 0 else 0.0,
            "step_share_ms": share,
        }

    # the XOR/POPC kernel on the same resident data (three untimed-region steps), for comparison with the tensor kernel
    if world_size == 1 and os.environ.get("LCD_NN_TENSOR", "1") != "0":
        eng.nn_select(0)
        eng.profile_enable(True)
        eng.profile_reset()
        for k in range(3):
            step_dev(k)
        torch.cuda.synchronize()
        p_ms, p_n = eng.profile_read(0)
        eng.profile_enable(False)
        eng.nn_select(1)
        p_s = (p_ms / max(p_n, 1)) * 1e-3
        roofline["popcount_kernel"] = {
            "kernel": "knn2_hamming_kernel<8,8,2> (lcd_nn_select(e, 0))", "avg_launch_ms": p_s * 1e3, "launches_timed": int(p_n),
            "bound": "integer pipes (POPC 16 lanes/clk/SM)", "popc_per_s": pairs * popc_per_pair / p_s if p_s > 0 else 0.0,
            "popc_peak_per_s": popc_peak, "popc_frac": (pairs * popc_per_pair / p_s) / popc_peak if p_s > 0 else 0.0,
            "hbm_GBps": alg_bytes / p_s / 1e9 if p_s > 0 else 0.0, "hbm_frac": (alg_bytes / p_s / 1e9) / hbm_peak if p_s > 0 else 0.0,
            "traffic": traffic,
        }

    # ---- CPU baseline (rank 0 at N=1) and the oracle cross-check of this very run (every N) -------------------------------
    cpu = None
    ref = None
    if not args.no_cpu_baseline:
        ref = CpuReference(world)
    if world_size == 1 and ref is not None:
        threads = max(1, min(os.cpu_count() or 1, 32))
        rate, dt, res = ref.rate(imgs_all, deps_all, threads, threads)
        cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "reference" if ref.rtflann else "port", "legs": ref.legs(),
               "sample": f"{threads} frames of the same workload ({dt:.1f} s wall), {threads} threads, one frame per thread"}
        # cross-check while we are here: the first frames against the GPU result (the parity tests proper are tests/)
        nchk = min(4, threads)
        nkp, w_g, l_g, hyp_c, res_c = eng.process_frames(imgs_all[:nchk], deps_all[:nchk], op, smap.sig_ids, S_SIGS + 1, vp, True, NNDR, True)
        for b in range(nchk):
            kp, d, words, like, hyp_o, v, x = res[b]
            assert nkp[b] == len(kp) and np.array_equal(w_g[b][:len(words)], words), "GPU/oracle word ids differ"
            assert np.allclose(l_g[b], like, atol=1e-4, rtol=1e-4), "GPU/oracle likelihood differ"
            assert hyp_o == hyp_c[b] and v["ok"] == res_c[b]["ok"] and len(v["inliers"]) == res_c[b]["n_inliers"], "GPU/oracle verification differ"
            if v["ok"]:
                assert np.allclose(v["rvec"], res_c[b]["rvec"], atol=1e-4) and np.allclose(v["tvec"], res_c[b]["tvec"], atol=1e-4)
                assert np.allclose(v["covariance"], res_c[b]["covariance"], rtol=1e-4, atol=1e-9)
    sharded_check = None
    if world_size > 1 and ref is not None:
        # the NCCL path against the oracle: rank 0's first frames of the LAST end-to-end step (full, unsharded dictionary on the CPU)
        kpool = (args.steps - 1) % n_pool
        nchk = 2
        try:
            for b in range(nchk):
                kp, d, words, like, hyp_o, v, x = ref.one(h_img[kpool][b].numpy(), h_dep[kpool][b].numpy().view(np.uint16))
                wg = h_words[b].numpy()
                assert np.array_equal(wg[:len(words)], words), "sharded run: GPU/oracle word ids differ"
                assert np.allclose(h_like[b].numpy(), like, atol=1e-4, rtol=1e-4), "sharded run: GPU/oracle likelihood differ"
                assert hyp_o == int(hyp_h[b]) and bool(v["ok"]) == bool(res_h[b]["ok"]), "sharded run: GPU/oracle verification differ"
                if v["ok"]:
                    assert len(v["inliers"]) == res_h[b]["n_inliers"], "sharded run: GPU/oracle inlier counts differ"
                    assert np.allclose(v["rvec"], res_h[b]["rvec"], atol=1e-4) and np.allclose(v["tvec"], res_h[b]["tvec"], atol=1e-4), "sharded run: poses differ"
            sharded_check = f"rank 0: {nchk} frames of the last step equal the CPU oracle (word ids exact, likelihood 1e-4, hypothesis, inlier count, pose 1e-4)"
        except AssertionError as ex:
            # reported in the line and through the exit code, AFTER the process group is torn down: raising here would leave the other
            # ranks waiting in a collective until the launcher's timeout
            sharded_check = f"FAILED: {ex}"
            log(f"[rank 0] {sharded_check}")

    extra = {}
    if world_size == 1 and not args.no_extras:
        extra = run_extras(eng, world, op, vp, d_sig, imgs_all, deps_all, args)

    # dominant STAGE next to the dominant kernel: ORB detect + describe, SURVEY 8(d) algorithmic bytes 2.9 MB per 640x480 frame
    orb_ms, orb_n = prof["orb"]
    orb_s = (orb_ms / max(orb_n, 1)) * 1e-3
    orb_bytes = (IMG_W * IMG_H * 3 + (IMG_W * IMG_H + IMG_W * IMG_H // 4 + IMG_W * IMG_H // 16) * 5) * BL
    roofline["stage_orb"] = {"stage": "detect (all orb_* kernels of one step)", "bound": "hbm (nominal; measured: instruction issue, DESIGN.md 4.3)",
                             "algorithmic_bytes_per_step": orb_bytes, "avg_ms": orb_s * 1e3, "achieved": orb_bytes / orb_s / 1e9 if orb_s > 0 else 0.0,
                             "peak": hbm_peak, "unit": "GB/s", "frac": (orb_bytes / orb_s / 1e9) / hbm_peak if orb_s > 0 else 0.0}
    roofline["traffic_source"] = "profiles/roofline_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this command, per launch"
    roofline["timing_note"] = "per-kernel times come from CUDA events recorded around every launch inside the timed region (lcd_profile_enable(1)): the step time includes those events"

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "config": job_config(args, world_size),
        "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(B * (img_bytes + dep_bytes) + S_SIGS * 4),
                "d2h_bytes_per_step": int(nq * 4 + B * S_SIGS * 4 + B * (4 + 4 + 124 + 288)),
                "api": "lcd_process_frames_submit/_wait (pinned host buffers, 2 batches in flight, L2 flush between steps inside the timed region)" if world_size == 1 else e2e_api,
                "top1_place_hit_rate": e2e_hit, "verified_rate": e2e_verified},
        "roofline": roofline, "cpu_baseline": cpu, "top1_place_hit_rate": hit, "verified_rate": verified, "ransac_iterations_hist_50": iters_hist,
        "wall_s_timed_region": t_wall, "host_enqueue_ms_per_step": host_enqueue_s * 1e3 / args.steps,
        "frames_pool": f"{n_pool} batches of {BL} frames cycled", "oracle_check": sharded_check, **extra,
    }
    print(json.dumps(line), flush=True)
    if world_size > 1:
        dist.destroy_process_group()
        try:
            with open(os.environ.get("NCCL_DEBUG_FILE", "")) as f:
                keep = [ln.rstrip() for ln in f if "Init COMPLETE" in ln or "nranks" in ln or "NCCL version" in ln or "Using network" in ln or "NVLS" in ln]
            for ln in keep[:24]:
                log("[nccl] " + ln)
        except OSError:
            pass
    return 1 if (sharded_check or "").startswith("FAILED") else 0


def run_extras(eng, world, op, vp, d_sig, imgs_all, deps_all, args):
    """Measurements beside the headline (single GPU): single-frame latency through the host C-ABI call, and the mixed workload when the
    headline ran on revisits.  Reported under their own keys; never mixed into `value`."""
    import torch

    from rtabmap_b200 import synth

    out = {}
    sm = world.smap
    # batch-1 latency: one frame in, one answer out, host buffers, nothing else in flight
    lat = []
    for k in range(13):
        t0 = time.perf_counter()
        eng.process_frames(imgs_all[k:k + 1], deps_all[k:k + 1], op, sm.sig_ids, S_SIGS + 1, vp, True, NNDR, True)
        lat.append((time.perf_counter() - t0) * 1e3)
    lat = np.sort(np.array(lat[3:]))
    out["latency_batch1_ms"] = {"median": float(np.median(lat)), "min": float(lat[0]), "max": float(lat[-1]), "samples": len(lat),
                                "api": "lcd_process_frames, 1 frame, pageable host buffers in, results out, wall clock"}
    if args.workload == "revisit":
        # the harder workload (SURVEY 8(d)): never-seen places run all 300 RANSAC iterations and are rejected; rotated / scaled views
        B = args.batch
        imgs, deps, places = synth.make_view_frames(world, B, seed=77, mode="mixed")
        d_i = torch.from_numpy(imgs).cuda()
        d_d = torch.from_numpy(deps.view(np.int16)).cuda()
        d_w = torch.zeros(B * F_FEATS, dtype=torch.int32, device="cuda")
        d_l = torch.zeros(B * S_SIGS, dtype=torch.float32, device="cuda")
        ext = torch.cuda.ExternalStream(eng.stream)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_it = 5
        for k in range(2 + n_it):
            if k == 2:
                torch.cuda.synchronize()
                ev0.record(ext)
            eng.process_frames_dev(d_i.data_ptr(), B, IMG_W, IMG_H, 3, d_d.data_ptr(), 1, op, d_sig.data_ptr(), S_SIGS, S_SIGS + 1, vp, d_w.data_ptr(),
                                   d_l.data_ptr(), True, NNDR, True)
        ev1.record(ext)
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / n_it
        hyp, res = eng.process_fetch(B)
        known = places >= 0
        out["mixed_workload"] = {"value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "frames_per_step": B,
                                 "never_seen_frames": int((~known).sum()), "verified_rate": float(np.mean([r["ok"] for r in res])),
                                 "verified_rate_known_places": float(np.mean([r["ok"] for r, kn in zip(res, known) if kn])),
                                 "false_accepts_on_never_seen": int(sum(r["ok"] for r, kn in zip(res, known) if not kn)),
                                 "ransac_iterations_hist_50": np.bincount(np.minimum(np.array([r["iterations_run"] for r in res]) // 50, 6), minlength=7).tolist(),
                                 "note": "device-resident inputs, CUDA events, same engine and map as the headline"}
    # mapping mode (the reference's default: incremental dictionary + growing map, frame t+1 depends on frame t): a sequential stream
    # through lcd_map_detect_async / lcd_map_frame on top of the same 49k-word / 10k-signature state.  Runs last: it mutates the engine.
    n_map = 48
    imgs, deps, places = synth.make_view_frames(world, n_map + 4, seed=91, mode="mixed")
    wm = np.ascontiguousarray(sm.sig_ids)
    n_sigs = int(sm.sig_ids.max())
    eng.map_detect_async(imgs[0], deps[0], op)
    t_frames, t_detect = [], []
    new_words = 0
    for t in range(n_map + 4):
        if t == 4:
            t0 = time.perf_counter()
        tb = time.perf_counter()
        if t + 1 < n_map + 4:
            eng.map_detect_async(imgs[t + 1], deps[t + 1], op)
        ta = time.perf_counter()
        n_kp, words, n_new, like = eng.map_frame(n_sigs + 1 + t, wm, n_sigs + 1 + t, True, NNDR, True)
        if t >= 4:
            t_frames.append((time.perf_counter() - ta) * 1e3)
            t_detect.append((ta - tb) * 1e3)
            new_words += n_new
    dt = time.perf_counter() - t0
    out["mapping_mode"] = {"value": n_map / dt, "unit": "frames/s", "frames": n_map, "ms_per_frame_median": float(np.median(t_frames)),
                           "ms_map_frame_max": float(np.max(t_frames)), "ms_detect_submit_median": float(np.median(t_detect)),
                           "ms_detect_submit_max": float(np.max(t_detect)),
                           "ms_per_frame_p90": float(np.percentile(t_frames, 90)),
                           "slowest_frames_ms": [[int(i), round(float(t_frames[i]), 2)] for i in np.argsort(t_frames)[::-1][:6]],
                           "new_words_per_frame": new_words / n_map, "dictionary_words_after": eng.size(),
                           "api": "lcd_map_detect_async (frame t+1) overlapped with lcd_map_frame (update + quantise with mutation + references + TF-IDF over "
                                  "10k signatures) of frame t; host images in, word ids + likelihood out, wall clock",
                           "note": "sequential by definition (SURVEY F7): one frame in flight through the dictionary; the batched headline is localisation mode"}
    return out


# ------------------------------------------------------------------------- BASELINE configs[3]: float descriptors, 1M words
C4_DIM = 64
C4_FEATS = 1000


def c4_sizes(args):
    return (args.words or 1_000_000), (args.signatures or 100_000)


def c4_config(args, W, S, batch):
    return {
        "workload": "BASELINE configs[3]: SURF-64-like float descriptors (unit norm, Laplacian components), 1M-word dictionary, 100k signatures",
        "words": W, "signatures": S, "features_per_frame": C4_FEATS, "descriptor": "64 x f32 (256 B)", "frames_per_step": batch,
        "mode": "localisation (frozen dictionary + map)",
        "stages": ["quantise (exact squared-L2 2-NN in rtflann's order + NNDR + intra-frame new words)", "score (TF-IDF over the inverted index)"],
        "not_in_this_config": "detect (cv::xfeatures2d::SURF is absent from this image: no extractor, no oracle; descriptors are given) and verify "
                              "(binary descriptors only)",
        "queries": "rows of the vocabulary + N(0, 0.02) noise, 20 % unrelated descriptors (NNDR rejects -> new words)",
        "l2": "the fp16 word image (128 MB) and the fp32 rows (256 MB) both exceed L2; no flush needed",
    }


def c4_world(args):
    from rtabmap_b200 import synth

    W, S = c4_sizes(args)
    t0 = time.time()
    vocab = synth.make_float_vocabulary(W, C4_DIM, 1)
    ids = np.arange(1, W + 1, dtype=np.int32)
    smap = synth.make_map(ids, S, C4_FEATS, seed=2)
    log(f"c4 world: {W} words, {S} signatures, {smap.nnz} postings in {time.time() - t0:.0f} s")
    return vocab, ids, smap


def c4_queries(vocab, smap, n_frames, seed):
    """Frames revisiting random signatures: their words' descriptors + noise, a fifth replaced by unrelated descriptors."""
    from rtabmap_b200 import synth

    rng = np.random.default_rng(seed)
    q = np.empty((n_frames, C4_FEATS, C4_DIM), np.float32)
    places = rng.integers(0, len(smap.sig_ids), n_frames)
    for f in range(n_frames):
        rows = smap.sig_words[places[f]].astype(np.int64) - 1
        d = vocab[rows] + rng.normal(0, 0.02, (C4_FEATS, C4_DIM)).astype(np.float32)
        idx = rng.permutation(C4_FEATS)[:C4_FEATS // 5]
        d[idx] = synth.make_float_vocabulary(len(idx), C4_DIM, 1000 + seed * 100 + f)
        q[f] = d
    return q, places


def run_reference_c4(args):
    """CPU arm of configs[3]: the index search by the reference's compiled rtflann (single thread per frame, as FlannIndex runs it), NNDR +
    TF-IDF by the oracle port; frames spread over the host threads.  One step = `per_step` frames, each a SAMPLE of 100 of its 1000
    descriptors (a full frame is ~40 s of rtflann scan); the rate is scaled to whole frames."""
    from oracle import oracle_py as orc

    W, S = c4_sizes(args)
    vocab, ids, smap = c4_world(args)
    threads = max(1, min(os.cpu_count() or 1, args.ref_threads or (os.cpu_count() or 1)))
    per_step = min(threads, 16)
    sample = 100
    q, places = c4_queries(vocab, smap, per_step, 3)
    use_ref = orc.ref_lib() is not None

    def one(b):
        d = q[b, :sample]
        if use_ref:
            return orc.ref_knn2(vocab, d)
        return orc.knn2_raw(vocab, d)

    def step():
        t0 = time.perf_counter()
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(one, range(per_step)))
        return time.perf_counter() - t0

    for _ in range(min(args.warmup, 1)):
        step()
    steps = args.steps
    total = sum(step() for _ in range(steps))
    value = per_step * steps * (sample / C4_FEATS) / total
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1),
            "ms_per_step": 1e3 * total / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": c4_config(args, W, S, args.batch),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "reference" if use_ref else "port",
                             "sample": f"{per_step} frames/step x {steps} steps, {sample} of the {C4_FEATS} descriptors of each frame through "
                                       f"{'the reference rtflann LinearIndex (oracle/_ref)' if use_ref else 'the oracle scan'} over all {W} rows, scaled to "
                                       "whole frames; the NNDR / TF-IDF legs (milliseconds) are not in the sample"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)
    return 0


def run_c4(args):
    """configs[3] on one B200: quantise + score of `batch` frames of 1000 float descriptors against 1M words / 100k signatures."""
    import torch

    from oracle import oracle_py as orc
    from rtabmap_b200 import Engine

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --config c4 needs a CUDA device; there is no CPU fallback")
    if int(os.environ.get("WORLD_SIZE", "1")) != 1:
        raise SystemExit("--config c4 is a single-GPU configuration (BASELINE configs[3])")
    torch.cuda.set_device(0)
    W, S = c4_sizes(args)
    B = args.batch if args.batch != 128 else 32
    vocab, ids, smap = c4_world(args)
    eng = Engine(device=0, desc_type=1, desc_dim=C4_DIM, max_words=W + 4096, max_signatures=S + 2, max_queries=C4_FEATS, max_batch=B)
    t0 = time.time()
    for r0 in range(0, W, 1 << 18):
        eng.add_words(ids[r0:r0 + (1 << 18)], vocab[r0:r0 + (1 << 18)])
    eng.last_word_id = W
    eng.update()
    eng.load_csr(smap.word_ids, smap.row_ptr, smap.sig, smap.cnt)
    eng.set_ni(smap.sig_ids, smap.ni)
    log(f"engine loaded in {time.time() - t0:.0f} s")
    n_pool = 3
    q_all, places = c4_queries(vocab, smap, B * n_pool, 3)
    ext = torch.cuda.ExternalStream(eng.stream)
    torch.cuda.set_stream(ext)
    d_q = [torch.from_numpy(q_all[k * B:(k + 1) * B].reshape(-1, C4_DIM)).cuda() for k in range(n_pool)]
    h_q = [torch.from_numpy(q_all[k * B:(k + 1) * B].reshape(-1, C4_DIM)).pin_memory() for k in range(n_pool)]
    d_sig = torch.from_numpy(smap.sig_ids).cuda()
    nq = B * C4_FEATS
    d_words = torch.zeros(nq, dtype=torch.int32, device="cuda")
    d_like = torch.zeros(B * S, dtype=torch.float32, device="cuda")
    h_words = torch.zeros((B, C4_FEATS), dtype=torch.int32).pin_memory()
    h_like = torch.zeros((B, S), dtype=torch.float32).pin_memory()

    def step_dev(k):
        eng.localize_batch_dev(d_q[k % n_pool].data_ptr(), B, C4_FEATS, d_sig.data_ptr(), S, S + 1, d_words.data_ptr(), d_like.data_ptr(), True, NNDR, True)

    for k in range(args.warmup):
        step_dev(k)
    torch.cuda.synchronize()
    assert eng.nn_last_kernel == 1, "the tensor-core float kernel did not run"
    eng.profile_enable(True)
    eng.profile_reset()
    launches0 = eng.launch_count
    sampler = ClockSampler(0)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    torch.cuda.synchronize()
    torch.cuda.cudart().cudaProfilerStart()
    t_wall0 = time.perf_counter()
    for k in range(args.steps):
        ev[k][0].record(ext)
        step_dev(k)
        ev[k][1].record(ext)
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    torch.cuda.cudart().cudaProfilerStop()
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    launches = eng.launch_count - launches0
    prof = {name: eng.profile_read(i) for i, name in enumerate(["nn", "resolve", "score"])}
    eng.profile_enable(False)
    value = B * args.steps / (dev_ms * 1e-3)
    n_fallback, n_cand, rows_conv = eng.nn_f32_stats(nq)
    outputs = step_outputs(d_words.view(B, C4_FEATS).cpu(), d_like.view(B, S).cpu()) if args.dump_outputs else None
    like_last = d_like.view(B, S).argmax(1).cpu().numpy()
    last_pool = (args.steps - 1) % n_pool
    hit = float(np.mean(smap.sig_ids[like_last] == smap.sig_ids[places[last_pool * B:(last_pool + 1) * B]]))

    # end to end: pinned host descriptors in, word ids + likelihood rows out, every step
    def step_host(k):
        eng.localize_batch(h_q[k % n_pool].numpy(), B, smap.sig_ids, S + 1, True, NNDR, True, out_words=h_words.numpy(), out_like=h_like.numpy())

    for k in range(2):
        step_host(k)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(args.steps):
        step_host(k)
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop()
    e2e_value = B * args.steps / e2e_s
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)

    hbm_peak, peak_src, _ = peaks()
    nn_ms, nn_n = prof["nn"]
    nn_s = (nn_ms / max(nn_n, 1)) * 1e-3
    flops = 2.0 * nq * W * C4_DIM
    alg_bytes = W * C4_DIM * 4 + nq * C4_DIM * 4 + nq * 16  # SURVEY 8(d): W*D + Q*D + Q*16
    tp = ROOT / "MEASURED_PEAKS.json"
    f16_peak = float(json.loads(tp.read_text()).get("bf16_tflops", 2250.0)) if tp.exists() else 2250.0
    traffic = None
    rt = ROOT / "profiles" / "roofline_traffic.json"
    if rt.exists():
        traffic = json.loads(rt.read_text()).get("knn2_tensor_f32_kernel_dram_bytes_per_launch")
    roofline = {
        "kernel": "float dictionary NN = knn2_tensor_f32_kernel (tcgen05.mma kind::f16, M128 N256 K16, pre-pass + main pass) + rerank_l2_kernel + "
                  "knn2_l2_fallback_kernel, timed together",
        "bound": "tensor", "achieved": flops / nn_s / 1e12 if nn_s > 0 else 0.0, "peak": f16_peak, "unit": "TFLOP/s",
        "frac": (flops / nn_s / 1e12) / f16_peak if nn_s > 0 else 0.0,
        "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst; fp16 and bf16 run at the same tcgen05 rate)" if tp.exists() else "nominal 2250 (B200_PROFILING.md)",
        "traffic": traffic, "algorithmic_flops_per_step": flops, "algorithmic_bytes_per_step": alg_bytes, "avg_ms": nn_s * 1e3, "steps_timed": int(nn_n),
        "hbm": {"achieved": alg_bytes / nn_s / 1e9 if nn_s > 0 else 0.0, "peak": hbm_peak, "unit": "GB/s", "frac": (alg_bytes / nn_s / 1e9) / hbm_peak if nn_s > 0 else 0.0,
                "peak_source": peak_src, "note": "algorithmic bytes of ONE step (vocabulary read once per batch of frames); the kernel is epilogue / tensor bound, "
                                                 "not HBM bound: the fp16 word image streams once per step (DESIGN.md 4.4)"},
        "step_share_ms": {k + "_ms": v[0] / args.steps for k, v in prof.items()},
        "filter": {"candidates_per_query": n_cand / nq, "queries_redone_by_exact_scan": n_fallback, "queries": nq,
                   "dictionary_rows_converted_to_fp16_since_start": rows_conv},
    }

    cpu = None
    if not args.no_cpu_baseline:
        # reference rtflann on a sample of one frame + full-frame oracle check of the GPU result
        sample = 100
        d = np.ascontiguousarray(q_all[0, :sample])
        t0 = time.perf_counter()
        ki, kd = orc.ref_knn2(vocab, d) if orc.ref_lib() is not None else orc.knn2_raw(vocab, d)
        dt = time.perf_counter() - t0
        cpu = {"value": (sample / C4_FEATS) / dt, "unit": UNIT, "cores": 1, "kind": "reference" if orc.ref_lib() is not None else "port",
               "sample": f"{sample} of the {C4_FEATS} descriptors of one frame through the reference's compiled rtflann LinearIndex over all {W} rows "
                         f"({dt:.1f} s, single thread as FlannIndex runs it), scaled to whole frames"}
        i1, d1, i2, d2 = eng.knn2(d)
        assert np.array_equal(i1, ids[ki[:, 0]]) and np.array_equal(i2, ids[ki[:, 1]]), "GPU / rtflann neighbours differ"
        assert np.array_equal(d1, kd[:, 0].astype(np.float32)) and np.array_equal(d2, kd[:, 1].astype(np.float32)), "GPU / rtflann distances differ"

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (fp16 tensor-core filter, exact fp32 re-rank)",
        "data": "synthetic", "config": c4_config(args, W, S, B), "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(nq * C4_DIM * 4 + S * 4), "d2h_bytes_per_step": int(nq * 4 + B * S * 4),
                "api": "lcd_localize_batch (pinned host descriptors in, word ids + likelihood rows out)"},
        "roofline": roofline, "cpu_baseline": cpu, "top1_place_hit_rate": hit, "wall_s_timed_region": t_wall,
    }
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=128, help="frames per step")
    ap.add_argument("--ref-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the latency / mixed-workload measurements beside the headline")
    ap.add_argument("--workload", default="revisit", choices=["revisit", "mixed"], help="query frames of the headline (mixed: SURVEY 8(d) hard case)")
    ap.add_argument("--config", default="c2", choices=["c2", "c4"], help="c2 = BASELINE configs[1] (headline); c4 = configs[3]: float descriptors, 1M words")
    ap.add_argument("--words", type=int, default=0, help="c4: dictionary rows (default 1 000 000)")
    ap.add_argument("--signatures", type=int, default=0, help="c4: signatures in the map (default 100 000)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path returned for its last step as DIR/<name>.npy "
                                                           "(float32 / float64, at most 64 MB: beyond that a fixed sample of the frames)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.impl == "reference":
        return run_reference(args)
    if args.config == "c4":
        return run_c4(args)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        # a rank that dies with the process group and the library's communicator still alive can hang in their teardown (and the other
        # ranks in a collective) until the launcher's timeout: report the error and leave without running any destructor
        try:
            return run_b200(args)
        except BaseException:
            import traceback

            traceback.print_exc()
            sys.stderr.flush()
            sys.stdout.flush()
            os._exit(1)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
