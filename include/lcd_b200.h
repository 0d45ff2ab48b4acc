/*
 * lcd_b200.h — C ABI of the B200-native loop-closure hot path
 * (detect -> quantise -> score -> verify) that drops in behind
 * rtabmap::Memory / VWDictionary / Signature / Feature2D.
 *
 * RTAB-Map has no C ABI or plugin loader for this path (SURVEY.md §8(b)); its
 * seams are C++ virtuals owned by rtabmap::Memory.  Every entry point below
 * names the reference member function (file:line under corelib/) whose work it
 * replaces.  INTEGRATION.md shows the two shim classes (VWDictionaryB200,
 * ORB_B200) a maintainer adds on the reference side to bind these symbols.
 *
 * Conventions (mirroring the reference's, SURVEY.md §8(b)):
 *   - all functions return 0 on success, <0 on error (never throw); the message
 *     is available through lcd_last_error(engine)  [reference: UERROR + empty
 *     return, VWDictionary.cpp:920-957];
 *   - all buffers are caller-owned HOST pointers, row-major, unless the function
 *     name ends in _dev (device pointers valid on the engine's device);
 *   - word ids are positive ints, 0 = invalid / no match; signature ids are
 *     positive ints (VWDictionary.cpp:875-878, Memory.cpp:6040-6058);
 *   - one engine = one VWDictionary instance + its inverted index on one GPU;
 *     several engines may coexist (RegistrationVis builds temporary
 *     dictionaries, RegistrationVis.cpp:1482-1503);
 *   - calls on one engine must be serialised by the caller, with ONE exception:
 *     the host-buffer lcd_orb_detect_describe may run on a second thread while
 *     lcd_dict_update runs (the reference runs VWDictionary::update() on
 *     PreUpdateThread beside feature extraction, Memory.cpp:5284, :5926).  The two
 *     calls share no buffers, run on different CUDA streams, and the counters they
 *     both touch are atomic (tests/test_gpu_concurrency.py).  lcd_profile_enable(1)
 *     suspends that exception (its event lists are not thread-safe);
 *   - the *_dev entry points of one engine must all be given the same stream (or
 *     NULL): scratch buffers are shared between them.
 */
#ifndef LCD_B200_H
#define LCD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LCD_OK 0
#define LCD_ERR_INVALID (-1)  /* bad argument / size or type mismatch            */
#define LCD_ERR_CUDA (-2)     /* CUDA runtime failure (message has the detail)   */
#define LCD_ERR_CAPACITY (-3) /* a configured capacity would be exceeded         */
#define LCD_ERR_STATE (-4)    /* call not valid in the current state             */

/* descriptor types: cv::Mat type()/cols of VisualWord::getDescriptor()
 * (VWDictionary.cpp:933-957 checks) */
#define LCD_DESC_U8 0  /* CV_8U rows, desc_dim bytes (ORB/BRIEF: 32)  -> Hamming   */
#define LCD_DESC_F32 1 /* CV_32F rows, desc_dim floats (SURF: 64/128) -> squared L2 */

typedef struct lcd_engine lcd_engine;

typedef struct lcd_config {
	int device;         /* CUDA device ordinal                                          */
	int desc_type;      /* LCD_DESC_U8 | LCD_DESC_F32                                   */
	int desc_dim;       /* bytes (U8: 16/32/64) or floats (F32: 64/128)                 */
	int max_words;      /* initial capacity hint for vocabulary rows (grows)            */
	int max_signatures; /* initial capacity hint for signature ids (grows)              */
	int max_queries;    /* max descriptors per lcd_dict_* call / per frame (<= 4096)    */
	int max_batch;      /* max frames per lcd_localize_batch call                       */
} lcd_config;

/* ---- lifetime ---------------------------------------------------------------- */
/* replaces: VWDictionary::VWDictionary / ~VWDictionary (VWDictionary.cpp:56-120) */
lcd_engine * lcd_create(const lcd_config * cfg);
void lcd_destroy(lcd_engine * e);
/* last error text of this engine (e may be NULL: error of the last failed lcd_create) */
const char * lcd_last_error(const lcd_engine * e);
/* library/ABI version, and the name of the CUDA arch the kernels were built for */
int lcd_abi_version(void); /* 2: lcd_verify_params / lcd_verify_result grew (covariance), lcd_verify_batch takes xyz_to */
const char * lcd_build_arch(void);
/* number of kernels this engine has launched since creation (bench "gpu_launches") */
long long lcd_launch_count(const lcd_engine * e);

/* ---- detect: Feature2D (ORB) ---------------------------------------------------------------
 * cv::KeyPoint fields the reference uses (Signature keypoints, Features2d.cpp:1657). */
typedef struct lcd_keypoint {
	float x, y;      /* pt, level-0 pixel coordinates */
	float size;      /* patchSize * scale of the level */
	float angle;     /* degrees, intensity-centroid orientation */
	float response;  /* Harris response */
	int octave;      /* pyramid level */
} lcd_keypoint;

typedef struct lcd_orb_params {
	int n_features;       /* Kp/MaxFeatures: nfeatures of cv::ORB and the limit of Feature2D::limitKeypoints */
	int n_levels;         /* ORB/NLevels (1..4) */
	float scale_factor;   /* ORB/ScaleFactor: 2.0 (the reference default) is the only value implemented */
	int edge_threshold;   /* ORB/EdgeThreshold (19) */
	int fast_threshold;   /* FAST/Threshold (20) */
	int patch_size;       /* ORB/PatchSize: 31 (the learned rBRIEF pattern) */
	float min_depth;      /* Kp/MinDepth */
	float max_depth;      /* Kp/MaxDepth (0 = unlimited) */
	int depth_as_mask;    /* Mem/DepthAsMask */
	float fx, fy, cx, cy; /* CameraModel of the frame (depth registered to the image, same size) */
} lcd_orb_params;

#define LCD_DEPTH_NONE 0
#define LCD_DEPTH_U16_MM 1 /* CV_16UC1, millimetres */
#define LCD_DEPTH_F32_M 2  /* CV_32FC1, metres     */
#define LCD_DEPTH_MASK_U8 3 /* not a depth image: the CV_8UC1 mask (0 / 255) Feature2D::generateKeypoints hands to
                               generateKeypointsImpl (Features2d.cpp:783-857); no 3-D points are produced */

/* replaces, for Kp/DetectorStrategy=2: cv::cvtColor(BGR2GRAY) (Memory.cpp:5447),
 * Feature2D::generateKeypoints incl. the depth mask and limitKeypoints (Features2d.cpp:775-878, :356-399)
 * -> cv::ORB::detect, Feature2D::generateDescriptors -> cv::ORB::compute (Features2d.cpp:1663-1718) and
 * Feature2D::generateKeypoints3D -> util3d::generateKeypoints3DDepth (util3d_features.cpp:67-120), for
 * n_frames images [n_frames][height][width][channels] (channels 1 = gray, 3 = BGR) with optional depth
 * [n_frames][height][width].  Outputs hold `cap` rows per frame: kp_out[n_frames*cap],
 * desc_out[n_frames*cap*32], xyz_out[n_frames*cap*3] (NaN = no depth), n_out[n_frames] valid rows. */
int lcd_orb_detect_describe(lcd_engine * e, int n_frames, const uint8_t * images, int width, int height, int channels,
                            const void * depth, int depth_type, const lcd_orb_params * params, int cap,
                            lcd_keypoint * kp_out, uint8_t * desc_out, float * xyz_out, int * n_out);
/* same with device-resident inputs and outputs (any output may be NULL), asynchronous on `stream`;
 * d_uv_out[n_frames*cap*2] optionally receives the keypoint coordinates as a plain float2 array. */
int lcd_orb_detect_describe_dev(lcd_engine * e, int n_frames, const uint8_t * d_images, int width, int height, int channels,
                                const void * d_depth, int depth_type, const lcd_orb_params * params, int cap,
                                lcd_keypoint * d_kp_out, uint8_t * d_desc_out, float * d_xyz_out, float * d_uv_out,
                                int * d_n_out, void * stream);
/* 1 if the last lcd_orb_* / lcd_process_frames* call on this engine truncated a FAST candidate list (more than 16 384 corners in
 * level 0, half as many per further level), else 0; synchronises the device.  The host-buffer entry points report the condition
 * themselves (LCD_ERR_CAPACITY); the *_dev variants return before the kernels ran, so their callers ask here. */
int lcd_orb_overflow(lcd_engine * e);
/* Which kernels the last detection used (bit flags; diagnostics for tests and benchmarks): 1 = FAST and blur tiles staged by TMA with a
 * tensor map (rows a multiple of 16 bytes), 2 = descriptors from shared-memory patches (rows a multiple of 4 bytes on every level, edge
 * threshold >= 19), 4 = vectorised gray / mask preparation (rows a multiple of 8 pixels, even height).  0 = the general kernels. */
int lcd_orb_last_path(const lcd_engine * e);

/* ---- detector choice: Kp/DetectorStrategy ------------------------------------------
 * Engine state, like the reference's Feature2D::create (Features2d.cpp:611-700): every entry point that detects
 * (lcd_orb_detect_describe[_dev], lcd_process_frames*, lcd_map_detect_async, lcd_shard_process_frames_dev) uses the
 * detector last set here; an engine that never calls lcd_set_detector detects with ORB.
 * Under LCD_DETECTOR_GFTT_ORB (GFTT/ORB, the reference's default Kp/DetectorStrategy and Vis/FeatureType): corners of
 * cv::GFTTDetector(maxCorners = n_features, quality_level, min_distance, block_size) inside the depth mask, described by
 * cv::ORB::compute (corners within ORB/EdgeThreshold of the border are dropped, the rest keep their order; descriptors on
 * pyramid level 0 with angle -1), then the 3-D lifting of the ORB path.  Of lcd_orb_params, n_features, edge_threshold,
 * patch_size (31), the depth fields and the camera apply; n_levels, scale_factor and fast_threshold are ignored, and
 * the image size needs no power-of-two divisibility.  More than 65 536 candidate corners (local maxima above the quality
 * threshold) in a frame is LCD_ERR_CAPACITY / lcd_orb_overflow, as for the FAST lists. */
#define LCD_DETECTOR_ORB 2       /* Kp/DetectorStrategy=2, the default of every engine */
#define LCD_DETECTOR_GFTT_ORB 8  /* Kp/DetectorStrategy=8: cv::GFTTDetector + cv::ORB::compute */
typedef struct lcd_gftt_params {
	double quality_level; /* GFTT/QualityLevel (0.001), > 0              */
	double min_distance;  /* GFTT/MinDistance (7), >= 0                  */
	int block_size;       /* GFTT/BlockSize (3): 3, 5 or 7               */
	int use_harris;       /* GFTT/UseHarrisDetector: must be 0           */
	double k;             /* GFTT/K (0.04): unused while use_harris is 0 */
} lcd_gftt_params;
/* strategy LCD_DETECTOR_ORB (gftt may be NULL) or LCD_DETECTOR_GFTT_ORB (gftt required); LCD_ERR_INVALID for anything
 * else, including the Harris score. */
int lcd_set_detector(lcd_engine * e, int strategy, const lcd_gftt_params * gftt);

/* ---- dictionary: VWDictionary ------------------------------------------------ */
/* replaces: VWDictionary::addWord (VWDictionary.cpp:1554-1580) for n words whose ids
 * the caller chose (DB load, LTM reactivation).  Words become "not indexed" until
 * lcd_dict_update, exactly like _notIndexedWords. */
int lcd_dict_add_words(lcd_engine * e, const int * ids, const void * desc, int n);
/* replaces: VWDictionary::removeWords / deleteUnusedWords (VWDictionary.cpp:1582-1607).
 * Indexed words leave the search structure at the next lcd_dict_update
 * (_removedIndexedWords); their posting lists are dropped immediately. */
int lcd_dict_remove_words(lcd_engine * e, const int * ids, int n);
/* replaces: VWDictionary::update (VWDictionary.cpp:475-701), Kp/NNStrategy=0 row order:
 * not-indexed words are appended in ascending id, removed rows are compacted out. */
int lcd_dict_update(lcd_engine * e);
/* replaces: VWDictionary::clear (VWDictionary.cpp:842-873) */
int lcd_dict_clear(lcd_engine * e);
/* _visualWords.size(), rows of the search index, _notIndexedWords.size(), _lastWordId */
int lcd_dict_size(const lcd_engine * e);
int lcd_dict_indexed_size(const lcd_engine * e);
int lcd_dict_not_indexed_size(const lcd_engine * e);
int lcd_dict_last_word_id(const lcd_engine * e);
int lcd_dict_set_last_word_id(lcd_engine * e, int id);
/* 1 if the word is in _visualWords (uContains), else 0 */
int lcd_dict_has_word(const lcd_engine * e, int word_id);
/* copy back the indexed rows in search order: ids[rows], desc[rows*dim] (either may be NULL).
 * Mirrors what _dataTree/_mapIndexId hold (VWDictionary.cpp:650-676). */
int lcd_dict_get_indexed(lcd_engine * e, int * ids, void * desc, int cap_rows);

/* The 2-NN of 32-byte binary descriptors has two bit-identical implementations: kernel 1 (default) computes the Hamming
 * distances as an exact s8 GEMM on the tensor cores (nn_tensor.cuh), kernel 0 with XOR + POPC on the integer pipes
 * (nn_hamming.cuh; the only one for other descriptor sizes).  Mirrors choosing Kp/NNStrategy in the reference
 * (VWDictionary::setNNStrategy, VWDictionary.cpp:316-338).  lcd_nn_last_kernel: which one the last search used. */
int lcd_nn_select(lcd_engine * e, int kernel);
int lcd_nn_last_kernel(const lcd_engine * e);
/* Float engines (LCD_DESC_F32) with >= 4096 rows search through the fp16 tensor-core filter + exact re-rank (kernel 1; kernel 0 = the
 * exact CUDA-core scan; results are bit-identical).  Diagnostics of the LAST search of nq queries: how many queries were redone by
 * the exact fallback scan, how many candidate rows the filter passed to the re-rank in total, and how many dictionary rows have been
 * converted to the cached fp16 image since the engine was created (it is converted once per dictionary change, not per search). */
int lcd_nn_f32_stats(lcd_engine * e, int nq, int * n_fallback, long long * n_candidates, long long * rows_converted);

/* replaces: FlannIndex::knnSearch(k=2) on a LinearIndex (FlannIndex.cpp:701-745 ->
 * rtflann linear_index.h:129-146 + result_set.h:151-172): exact 2-NN of every query
 * row over the INDEXED words; ties -> lowest row.  id = 0 and dist = -1 where fewer
 * than 1 (2) indexed words exist.  dist: Hamming count, or squared L2, as float. */
int lcd_dict_knn2(lcd_engine * e, const void * queries, int nq,
                  int * id1, float * d1, int * id2, float * d2);

/* replaces: VWDictionary::addNewWords (VWDictionary.cpp:913-1229) incl. the NNDR test,
 * intra-frame new-word comparison (Kp/NewWordsComparedTogether) and addWordRef for
 * sig_id (VWDictionary.cpp:880-897).  incremental = Kp/IncrementalDictionary,
 * nndr = Kp/NndrRatio.  word_ids_out[nq]; *n_new_out = words created.
 * sig_id <= 0: quantise only, add no references. */
int lcd_dict_quantize(lcd_engine * e, const void * queries, int nq, int sig_id,
                      int incremental, float nndr, int new_words_compared_together,
                      int * word_ids_out, int * n_new_out);

/* replaces: VWDictionary::findNN(cv::Mat) (VWDictionary.cpp:1273-1552): read-only,
 * also searches the not-indexed words; 0 where NNDR rejects. */
int lcd_dict_find_nn(lcd_engine * e, const void * queries, int nq, int incremental,
                     float nndr, int * word_ids_out);

/* ---- inverted index: VisualWord::_references + Memory::computeLikelihood ------ */
/* replaces: VWDictionary::addWordRef (VWDictionary.cpp:880-897) / VisualWord::addRef
 * (VisualWord.cpp:51-63) for the n words of one signature (duplicates count). */
int lcd_index_add_refs(lcd_engine * e, int sig_id, const int * word_ids, int n);
/* replaces: VWDictionary::removeAllWordRef (VWDictionary.cpp:899-911) for every word of
 * sig_id (what Memory::disableWordsRef does, Memory.cpp:6871-6897). */
int lcd_index_remove_sig(lcd_engine * e, int sig_id);
/* ni of Memory::getNi (Memory.cpp:4955-4968): total words of the signature, including
 * un-quantised (<=0) ones.  lcd_index_add_refs / lcd_dict_quantize add n to it; this
 * overrides it. */
int lcd_index_set_ni(lcd_engine * e, const int * sig_ids, const int * ni, int n);
/* bulk load of a word->(signature,count) table in CSR form (cold start from a database,
 * Memory::loadDataFromDb, Memory.cpp:410-438): word_ids[nw], row_ptr[nw+1],
 * sig[row_ptr[nw]], cnt[row_ptr[nw]].  Words must exist in the dictionary. */
int lcd_index_load_csr(lcd_engine * e, const int * word_ids, int nw, const int64_t * row_ptr,
                       const int * sig, const int * cnt);
/* number of signatures referencing word (VisualWord::getReferences().size()), total refs */
int lcd_index_word_nw(lcd_engine * e, int word_id);
long long lcd_index_total_refs(const lcd_engine * e);
/* copy back the posting list of one word sorted by signature id (cap entries max);
 * returns the list length or <0. */
int lcd_index_get_refs(lcd_engine * e, int word_id, int * sig, int * cnt, int cap);

/* replaces: the TF-IDF branch of Memory::computeLikelihood (Memory.cpp:2215-2291):
 * query_word_ids = the new signature's words (any order, duplicates and ids <= 0
 * allowed: uUniqueKeys + the *i>0 test are applied), sig_ids[ns] = the ids to score,
 * n_total = N = Memory::getSignatures().size().  likelihood_out[ns] float. */
int lcd_index_score(lcd_engine * e, const int * query_word_ids, int nq,
                    const int * sig_ids, int ns, int n_total, float * likelihood_out);

/* ---- Bayes filter over the loop-closure hypotheses (SURVEY.md 8(f) #1) ---------------------------
 * replaces: BayesFilter::computePosterior (BayesFilter.cpp:145-270): prior = prediction x last posterior, posterior = likelihood .* prior,
 * normalised; the prediction is the matrix of generatePrediction / addNeighborProb / normalize (:272-505) kept in its sparse form (the
 * reference builds it dense: S x S floats).  The engine keeps the last posterior by place id between calls (updatePosterior, :712-737);
 * lcd_bayes_reset = BayesFilter::reset.
 *   ids[n]         uKeys(likelihood): ascending place ids, ids[0] < 0 = the virtual place (Rtabmap::adjustLikelihood adds it)
 *   likelihood[n]  the adjusted likelihood of each id
 *   col_ptr[n+1], nbr_row[nnz], nbr_level[nnz]   for every place (column) the places its probability mass spreads to:
 *                  Memory::getNeighborsId(id, n_lc - 1, ...) restricted to the places of this call and outside the short-term memory,
 *                  as (position in ids, graph margin) pairs in ascending id order; the place itself (margin 0) must be listed — the
 *                  graph walk is the caller's (Memory), the probability model is computed here.  Columns of loop-closure partners that
 *                  share a neighbour tree (BayesFilter.cpp:378-391) simply carry the same list.  The virtual place has an empty list.
 *   prediction_lc[n_lc]  Bayes/PredictionLC {virtual place, loop closure, level 1, level 2, ...}, virtual_place_prior = Bayes/VirtualPlacePriorThr
 *   posterior_out[n]
 * Float results agree with the reference's dense float product to ~1e-6 relative. */
int lcd_bayes_compute_posterior(lcd_engine * e, const int * ids, const float * likelihood, int n, const int64_t * col_ptr, const int * nbr_row,
                                const int * nbr_level, const double * prediction_lc, int n_lc, float virtual_place_prior, float * posterior_out);
int lcd_bayes_reset(lcd_engine * e);

/* ---- fused, batched localisation query (frozen dictionary + frozen map) ---------
 * One call = B independent queries of the quantise -> score half of the hot path with
 * NO mutation of the engine (SURVEY.md App. C.5): for each frame b
 *   addNewWords(desc_b, sigId) -> computeLikelihood(sig, sig_ids) -> roll back.
 * queries: B*nq_per_frame descriptors (frame-major); n_total = N including the query
 * itself; word_ids_out[B*nq] (new words get ids last_word_id+1.. per frame, not kept);
 * likelihood_out[B*ns]. Either output may be NULL. */
int lcd_localize_batch(lcd_engine * e, const void * queries, int n_frames, int nq_per_frame,
                       int incremental, float nndr, int new_words_compared_together,
                       const int * sig_ids, int ns, int n_total,
                       int * word_ids_out, float * likelihood_out);

/* Same work on device-resident inputs/outputs, asynchronous on `stream` (a cudaStream_t
 * passed as void*; NULL = the engine's stream).  d_queries as above; d_sig_ids[ns];
 * outputs may be NULL.  Used by bench.py for the HBM-resident timing and by the
 * word-range-sharded multi-GPU path. */
int lcd_localize_batch_dev(lcd_engine * e, const void * d_queries, int n_frames, int nq_per_frame,
                           int incremental, float nndr, int new_words_compared_together,
                           const int * d_sig_ids, int ns, int n_total,
                           int * d_word_ids_out, float * d_likelihood_out, void * stream);

/* ---- geometric verification: Memory::computeTransform ----------------------------------
 * Batched verification of n_pairs (FROM = old signature with 3-D points, TO = new signature with
 * 2-D keypoints) hypotheses.  Buffers are [n_pairs][cap] row-major; n_from/n_to give the valid
 * rows of each pair.  Single camera, identity local transform, rectified (no distortion). */
typedef struct lcd_verify_params {
	float nndr;            /* Vis/CorNNDR (0.8)                                             */
	int min_inliers;       /* Vis/MinInliers (20)                                           */
	int iterations;        /* Vis/Iterations (300, <= 320)                                  */
	float reproj_error;    /* Vis/PnPReprojError (2): RANSAC compares the error with its square */
	int refine_iterations; /* Vis/PnPRefineIterations (1)                                   */
	float refine_sigma;    /* refineSigma of util3d::solvePnPRansac (3.0)                   */
	double fx, fy, cx, cy; /* CameraModel::K() of the TO signature                          */
	int var_median_ratio;  /* Vis/PnPVarianceMedianRatio (4, must be > 1)                   */
	float max_variance;    /* Vis/PnPMaxVariance (0 = off): reject when the linear variance exceeds it */
	int split_linear_cov;  /* Vis/PnPSplitLinearCovComponents (0)                           */
	int image_width, image_height; /* CameraModel::imageSize() of the TO camera (0, 0 = not set) */
	int repeat_once;       /* Reg/RepeatOnce (1 in the reference): after a successful first pass, register again with its transform as
	                          the guess (projection + window matching); needs the image size */
	int guess_win_size;    /* Vis/CorGuessWinSize (40 pixels; 0 = no second pass) */
} lcd_verify_params;

typedef struct lcd_verify_result {
	int ok;               /* 1: inliers >= min_inliers (and variance accepted), transform valid */
	int n_matches;        /* correspondences given to PnP                                    */
	int n_inliers;
	int iterations_run;   /* RANSAC iterations the sequential reference would have executed  */
	double rvec[3];       /* PnP pose (object -> camera), Rodrigues vector                   */
	double tvec[3];
	float transform[12];  /* (localTransform * pnp)^-1 as rtabmap::Transform 3x4             */
	double covariance[36]; /* RegistrationInfo::covariance, 6x6 row-major (util3d_motion_estimation.cpp:156-258): identity scaled by
	                          2.1981 x the [n/ratio]-th smallest squared 3-D error (rows 0-2) and angular error (rows 3-5) of the inliers */
} lcd_verify_result;

/* replaces: the global matching of RegistrationVis::computeTransformationImpl through a temporary
 * VWDictionary (RegistrationVis.cpp:1482-1503), Vis/CorNNType 0/3: from_ids/to_ids[n_pairs*cap] word
 * ids of every descriptor (ids start at 1 per pair). */
int lcd_match_pairs(lcd_engine * e, int n_pairs, int cap, const void * desc_from, const int * n_from,
                    const void * desc_to, const int * n_to, float nndr, int * from_ids, int * to_ids);

/* replaces: Memory::computeTransform -> RegistrationVis (global matching, RegistrationVis.cpp:1482-1546)
 * -> util3d::estimateMotion3DTo2D (util3d_motion_estimation.cpp:59-289, incl. the covariance :156-258) -> util3d::solvePnPRansac
 * (:843-990) -> cv3::solvePnPRansac (opencv/solvepnp.cpp:112-417).  xyz_from: NaN where a keypoint has no depth.  xyz_to: the 3-D
 * points of the TO signature (words3B; NaN = none) or NULL when it has none — the covariance then comes from the 10 %-depth ray
 * model (image size set) or from the reprojection RMS (image size 0 x 0), as in the reference.
 * match_ids / inlier_ids [n_pairs*cap] (word ids, ascending / in inlier order) may be NULL. */
int lcd_verify_batch(lcd_engine * e, int n_pairs, int cap, const void * desc_from, const float * xyz_from, const int * n_from,
                     const void * desc_to, const float * uv_to, const float * xyz_to, const int * n_to,
                     const lcd_verify_params * params, lcd_verify_result * results, int * match_ids, int * inlier_ids);

/* replaces: util3d::solvePnPRansac (util3d_motion_estimation.cpp:843-990; argument for argument: objectPoints, imagePoints,
 * cameraMatrix, distCoeffs, rvec, tvec, useExtrinsicGuess, iterationsCount, reprojectionError, minInliersCount, inliers, flags,
 * refineIterations, refineSigma) = cv3::solvePnPRansac (opencv/solvepnp.cpp:112-211: EPnP on 6-point samples drawn with
 * cv::RNG(-1), strict-best model, adaptive iteration count at confidence 0.99, returned pose = best minimal-sample model) followed
 * by the PCL-style refinement loop (:882-989).  object_points[n*3], image_points[n*2] float; K[9] row-major 3x3 double;
 * dist_coeffs[n_dist] must be all zero (or NULL): RTAB-Map passes CameraModel::D(), zeros for rectified images — anything else is
 * rejected with LCD_ERR_INVALID, as are flags != 0 (SOLVEPNP_ITERATIVE) and n == 4 (the reference switches to P3P).
 * rvec / tvec: in = the extrinsic guess (EPnP ignores it, exactly as in the reference), out = the refined pose; left untouched when
 * RANSAC finds no model.  inliers_out[n] (indices into the input, ascending), *n_inliers_out. */
int lcd_pnp_ransac(lcd_engine * e, const float * object_points, const float * image_points, int n, const double K[9],
                   const double * dist_coeffs, int n_dist, double rvec[3], double tvec[3], int use_extrinsic_guess,
                   int iterations, float reproj_error, int min_inliers, int flags, int refine_iterations, float refine_sigma,
                   int * inliers_out, int * n_inliers_out);
/* n_sets independent problems in one launch (one CTA each): object_points[n_sets][cap][3], image_points[n_sets][cap][2],
 * n_points[n_sets], rvec / tvec [n_sets][3], inliers_out[n_sets][cap], n_inliers_out / iterations_run_out [n_sets] (may be NULL). */
int lcd_pnp_ransac_batch(lcd_engine * e, int n_sets, int cap, const float * object_points, const float * image_points, const int * n_points,
                         const double K[9], const double * dist_coeffs, int n_dist, double * rvec, double * tvec, int use_extrinsic_guess,
                         int iterations, float reproj_error, int min_inliers, int flags, int refine_iterations, float refine_sigma,
                         int * inliers_out, int * n_inliers_out, int * iterations_run_out);

/* replaces: cv::BFMatcher on the descriptors of a signature pair (NORM_HAMMING for LCD_DESC_U8 engines, NORM_L2SQR for LCD_DESC_F32):
 *   LCD_MATCH_KNN2       knnMatch(query, train, k = 2)          (RegistrationVis.cpp:1128-1141, :1280-1300; VWDictionary.cpp:1027-1028)
 *   LCD_MATCH_CROSSCHECK BFMatcher(norm, crossCheck = true).match(query, train)   (RegistrationVis.cpp:1452-1453, Vis/CorNNType = 5)
 * for n_pairs independent pairs, [n_pairs][cap] rows each.  idx1 / dist1 [n_pairs*cap]: train index and distance of the best match of
 * every query row (-1 / -1 = none: in cross-check mode the queries OpenCV returns no DMatch for); idx2 / dist2: second neighbour
 * (KNN2 only; may be NULL in cross-check mode).  Ties resolve to the lowest index, as in cv::batchDistance.  Float distances are summed in
 * rtflann's order (dist.h:158-166), which can differ from OpenCV's SIMD order in the last ulp. */
#define LCD_MATCH_KNN2 0
#define LCD_MATCH_CROSSCHECK 1
int lcd_match_bf(lcd_engine * e, int n_pairs, int cap, const void * desc_query, const int * n_query, const void * desc_train,
                 const int * n_train, int mode, int * idx1, float * dist1, int * idx2, float * dist2);

/* ---- signature store + fused query ----------------------------------------------------------
 * The per-node data Memory keeps for verification (Signature::getWordsDescriptors / getWords3,
 * corelib/include/rtabmap/core/Signature.h:155-164), resident in HBM so that the hypothesis picked
 * from the likelihood can be verified without a host round trip.
 * desc [n_sigs][cap][dim], xyz [n_sigs][cap][3] (NaN = no depth), n[n_sigs] valid rows. */
int lcd_sig_add_batch(lcd_engine * e, const int * sig_ids, int n_sigs, int cap, const void * desc,
                      const float * xyz, const int * n);
int lcd_sig_remove(lcd_engine * e, int sig_id);
int lcd_sig_count(const lcd_engine * e);
/* rows the store has allocated so far (freed rows are reused before it grows) */
int lcd_sig_slots(const lcd_engine * e);

/* One call = n_frames independent loop-closure queries through quantise -> score -> verify:
 * lcd_localize_batch, then for every frame the signature with the highest likelihood (first maximum,
 * > 0) is verified against the frame (Memory::computeTransform(hypothesis, frame), FROM = hypothesis
 * with its stored 3-D points, TO = the frame's descriptors + keypoints uv[n_frames][nq][2]).
 * hypothesis_out[n_frames] = verified signature id (0 = none).  Outputs may be NULL. */
int lcd_process_batch(lcd_engine * e, const void * queries, const float * uv, int n_frames, int nq_per_frame,
                      int incremental, float nndr, int new_words_compared_together,
                      const int * sig_ids, int ns, int n_total, const lcd_verify_params * vp,
                      int * word_ids_out, float * likelihood_out, int * hypothesis_out,
                      lcd_verify_result * results);
/* replaces: Rtabmap::adjustLikelihood (Rtabmap.cpp:5691-5760; uMean / uVariance of the values > 0, UMath.h:419-431, :512-526),
 * the step between Memory::computeLikelihood and the Bayes filter.  likelihood[n_frames*ns] are rows in ascending signature id
 * order (as lcd_index_score / lcd_localize_batch return them); adjusted_out[n_frames*(ns+1)]: element 0 of every row is the virtual
 * place, then the ns adjusted values.  virtual_place_ratio = Rtabmap/VirtualPlaceLikelihoodRatio (0 or 1).  Bit-identical to the
 * reference's float arithmetic (the sums run in list order). */
int lcd_adjust_likelihood(lcd_engine * e, const float * likelihood, int n_frames, int ns, int virtual_place_ratio,
                          float * adjusted_out);
int lcd_adjust_likelihood_dev(lcd_engine * e, const float * d_likelihood, int n_frames, int ns, int virtual_place_ratio,
                              float * d_adjusted_out, void * stream);
/* Same on device-resident inputs, asynchronous on `stream`; results stay in engine buffers until
 * lcd_process_fetch copies them back (hypothesis ids, verification results). */
int lcd_process_batch_dev(lcd_engine * e, const void * d_queries, const float * d_uv, int n_frames, int nq_per_frame,
                          int incremental, float nndr, int new_words_compared_together,
                          const int * d_sig_ids, int ns, int n_total, const lcd_verify_params * vp,
                          int * d_word_ids_out, float * d_likelihood_out, void * stream);
int lcd_process_fetch(lcd_engine * e, int n_frames, int * hypothesis_out, lcd_verify_result * results);
/* The same download queued on `stream` (NULL: the engine's stream) behind the step that produced the results, without any
 * synchronisation: a caller that keeps steps in flight (pinned output buffers, one set per step in flight) reads them after its own
 * event / stream synchronisation, while the next step already runs. */
int lcd_process_fetch_async(lcd_engine * e, int n_frames, int * hypothesis_out, lcd_verify_result * results, void * stream);
/* The whole hot path for n_frames frames: Memory::update (detect + quantise, Rtabmap.cpp:1470) ->
 * Memory::computeLikelihood (:2117) -> Memory::computeTransform of the top hypothesis (:3143), as
 * independent localisation queries (no mutation).  Host buffers in, host results out: n_kp_out[n_frames]
 * keypoints found, word_ids_out[n_frames * params->n_features] (0 in the padding rows of short frames),
 * likelihood_out[n_frames*ns], hypothesis_out / results as lcd_process_batch (vp may be NULL: no verify). */
int lcd_process_frames(lcd_engine * e, int n_frames, const uint8_t * images, int width, int height, int channels,
                       const void * depth, int depth_type, const lcd_orb_params * params,
                       int incremental, float nndr, int new_words_compared_together,
                       const int * sig_ids, int ns, int n_total, const lcd_verify_params * vp,
                       int * n_kp_out, int * word_ids_out, float * likelihood_out, int * hypothesis_out,
                       lcd_verify_result * results);
/* Pipelined form of lcd_process_frames for a stream of batches (a relocalisation service): _submit queues the upload
 * and the kernels of a batch and returns; _wait blocks until the OLDEST submitted batch is complete and its output
 * arrays are filled.  Two batches may be in flight, so the PCIe upload of batch k+1 runs under the kernels of batch k.
 * Input and output host arrays must stay valid (and should be pinned) until the matching _wait returns. */
int lcd_process_frames_submit(lcd_engine * e, int n_frames, const uint8_t * images, int width, int height, int channels,
                              const void * depth, int depth_type, const lcd_orb_params * params,
                              int incremental, float nndr, int new_words_compared_together,
                              const int * sig_ids, int ns, int n_total, const lcd_verify_params * vp,
                              int * n_kp_out, int * word_ids_out, float * likelihood_out, int * hypothesis_out,
                              lcd_verify_result * results);
int lcd_process_frames_wait(lcd_engine * e);
int lcd_process_frames_dev(lcd_engine * e, int n_frames, const uint8_t * d_images, int width, int height, int channels,
                           const void * d_depth, int depth_type, const lcd_orb_params * params,
                           int incremental, float nndr, int new_words_compared_together,
                           const int * d_sig_ids, int ns, int n_total, const lcd_verify_params * vp,
                           int * d_word_ids_out, float * d_likelihood_out, void * stream);

/* ---- mapping mode: Memory::update + Memory::computeLikelihood for a STREAM of frames (Rtabmap.cpp:1470, :2117) --------------------------
 * Frame t+1 depends on frame t (its new words, its references), so the frames of one map cannot be batched; what can overlap is the
 * detection of the next frame.  lcd_map_detect_async uploads one image (+ depth) and runs ORB detect + describe + 3-D lifting on the
 * engine's ORB stream and returns at once (two detections may be in flight; host buffers must stay valid until the matching
 * lcd_map_frame).  lcd_map_frame takes the OLDEST detection and does, in the reference's order: VWDictionary::update (Memory::preUpdate,
 * Memory.cpp:1004-1016), addNewWords of the frame's descriptors for sig_id incl. the references (the descriptors never leave the device),
 * and — when wm_sig_ids is given — the TF-IDF likelihood against those signatures (n_total = Memory::getSignatures().size()).
 * Outputs: *n_kp_out, kp_out / desc_out / xyz_out [n_kp] (any may be NULL), word_ids_out[Kp/MaxFeatures] (first n_kp valid), *n_new_out,
 * likelihood_out[ns].  Identical, call for call, to lcd_orb_detect_describe + lcd_dict_update + lcd_dict_quantize + lcd_index_score. */
int lcd_map_detect_async(lcd_engine * e, const uint8_t * image, int width, int height, int channels, const void * depth, int depth_type,
                         const lcd_orb_params * params);
int lcd_map_frame(lcd_engine * e, int sig_id, int incremental, float nndr, int new_words_compared_together, const int * wm_sig_ids, int ns,
                  int n_total, int * n_kp_out, lcd_keypoint * kp_out, uint8_t * desc_out, float * xyz_out, int * word_ids_out, int * n_new_out,
                  float * likelihood_out);

/* The verification half alone, for likelihood rows that already exist on the device (the sharded
 * multi-GPU path all-reduces the scores first, then every rank verifies its share of the frames):
 * arg-max hypothesis of each of the n_frames rows of d_likelihood[n_frames][ns], then
 * Memory::computeTransform(hypothesis, frame).  Results via lcd_process_fetch. */
int lcd_verify_top_dev(lcd_engine * e, const void * d_queries, const float * d_uv, int n_frames, int nq_per_frame,
                       const float * d_likelihood, const int * d_sig_ids, int ns, const lcd_verify_params * vp, void * stream);

/* ---- word-range sharding across GPUs (SURVEY.md §8(e)) ---------------------------
 * Each rank owns the words whose row (in ascending id order) falls in its range; rows
 * are numbered globally: set the global row offset of this shard so that packed top-2
 * keys (dist<<22 | global_row) from different ranks merge with the reference's
 * tie-break (lowest row = lowest id). */
int lcd_shard_set_row_offset(lcd_engine * e, int global_row_offset);
/* stage 1: local top-2 keys of every query over this rank's rows -> d_keys_out[2*nq] u32
 * (0xFFFFFFFF = none).  All-gather these across ranks, then call stage 2 on every rank. */
int lcd_shard_knn2_keys_dev(lcd_engine * e, const void * d_queries, int nq, uint32_t * d_keys_out,
                            void * stream);
/* stage 2, sharded by FRAME (what scales): every rank resolves only its own frames [frame0, frame0+n_frames) of the job's
 * n_frames_total — merge of the G gathered key sets [G][2 * n_frames_total * nq] + NNDR / new-word pass — and writes their
 * word ids (d_word_ids_out[n_frames*nq], 0 in padding rows; d_n_per_frame[n_frames_total] valid descriptors per frame or NULL).
 * All-gather the word ids, then lcd_shard_score_ids_dev on every rank accumulates this rank's share (its word range) of the
 * TF-IDF scores of ALL frames from the ids (uUniqueKeys + "id > 0" filter of Memory::computeLikelihood, Memory.cpp:2238-2256)
 * into d_scores_out[n_frames*ns]; all-reduce(sum), then lcd_shard_finalize_dev. */
int lcd_shard_resolve_frames_dev(lcd_engine * e, const void * d_queries_all, int frame0, int n_frames, int n_frames_total,
                                 int nq_per_frame, const uint32_t * d_keys_gathered, int n_ranks, const int * d_row_ids,
                                 int last_word_id, int incremental, float nndr, int new_words_compared_together,
                                 const int * d_n_per_frame, int * d_word_ids_out, void * stream);
int lcd_shard_score_ids_dev(lcd_engine * e, const int * d_word_ids_all, int n_frames, int nq_per_frame,
                            const int * d_sig_ids, int ns, int n_total, long long * d_scores_out, void * stream);
/* stage 2: merge G gathered key sets [G][2*nq], run the replicated NNDR / new-word pass,
 * and accumulate this rank's share of the TF-IDF scores into d_scores_out[n_frames*ns]
 * (fixed-point int64, exact and order-independent; all-reduce(sum) them, then call
 * lcd_shard_finalize_dev).  d_row_ids: global row -> word id table [total_rows]. */
int lcd_shard_resolve_score_dev(lcd_engine * e, const void * d_queries, int n_frames, int nq_per_frame,
                                const uint32_t * d_keys_gathered, int n_ranks,
                                const int * d_row_ids, int total_rows, int last_word_id,
                                int incremental, float nndr, int new_words_compared_together,
                                const int * d_sig_ids, int ns, int n_total,
                                int * d_word_ids_out, long long * d_scores_out, void * stream);
int lcd_shard_finalize_dev(lcd_engine * e, const long long * d_scores, int n, float * d_likelihood_out,
                           void * stream);

/* ---- the exchanges behind the C ABI: one engine = one rank of a word-range-sharded job ----------------------------------
 * NCCL is loaded at run time (dlopen of libnccl.so.2: the host's own copy when it has one).  Bootstrap as any NCCL program: rank 0 calls
 * lcd_shard_unique_id, the host sends the 128 bytes to the other ranks over whatever channel it has (MPI, sockets, a file), every rank
 * calls lcd_shard_comm_init; or hand over a communicator the host already owns with lcd_shard_comm_adopt (ncclComm_t as void *). */
int lcd_shard_unique_id(char id_out[128]);
int lcd_shard_comm_init(lcd_engine * e, const char id[128], int rank, int n_ranks);
int lcd_shard_comm_adopt(lcd_engine * e, void * nccl_comm, int rank, int n_ranks);
int lcd_shard_comm_destroy(lcd_engine * e);
/* One step of the sharded job on this rank, entirely on the device: detect + describe the n_frames LOCAL frames, all-gather of the
 * descriptors, top-2 keys of every rank's descriptors over the local word range (lcd_shard_set_row_offset), all-to-all so that every rank
 * receives the keys of ITS frames, merge + NNDR / new-word pass of the local frames, all-gather of their word ids, TF-IDF of all frames
 * over the local word range, reduce-scatter of the exact 64-bit fixed-point sums, likelihood + verification of the local frames'
 * top hypotheses (results through lcd_process_fetch).  The dictionary search runs as two halves of the local batch so that the
 * descriptor and key exchanges (on the engine's communication stream) overlap a search kernel; the later stages run once on the whole
 * batch.  LCD_SHARD_TRACE=1|2 (environment) prints a per-stage timeline of the step to stderr.  d_row_ids_global: global row -> word id of the WHOLE dictionary
 * (rows of all ranks in ascending id order); d_word_ids_out[n_frames * n_features] (may be NULL), d_likelihood_out[n_frames * ns].
 * Every rank must call it with the same n_frames.  Results equal the unsharded engine's: word ids bit for bit, likelihood from the same
 * exact sums. */
int lcd_shard_process_frames_dev(lcd_engine * e, int n_frames, const uint8_t * d_images, int width, int height, int channels, const void * d_depth,
                                 int depth_type, const lcd_orb_params * params, int incremental, float nndr, int new_words_compared_together,
                                 const int * d_sig_ids, int ns, int n_total, const int * d_row_ids_global, int last_word_id,
                                 const lcd_verify_params * vp, int * d_word_ids_out, float * d_likelihood_out, void * stream);

/* ---- measurement hooks ---------------------------------------------------------------
 * Optional per-kernel timing with CUDA events recorded on the launching stream around
 * every launch of kernel class `which` (0 = dictionary NN, 1 = resolve, 2 = score, 3 = pair
 * matching, 4 = PnP RANSAC, 5 = all detect kernels: ORB or GFTT/ORB).
 * lcd_profile_read synchronises, returns the summed device time and the launch count
 * since the last reset. */
#define LCD_PROF_NN 0
#define LCD_PROF_RESOLVE 1
#define LCD_PROF_SCORE 2
#define LCD_PROF_MATCH 3
#define LCD_PROF_PNP 4
#define LCD_PROF_ORB 5
int lcd_profile_enable(lcd_engine * e, int on);
int lcd_profile_read(lcd_engine * e, int which, double * total_ms, long long * launches);
int lcd_profile_reset(lcd_engine * e);

/* copy an internal ORB buffer of the last lcd_orb_* call back to the host (diagnostics / tests):
 * which = 0 gray pyramid, 1 mask pyramid, 2 blurred pyramid, 3 FAST candidate keys, 4 candidate counts,
 * 5 keypoints per level counts, 6 FAST score pyramid, 10 GFTT minimum-eigenvalue map (float [n_frames][h][w]).  Returns the number of bytes copied (<= cap_bytes) or <0. */
long long lcd_debug_orb_buffer(lcd_engine * e, int which, void * out, long long cap_bytes);

/* engine stream (cudaStream_t as void*) and a full device sync, for harnesses */
void * lcd_stream(lcd_engine * e);
int lcd_synchronize(lcd_engine * e);

#ifdef __cplusplus
}
#endif
#endif /* LCD_B200_H */
