// engine.cu — host side of the loop-closure engine and the C ABI (include/lcd_b200.h).
//
// One lcd_engine = the device-resident state of one rtabmap::VWDictionary
// (corelib/include/rtabmap/core/VWDictionary.h:46-160): the vocabulary matrix in search
// order (_dataTree + _mapIndexId), the not-indexed tail (_notIndexedWords), and the inverted
// index (VisualWord::_references of every word) as an arena of posting lists.  The host keeps
// only the bookkeeping the reference keeps in std::map's (id -> row, list extents, the words
// of each signature); all descriptor and posting data lives in HBM and every distance,
// decision and score is computed by the kernels in nn_hamming.cuh / resolve.cuh / score.cuh.
// There is deliberately no CPU fallback: every entry point fails with LCD_ERR_CUDA if the
// device is missing.
#include "../../include/lcd_b200.h"
#include "common.cuh"
#include "nn_hamming.cuh"
#include "nn_tensor.cuh"
#include "l2_path.cuh"
#include "nn_tensor_f32.cuh"
#include "resolve.cuh"
#include "score.cuh"
#include "bayes.cuh"
#include "verify.cuh"
#include "match_bf.cuh"
#include "orb.cuh"
#include "gftt.cuh"

#include <cuda.h>
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <utility>
#include <chrono>
#include <vector>

using namespace lcd;

namespace {

thread_local std::string g_create_error;

template <typename T>
struct DevBuf
{
	T * p = nullptr;
	size_t cap = 0; // elements
	~DevBuf() { release(); }
	void release()
	{
		if (p) cudaFree(p);
		p = nullptr;
		cap = 0;
	}
	// grow to at least n elements; keep the first `keep` elements; zero the rest if asked.
	// A re-growth replaces a buffer that kernels on ANY stream of the engine (caller streams of the _dev entry points, the ORB side
	// streams) may still be reading or writing: the device is drained first, so the copy sees final data and the free is safe.
	cudaError_t reserve(size_t n, size_t keep, bool zero_new, cudaStream_t s)
	{
		if (n <= cap) return cudaSuccess;
		size_t ncap = std::max(n, cap + cap / 2 + 16);
		T * np = nullptr;
		cudaError_t err = cudaMalloc(&np, ncap * sizeof(T));
		if (err != cudaSuccess) return err;
		if (p) err = cudaDeviceSynchronize();
		if (err == cudaSuccess && zero_new) err = cudaMemsetAsync(np, 0, ncap * sizeof(T), s);
		if (err == cudaSuccess && p && keep) err = cudaMemcpyAsync(np, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, s);
		if (err == cudaSuccess && p) err = cudaStreamSynchronize(s);
		if (err != cudaSuccess)
		{
			cudaFree(np);
			return err;
		}
		if (p) cudaFree(p);
		p = np;
		cap = ncap;
		return cudaSuccess;
	}
};

template <typename T>
struct PinBuf
{
	T * p = nullptr;
	size_t cap = 0;
	~PinBuf()
	{
		if (p) cudaFreeHost(p);
	}
	cudaError_t reserve(size_t n)
	{
		if (n <= cap) return cudaSuccess;
		if (p) cudaFreeHost(p);
		p = nullptr;
		cap = 0;
		size_t ncap = n + n / 2 + 16;
		cudaError_t err = cudaMallocHost(&p, ncap * sizeof(T));
		if (err == cudaSuccess) cap = ncap;
		return err;
	}
};

// Zero-fill on the SMs.  cudaMemsetAsync may be scheduled on a copy engine, where it queues behind the (much longer) host ->
// device upload of the NEXT batch and stalls the kernels of the current one (measured: 1.8 ms per step in the pipelined path).
__global__ void zero_fill_kernel(uint4 * __restrict__ p16, size_t n16, unsigned char * __restrict__ tail, size_t n_tail)
{
	const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i < n16) p16[i] = make_uint4(0, 0, 0, 0);
	if (i < n_tail) tail[i] = 0;
}
static cudaError_t zero_fill_async(void * p, size_t bytes, cudaStream_t s)
{
	if (!bytes) return cudaSuccess;
	if (reinterpret_cast<uintptr_t>(p) & 15) return cudaMemsetAsync(p, 0, bytes, s);
	const size_t n16 = bytes / 16, n_tail = bytes % 16;
	const size_t n = std::max(n16, n_tail);
	zero_fill_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(static_cast<uint4 *>(p), n16, static_cast<unsigned char *>(p) + n16 * 16, n_tail);
	return cudaGetLastError();
}

size_t depth_elem_bytes(int depth_type) { return depth_type == LCD_DEPTH_U16_MM ? 2 : (depth_type == LCD_DEPTH_MASK_U8 ? 1 : 4); }

// NCCL is loaded at run time (dlopen): single-GPU users of liblcd_b200.so need no NCCL, and a host that already carries one
// (PyTorch's bundled libnccl.so.2, or the system's) shares it with the library.
struct NcclApi
{
	ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
	ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
	ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
	ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*ReduceScatter)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*GroupStart)() = nullptr;
	ncclResult_t (*GroupEnd)() = nullptr;
	const char * (*GetErrorString)(ncclResult_t) = nullptr;
	bool ok = false;
	std::string why;
};
const NcclApi & nccl_api()
{
	static NcclApi api = []() {
		NcclApi a;
		void * h = nullptr;
		for (const char * name : {"libnccl.so.2", "libnccl.so"})
		{
			h = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
			if (h) break;
		}
		if (!h)
		{
			a.why = std::string("libnccl.so.2 not found: ") + (dlerror() ? dlerror() : "");
			return a;
		}
#define LCD_NCCL_SYM(field, sym)                                         \
	a.field = reinterpret_cast<decltype(a.field)>(dlsym(h, sym));       \
	if (!a.field)                                                        \
	{                                                                    \
		a.why = std::string("NCCL symbol missing: ") + sym;              \
		return a;                                                        \
	}
		LCD_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
		LCD_NCCL_SYM(CommInitRank, "ncclCommInitRank")
		LCD_NCCL_SYM(CommDestroy, "ncclCommDestroy")
		LCD_NCCL_SYM(AllGather, "ncclAllGather")
		LCD_NCCL_SYM(ReduceScatter, "ncclReduceScatter")
		LCD_NCCL_SYM(Send, "ncclSend")
		LCD_NCCL_SYM(Recv, "ncclRecv")
		LCD_NCCL_SYM(GroupStart, "ncclGroupStart")
		LCD_NCCL_SYM(GroupEnd, "ncclGroupEnd")
		LCD_NCCL_SYM(GetErrorString, "ncclGetErrorString")
#undef LCD_NCCL_SYM
		a.ok = true;
		return a;
	}();
	return api;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder()
{
	static EncodeTiledFn fn = []() -> EncodeTiledFn {
		void * p = nullptr;
		cudaDriverEntryPointQueryResult q;
		if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return nullptr;
		return reinterpret_cast<EncodeTiledFn>(p);
	}();
	return fn;
}

// 3-D tensor map over the u8 planes [frames][h][w] of one pyramid level (frame pitch `frame_stride` bytes), box = box_w x box_h x 1,
// zero fill outside.  false: the geometry does not meet the TMA alignment rules (or the driver lacks the call): plain loads instead.
static_assert(sizeof(CUtensorMap) == sizeof(lcd::OrbTensorMap), "tensor map size");
bool make_plane_tensor_map(lcd::OrbTensorMap * out, const uint8_t * base, int w, int h, int n_frames, size_t frame_stride, int box_w, int box_h)
{
	EncodeTiledFn enc = tensor_map_encoder();
	if (!enc || (w % 16) || (frame_stride % 16) || (reinterpret_cast<uintptr_t>(base) % 16) || n_frames <= 0) return false;
	const cuuint64_t dims[3] = {static_cast<cuuint64_t>(w), static_cast<cuuint64_t>(h), static_cast<cuuint64_t>(n_frames)};
	const cuuint64_t strides[2] = {static_cast<cuuint64_t>(w), static_cast<cuuint64_t>(frame_stride)};
	const cuuint32_t box[3] = {static_cast<cuuint32_t>(box_w), static_cast<cuuint32_t>(box_h), 1u};
	const cuuint32_t estr[3] = {1u, 1u, 1u};
	return enc(reinterpret_cast<CUtensorMap *>(out), CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t *>(base), dims, strides, box, estr,
	           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int env_int(const char * name, int def)
{
	const char * v = getenv(name);
	return v && *v ? atoi(v) : def;
}

} // namespace

struct lcd_engine
{
	lcd_config cfg{};
	int nw = 0; // 32-bit words per descriptor
	mutable std::string err;
	mutable std::mutex err_mu;                // lcd_orb_* may fail on another thread than the dictionary calls
	cudaStream_t stream = nullptr;
	cudaStream_t orb_stream = nullptr;        // host-buffer lcd_orb_detect_describe: its own stream, so that it overlaps lcd_dict_update
	cudaStream_t copy_stream = nullptr;       // host -> device image chunks of lcd_process_frames
	std::vector<cudaEvent_t> copy_events;     // one per chunk
	cudaEvent_t copy_fence = nullptr;
	cudaStream_t aux_stream[4] = {nullptr, nullptr, nullptr, nullptr}; // fork/join side streams (coarse pyramid levels of the ORB selection)
	cudaEvent_t aux_fork = nullptr, aux_blur_done = nullptr, aux_join[4] = {nullptr, nullptr, nullptr, nullptr};
	// lcd_process_frames_submit / _wait: two batches in flight
	struct Flight
	{
		DevBuf<uint8_t> img;
		DevBuf<unsigned char> depth;
		DevBuf<int> sig_ids;
		PinBuf<PackedVerifyResult> res;
		PinBuf<int> overflow;                  // ORB candidate overflow flag of the batch
		cudaEvent_t uploaded = nullptr, done = nullptr;
		lcd_verify_result * user_results = nullptr;
		int n_frames = 0;
		cudaEvent_t t_h0 = nullptr, t_h1 = nullptr, t_c0 = nullptr, t_c1 = nullptr; // LCD_DEBUG_TIMELINE
	};
	cudaEvent_t t_base = nullptr;
	Flight flights[2];
	int flight_head = 0, flights_busy = 0;
	DevBuf<PackedVerifyResult> v_packed;
	PinBuf<PackedVerifyResult> h_packed;
	PinBuf<int> h_overflow;
	std::atomic<long long> launches{0};
	int sm_count = 148;
	int smem_optin = 0;

	// --- vocabulary: rows [0,n_indexed) searchable, [n_indexed, n_indexed+n_pending) not indexed
	DevBuf<uint32_t> vocab, vocab_alt;
	DevBuf<int> row_ids, row_ids_alt;
	std::vector<int> h_row_ids;
	std::unordered_map<int, int> id2row;
	std::unordered_set<int> removed_rows; // indexed rows leaving at the next update
	int n_indexed = 0, n_pending = 0;
	bool pending_sorted = true;
	int last_word_id = 0;
	int row_offset = 0;

	// --- inverted index
	DevBuf<uint32_t> post_off;
	DevBuf<int> post_len;
	std::vector<uint32_t> h_off;
	std::vector<int> h_len, h_cap;
	DevBuf<int2> postings;
	size_t post_used = 0;
	DevBuf<int> ni;
	std::vector<int> h_ni;
	std::unordered_map<int, std::vector<std::pair<int, int>>> sig_words; // sig -> sorted (word,count)
	long long total_refs = 0;

	// --- scratch
	DevBuf<uint32_t> d_queries;
	DevBuf<uint2> d_partial;
	DevBuf<uint4> tc_words;             // cached +-1 byte image of the vocabulary rows [0, tc_rows) for the tensor-core 2-NN
	int tc_rows = 0;
	DevBuf<uint32_t> d_keys;
	DevBuf<int> d_word_ids, d_n_new, d_in_ids;
	DevBuf<int> uq_count, uq_word, uq_prefix;
	DevBuf<float> uq_idf;
	DevBuf<long long> acc;
	int acc_stride = 0;
	DevBuf<int> d_sig_ids;
	DevBuf<float> d_like;
	DevBuf<int> d_i1, d_i2;
	DevBuf<float> d_f1, d_f2;
	DevBuf<RefOp> d_ops;
	DevBuf<MoveOp> d_moves;
	DevBuf<int> d_perm;
	// Bayes filter (bayes.cuh): the last posterior by place id + per-call scratch
	DevBuf<int> by_ids, by_colptr, by_row, by_level, by_entry_col, by_state_ids;
	DevBuf<float> by_like, by_last, by_u, by_scale, by_delta, by_post, by_state_post;
	DevBuf<double> by_lc, by_prior, by_sums;
	int by_n_state = 0;
	// verification scratch
	DevBuf<uint32_t> v_df, v_dt;
	DevBuf<float> v_xyz, v_uv, v_obj, v_img, v_T, v_xyz_to, v_obj_to;
	DevBuf<double> v_cov6;
	DevBuf<ulonglong2> bf_keys_a, bf_keys_b;
	DevBuf<unsigned long long> bf_best;
	DevBuf<long long> v_clk;
	DevBuf<int> v_nf, v_nt, v_mid, v_mfrom, v_mto, v_nm, v_fid, v_tid, v_inl, v_ninl, v_iters, v_ok, v_inl_ids;
	DevBuf<double> v_rvec, v_tvec;
	// signature store (Signature::getWordsDescriptors / getWords3 of the nodes in working memory)
	DevBuf<uint32_t> st_desc;
	DevBuf<float> st_xyz;
	DevBuf<int> st_n, st_slot_of_sig;
	std::vector<int> h_slot_of_sig, free_slots;
	int st_cap = 0, st_slots = 0;
	DevBuf<int> d_hyp_id, d_hyp_slot;
	// ORB workspace
	DevBuf<uint8_t> o_img, o_gray, o_mask, o_blur, o_desc;
	DevBuf<unsigned char> o_depth;
	DevBuf<uint32_t> o_cand;
	DevBuf<int> o_cand_count, o_level_n, o_n, o_overflow;
	DevBuf<OrbKeypoint> o_level_kp, o_kp;
	DevBuf<float> o_xyz, o_uv;
	float gauss_sigma_loaded = -1.f;
	int orb_tma_used = 0; // the last FAST launch staged its tiles through a tensor map
	int orb_path = 0;     // lcd_orb_last_path flags of the last detection
	// detector choice (lcd_set_detector) and the GFTT/ORB workspace
	int detector = LCD_DETECTOR_ORB;
	lcd_gftt_params gftt{0.001, 7.0, 3, 0, 0.04};
	DevBuf<float> g_eig;
	DevBuf<uint32_t> g_max, g_occ;
	DevBuf<unsigned long long> g_cand;
	DevBuf<int> g_cand_count;
	DevBuf<double> g_rowsum;
	DevBuf<float> d_uv;

	// measurement hooks (lcd_profile_*)
	bool prof_on = false;
	struct Prof
	{
		std::vector<cudaEvent_t> ev; // start/stop pairs
		size_t used = 0;
	} prof[6];

	// tuning knobs (env: LCD_NN_CTAS_PER_SM, LCD_NN_TQ, LCD_NN_VARIANT, LCD_SCORE_BLOCKS)
	int nn_ctas_per_sm = 2, nn_tq = 8, nn_variant = 2, score_blocks = 32;
	bool f32 = false;    // LCD_DESC_F32: squared-L2 path (l2_path.cuh)
	DevBuf<ulonglong2> d_partial64, tf_fb_scratch;
	// float descriptors on the tensor cores (nn_tensor_f32.cuh): cached fp16 image of rows [0, tf_rows) + their norms
	DevBuf<uint4> tf_words, tf_queries, tf_words_aug, tf_queries_aug;
	DevBuf<float> tf_qn;
	DevBuf<uint32_t> tf_tau, tf_cand, tf_wmax2;  // tf_wmax2[0] = bits of the largest |w|^2 seen
	DevBuf<int> tf_cand_count, tf_fb_list, tf_flags; // tf_flags[0] = fallback count, tf_flags[1] = "a row does not fit fp16"
	int tf_rows = 0;            // rows of the vocabulary whose image is current
	bool tf_disabled = false;   // a dictionary row does not fit fp16: exact CUDA-core path from then on
	int nn_f32_tensor = 1;      // LCD_NN_F32_TENSOR=0 forces the exact CUDA-core kernel
	int nn_last_f32_tensor = 0;
	long long tf_img_builds = 0; // rows expanded so far (diagnostics: the image is built once per dictionary change)
	int nn_tensor = 1;   // 256-bit descriptors: tcgen05 int8 path (nn_tensor.cuh); 0 = POPC kernel (nn_hamming.cuh)
	int nn_last_tensor = 0; // which kernel the last run_knn used (bench / diagnostics)
	// mapping mode (lcd_map_*): detection of frame t+1 on the ORB stream while frame t is quantised and scored
	struct MapSlot
	{
		DevBuf<uint8_t> img, desc;
		DevBuf<unsigned char> depth;
		DevBuf<OrbKeypoint> kp;
		DevBuf<float> xyz;
		DevBuf<int> n;
		PinBuf<int> h_n, h_overflow;
		cudaEvent_t done = nullptr;
		int cap = 0;
		bool busy = false;
	};
	MapSlot map_slots[2];
	int map_head = 0, map_busy = 0;
	PinBuf<int> map_h_words, map_h_scalars;
	// word-range sharding across GPUs (lcd_shard_*): NCCL communicator + exchange buffers of the fused sharded step
	ncclComm_t comm = nullptr;
	bool comm_owned = false;
	int sh_rank = 0, sh_ranks = 1;
	cudaStream_t comm_stream = nullptr;
	cudaEvent_t sh_ev[2][8] = {};
	cudaEvent_t sh_tr[2] = {};         // LCD_SHARD_TRACE=1: first / last kernel of the step on the compute stream
	int sh_trace = 0, sh_ring_step = 0;
	bool sh_trace_armed = false;
	std::vector<cudaEvent_t> sh_ring;  // [step][half][8 stage events + 1 begin/end]
	DevBuf<uint8_t> sh_desc_all[2];
	DevBuf<int> sh_n_all, sh_words_loc[2], sh_words_all[2];
	DevBuf<uint32_t> sh_keys[2], sh_keys_mine[2];
	DevBuf<long long> sh_scores[2], sh_scores_loc[2];
	bool match_has_xyz_to = false; // verify_upload staged xyz_to for the next launch_match
	bool pnp_has_obj_to = false;   // the last launch_match gathered obj_to for launch_pnp
};

#define LCD_FAIL(e, code, ...)                          \
	do                                                  \
	{                                                   \
		char _b[512];                                   \
		snprintf(_b, sizeof(_b), __VA_ARGS__);          \
		{                                               \
			std::lock_guard<std::mutex> _g((e)->err_mu); \
			(e)->err = _b;                              \
		}                                               \
		return (code);                                  \
	} while (0)

#define LCD_CUDA(e, call)                                                                          \
	do                                                                                             \
	{                                                                                              \
		cudaError_t _c = (call);                                                                   \
		if (_c != cudaSuccess)                                                                     \
		{                                                                                          \
			LCD_FAIL(e, LCD_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_c), __FILE__, __LINE__); \
		}                                                                                          \
	} while (0)

#define LCD_NCCL(e, call)                                                                                     \
	do                                                                                                        \
	{                                                                                                         \
		ncclResult_t _n = (call);                                                                             \
		if (_n != ncclSuccess) LCD_FAIL(e, LCD_ERR_CUDA, "%s failed: %s", #call, nccl_api().GetErrorString(_n)); \
	} while (0)

#define LCD_CHECK_LAUNCH(e)                 \
	do                                      \
	{                                       \
		++(e)->launches;                    \
		LCD_CUDA(e, cudaGetLastError());    \
	} while (0)

#define LCD_TRY(expr)              \
	do                             \
	{                              \
		int _r = (expr);           \
		if (_r != LCD_OK) return _r; \
	} while (0)

namespace {

int total_rows(const lcd_engine * e) { return e->n_indexed + e->n_pending; }

int set_device(lcd_engine * e)
{
	LCD_CUDA(e, cudaSetDevice(e->cfg.device));
	return LCD_OK;
}

int ensure_rows(lcd_engine * e, int rows)
{
	const size_t keep = static_cast<size_t>(total_rows(e));
	LCD_CUDA(e, e->vocab.reserve(static_cast<size_t>(rows) * e->nw, keep * e->nw, false, e->stream));
	LCD_CUDA(e, e->row_ids.reserve(static_cast<size_t>(rows), keep, false, e->stream));
	return LCD_OK;
}

int ensure_ids(lcd_engine * e, int max_id)
{
	const size_t need = static_cast<size_t>(max_id) + 1;
	if (need > e->h_len.size())
	{
		const size_t old = e->h_len.size();
		const size_t ncap = std::max(need, old + old / 2 + 1024);
		LCD_CUDA(e, e->post_off.reserve(ncap, old, true, e->stream));
		LCD_CUDA(e, e->post_len.reserve(ncap, old, true, e->stream));
		e->h_off.resize(e->post_off.cap, 0u);
		e->h_len.resize(e->post_off.cap, 0);
		e->h_cap.resize(e->post_off.cap, 0);
	}
	return LCD_OK;
}

int ensure_sigs(lcd_engine * e, int max_sig)
{
	const size_t need = static_cast<size_t>(max_sig) + 1;
	if (need > e->h_ni.size())
	{
		const size_t old = e->h_ni.size();
		const size_t ncap = std::max(need, old + old / 2 + 1024);
		LCD_CUDA(e, e->ni.reserve(ncap, old, true, e->stream));
		e->h_ni.resize(e->ni.cap, 0);
	}
	return LCD_OK;
}

int ensure_acc(lcd_engine * e, int n_frames)
{
	const int stride = static_cast<int>(e->h_ni.size());
	if (stride != e->acc_stride || e->acc.cap < static_cast<size_t>(stride) * n_frames)
	{
		LCD_CUDA(e, e->acc.reserve(static_cast<size_t>(std::max(stride, 1)) * n_frames, 0, false, e->stream));
		e->acc_stride = stride;
	}
	return LCD_OK;
}

int ensure_postings(lcd_engine * e, size_t extra)
{
	if (e->post_used + extra > 0xFFFFFFF0ull) LCD_FAIL(e, LCD_ERR_CAPACITY, "posting arena exceeds 2^32 entries");
	LCD_CUDA(e, e->postings.reserve(e->post_used + extra, e->post_used, false, e->stream));
	return LCD_OK;
}

// ---- measurement hooks ------------------------------------------------------------------
void prof_mark(lcd_engine * e, int which, cudaStream_t s)
{
	if (!e->prof_on) return;
	auto & p = e->prof[which];
	if (p.used == p.ev.size())
	{
		cudaEvent_t ev;
		if (cudaEventCreate(&ev) != cudaSuccess) return;
		p.ev.push_back(ev);
	}
	cudaEventRecord(p.ev[p.used++], s);
}

// ---- kernel launch helpers --------------------------------------------------------------
template <int NW, int TQ, int VARIANT>
int launch_knn_t(lcd_engine * e, const uint32_t * d_q, int nq_total, int n_rows, int n_chunks, int rows_per_cta,
                 uint2 * d_partial, cudaStream_t s)
{
	auto kern = knn2_hamming_kernel<NW, TQ, VARIANT>;
	const size_t smem = 16 + static_cast<size_t>(rows_per_cta) * NW * 4;
	if (smem > 48 * 1024)
	{
		LCD_CUDA(e, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
	}
	prof_mark(e, LCD_PROF_NN, s);
	kern<<<n_chunks, kNnThreads, smem, s>>>(e->vocab.p, n_rows, e->row_offset, d_q, nq_total, d_partial, rows_per_cta);
	prof_mark(e, LCD_PROF_NN, s);
	LCD_CHECK_LAUNCH(e);
	return LCD_OK;
}

template <int NW>
int launch_knn_nw(lcd_engine * e, const uint32_t * d_q, int nq_total, int n_rows, int n_chunks, int rows_per_cta,
                  uint2 * d_partial, cudaStream_t s)
{
	const int tq = e->nn_tq, var = (NW == 8) ? e->nn_variant : 0;
#define LCD_KNN_CASE(TQ_, V_) \
	if (tq == TQ_ && var == V_) return launch_knn_t<NW, TQ_, V_>(e, d_q, nq_total, n_rows, n_chunks, rows_per_cta, d_partial, s);
	LCD_KNN_CASE(4, 0)
	LCD_KNN_CASE(2, 0)
	LCD_KNN_CASE(8, 0)
	if constexpr (NW == 8)
	{
		LCD_KNN_CASE(4, 1)
		LCD_KNN_CASE(2, 1)
		LCD_KNN_CASE(8, 1)
		LCD_KNN_CASE(4, 2)
		LCD_KNN_CASE(2, 2)
		LCD_KNN_CASE(8, 2)
	}
#undef LCD_KNN_CASE
	return launch_knn_t<NW, 4, 0>(e, d_q, nq_total, n_rows, n_chunks, rows_per_cta, d_partial, s);
}

// ---- float descriptors on the tensor cores ------------------------------------------------------------------------
// rows of the vocabulary changed from `row` on (compaction, re-sorted tail): their image is stale
void tf_invalidate_from(lcd_engine * e, int row)
{
	e->tf_rows = std::min(e->tf_rows, std::max(row, 0));
	e->tc_rows = std::min(e->tc_rows, std::max(row, 0));
}

// (1) the cached word image: only rows that are new since the last search are converted.  When rows were converted, the "does not
// fit fp16" flag is read back at once (a synchronisation that only happens right after the dictionary changed): such a dictionary
// stays on the exact kernel.
template <int DIM>
int tf_prepare_words(lcd_engine * e, int n_rows, cudaStream_t s)
{
	if (e->tf_rows >= n_rows) return LCD_OK;
	const int n_tiles = (n_rows + kTfBN - 1) / kTfBN;
	const float * vocab = reinterpret_cast<const float *>(e->vocab.p);
	LCD_CUDA(e, e->tf_flags.reserve(4, 0, true, s));
	LCD_CUDA(e, e->tf_wmax2.reserve(1, 0, true, s));
	const size_t tile16 = static_cast<size_t>(kTfBN) * (DIM / 8);
	const int old_tiles = static_cast<int>(e->tf_words.cap / tile16);
	if (n_tiles > old_tiles)
	{
		const int want = std::max(n_tiles, old_tiles + old_tiles / 2 + 64);
		LCD_CUDA(e, e->tf_words.reserve(static_cast<size_t>(want) * tile16, static_cast<size_t>(e->tf_rows / kTfBN) * tile16, false, s));
		LCD_CUDA(e, e->tf_words_aug.reserve(static_cast<size_t>(want) * kTfBN * 2, static_cast<size_t>(e->tf_rows / kTfBN) * kTfBN * 2, false, s));
	}
	const int t0 = e->tf_rows / kTfBN;
	const size_t rows_todo = static_cast<size_t>(n_tiles - t0) * kTfBN, chunks = rows_todo * (DIM / 8);
	tf_expand_kernel<DIM><<<static_cast<unsigned>((chunks + 255) / 256), 256, 0, s>>>(vocab, t0 * kTfBN, n_rows, kTfBN, e->tf_words.p, e->tf_flags.p + 1, -2.0f);
	LCD_CHECK_LAUNCH(e);
	tf_aug_kernel<DIM><<<static_cast<unsigned>((rows_todo + 255) / 256), 256, 0, s>>>(vocab, t0 * kTfBN, n_rows, kTfBN, e->tf_words_aug.p, 0, e->tf_wmax2.p,
	                                                                                  e->tf_flags.p + 1);
	LCD_CHECK_LAUNCH(e);
	e->tf_img_builds += n_rows - e->tf_rows;
	e->tf_rows = n_rows;
	int bad = 0;
	LCD_CUDA(e, cudaMemcpyAsync(&bad, e->tf_flags.p + 1, sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	if (bad) e->tf_disabled = true;
	return LCD_OK;
}

template <int DIM>
int tf_search(lcd_engine * e, const float * d_q, int nq, int n_rows, cudaStream_t s)
{
	using Cfg = TfCfg<DIM>;
	const int n_tiles = (n_rows + kTfBN - 1) / kTfBN, n_qtiles = (nq + kTfBM - 1) / kTfBM;
	const float * vocab = reinterpret_cast<const float *>(e->vocab.p);
	// (2) per-call query image and per-query state
	const size_t qtile16 = static_cast<size_t>(kTfBM) * (DIM / 8);
	LCD_CUDA(e, e->tf_queries.reserve(static_cast<size_t>(n_qtiles) * qtile16, 0, false, s));
	LCD_CUDA(e, e->tf_qn.reserve(nq, 0, false, s));
	LCD_CUDA(e, e->tf_tau.reserve(nq, 0, false, s));
	LCD_CUDA(e, e->tf_cand_count.reserve(nq, 0, false, s));
	LCD_CUDA(e, e->tf_cand.reserve(static_cast<size_t>(nq) * kTfCandCap, 0, false, s));
	LCD_CUDA(e, e->tf_fb_list.reserve(nq, 0, false, s));
	LCD_CUDA(e, e->d_partial64.reserve(nq, 0, false, s));
	LCD_CUDA(e, zero_fill_async(e->tf_flags.p, sizeof(int), s)); // fallback count
	{
		const size_t chunks = static_cast<size_t>(n_qtiles) * kTfBM * (DIM / 8);
		tf_expand_kernel<DIM><<<static_cast<unsigned>((chunks + 255) / 256), 256, 0, s>>>(d_q, 0, nq, kTfBM, e->tf_queries.p, nullptr, 1.0f);
		LCD_CHECK_LAUNCH(e);
		LCD_CUDA(e, e->tf_queries_aug.reserve(static_cast<size_t>(n_qtiles) * kTfBM * 2, 0, false, s));
		tf_aug_kernel<DIM><<<(n_qtiles * kTfBM + 255) / 256, 256, 0, s>>>(d_q, 0, nq, kTfBM, e->tf_queries_aug.p, 1, nullptr, nullptr);
		LCD_CHECK_LAUNCH(e);
		tf_query_init_kernel<DIM><<<(nq + 255) / 256, 256, 0, s>>>(d_q, nq, e->tf_qn.p, e->tf_cand_count.p, e->tf_tau.p);
		LCD_CHECK_LAUNCH(e);
	}
	// (3) bound-only pre-pass over the first rows, then the emitting pass over all rows
	LCD_CUDA(e, cudaFuncSetAttribute(knn2_tensor_f32_kernel<DIM>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(Cfg::smem)));
	TfArgs a{};
	a.word_img = e->tf_words.p;
	a.word_aug = e->tf_words_aug.p;
	a.query_aug = e->tf_queries_aug.p;
	a.n_rows = n_rows;
	a.query_img = e->tf_queries.p;
	a.qn = e->tf_qn.p;
	a.nq = nq;
	a.wmax2_bits = e->tf_wmax2.p;
	a.tau = e->tf_tau.p;
	a.cand = e->tf_cand.p;
	a.cand_count = e->tf_cand_count.p;
	prof_mark(e, LCD_PROF_NN, s);
	a.tile_begin = 0;
	a.tile_end = std::min(n_tiles, kTfPrepassTiles);
	a.tiles_per_split = a.tile_end;
	a.emit = 0;
	knn2_tensor_f32_kernel<DIM><<<dim3(n_qtiles, 1), kTfThreads, Cfg::smem, s>>>(a);
	LCD_CHECK_LAUNCH(e);
	// splits: a split's slice of the word image should sit in L2 while the query tiles of that split stream it (CTAs with the same
	// blockIdx.y are scheduled together), and small query batches still have to fill the machine
	const int tiles_l2 = std::max(1, static_cast<int>((24u << 20) / Cfg::b_bytes));
	int splits = std::max((n_tiles + tiles_l2 - 1) / tiles_l2, (2 * e->sm_count + n_qtiles - 1) / n_qtiles);
	splits = std::max(1, std::min(splits, n_tiles));
	const int tps = (n_tiles + splits - 1) / splits;
	splits = (n_tiles + tps - 1) / tps;
	a.tile_begin = 0;
	a.tile_end = n_tiles;
	a.tiles_per_split = tps;
	a.emit = 1;
	knn2_tensor_f32_kernel<DIM><<<dim3(n_qtiles, splits), kTfThreads, Cfg::smem, s>>>(a);
	LCD_CHECK_LAUNCH(e);
	// (4) exact re-rank of the candidates; overflowed lists are redone by an exact scan
	rerank_l2_kernel<DIM><<<(nq + 7) / 8, 256, 0, s>>>(vocab, e->row_offset, d_q, nq, e->tf_cand.p, e->tf_cand_count.p, e->d_partial64.p, e->tf_fb_list.p,
	                                                   e->tf_flags.p);
	LCD_CHECK_LAUNCH(e);
	const int fb_slots = std::max(4 * nq, 1 << 18), fb_ctas = 2 * e->sm_count;
	LCD_CUDA(e, e->tf_fb_scratch.reserve(static_cast<size_t>(fb_slots), 0, false, s));
	LCD_CUDA(e, cudaFuncSetAttribute(knn2_l2_fallback_kernel<DIM>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(fallback_smem_bytes<DIM>())));
	knn2_l2_fallback_kernel<DIM><<<fb_ctas, 256, fallback_smem_bytes<DIM>(), s>>>(vocab, n_rows, e->row_offset, d_q, e->tf_fb_list.p, e->tf_flags.p,
	                                                                              e->tf_fb_scratch.p, fb_slots);
	LCD_CHECK_LAUNCH(e);
	knn2_l2_fallback_merge_kernel<<<64, 256, 0, s>>>(e->tf_fb_list.p, e->tf_flags.p, e->tf_fb_scratch.p, fb_slots, fb_ctas, e->d_partial64.p);
	prof_mark(e, LCD_PROF_NN, s);
	LCD_CHECK_LAUNCH(e);
	return LCD_OK;
}

// exact 2-NN of nq_total queries over rows [0,n_rows): fills e->d_partial, returns chunk count
int run_knn(lcd_engine * e, const uint32_t * d_q, int nq_total, int n_rows, int * n_chunks_out, cudaStream_t s)
{
	if (e->row_offset + n_rows > kMaxRowsPacked) LCD_FAIL(e, LCD_ERR_CAPACITY, "more than %d indexed words", kMaxRowsPacked);
	e->nn_last_tensor = 0;
	e->nn_last_f32_tensor = 0;
	if (e->f32 && e->nn_f32_tensor && !e->tf_disabled && n_rows >= kTfMinRows && nq_total > 0 &&
	    TfCfg<64>::smem <= static_cast<size_t>(e->smem_optin))
		LCD_TRY(e->nw == 64 ? tf_prepare_words<64>(e, n_rows, s) : tf_prepare_words<128>(e, n_rows, s));
	if (e->f32 && e->nn_f32_tensor && !e->tf_disabled && n_rows >= kTfMinRows && nq_total > 0 &&
	    TfCfg<64>::smem <= static_cast<size_t>(e->smem_optin))
	{
		// float descriptors, large dictionary: distance matrix on the tensor cores as a filter + exact re-rank (nn_tensor_f32.cuh)
		const float * q = reinterpret_cast<const float *>(d_q);
		e->nn_last_f32_tensor = 1;
		*n_chunks_out = 1;
		return e->nw == 64 ? tf_search<64>(e, q, nq_total, n_rows, s) : tf_search<128>(e, q, nq_total, n_rows, s);
	}
	if (e->f32)
	{
		// float descriptors: exact squared-L2 2-NN, one query per thread, rows split over blockIdx.y to fill the machine
		const int q_blocks = (nq_total + kL2Threads - 1) / kL2Threads;
		int splits = std::max(1, std::min((2 * e->sm_count + q_blocks - 1) / q_blocks, std::max(1, n_rows / (4 * kL2TileRows))));
		const int rps = std::max(1, (n_rows + splits - 1) / splits);
		splits = std::max(1, (n_rows + rps - 1) / rps);
		LCD_CUDA(e, e->d_partial64.reserve(static_cast<size_t>(splits) * nq_total, 0, false, s));
		const float * v = reinterpret_cast<const float *>(e->vocab.p);
		const float * q = reinterpret_cast<const float *>(d_q);
		prof_mark(e, LCD_PROF_NN, s);
		if (e->nw == 64) knn2_l2_kernel<64><<<dim3(q_blocks, splits), kL2Threads, 0, s>>>(v, n_rows, e->row_offset, q, nq_total, e->d_partial64.p, rps);
		else knn2_l2_kernel<128><<<dim3(q_blocks, splits), kL2Threads, 0, s>>>(v, n_rows, e->row_offset, q, nq_total, e->d_partial64.p, rps);
		prof_mark(e, LCD_PROF_NN, s);
		LCD_CHECK_LAUNCH(e);
		*n_chunks_out = splits;
		return LCD_OK;
	}
	if (e->nn_tensor && e->nw == 8 && n_rows > 0 && nq_total > 0 && kTcSmemBytes <= static_cast<size_t>(e->smem_optin))
	{
		// tensor-core path: expand both operands to the int8 images, then one CTA per (query tile, word split)
		const int n_wtiles = (n_rows + kTcBN - 1) / kTcBN, n_qtiles = (nq_total + kTcBM - 1) / kTcBM;
		int best_split = 1;
		long best_cost = -1;
		for (int sp = 1; sp <= std::min(n_wtiles, 16); ++sp)
		{
			const int tps = (n_wtiles + sp - 1) / sp;
			const int real_sp = (n_wtiles + tps - 1) / tps;
			if (real_sp != sp) continue;
			const long waves = (static_cast<long>(n_qtiles) * sp + e->sm_count - 1) / e->sm_count;
			const long cost = waves * (tps + 3); // +3: prologue (TMEM alloc, first loads) and drain, in tile times
			if (best_cost < 0 || cost < best_cost)
			{
				best_cost = cost;
				best_split = sp;
			}
		}
		const int tps = (n_wtiles + best_split - 1) / best_split;
		LCD_CUDA(e, e->d_partial.reserve(static_cast<size_t>(best_split) * kTcEpiGroups * nq_total, 0, false, s));
		static const int tc_recache = env_int("LCD_TC_RECACHE", 0); // experiment: rebuild the word image on every search (as r01 did)
		if (tc_recache) e->tc_rows = 0;
		if (e->tc_rows < n_rows)
		{
			// the +-1 byte image of the words is cached with the dictionary: only tiles that gained rows since the last search are written
			const int t0 = e->tc_rows / kTcBN;
			const size_t tile16 = static_cast<size_t>(kTcBN) * 16;
			const int old_tiles = static_cast<int>(e->tc_words.cap / tile16);
			if (n_wtiles > old_tiles)
				LCD_CUDA(e, e->tc_words.reserve(static_cast<size_t>(std::max(n_wtiles, old_tiles + old_tiles / 2 + 16)) * tile16, static_cast<size_t>(t0) * tile16, false, s));
			const size_t todo = static_cast<size_t>(n_wtiles - t0) * tile16;
			tc_expand_kernel<<<static_cast<unsigned>((todo + 255) / 256), 256, 0, s>>>(e->vocab.p, n_rows, kTcBN, t0, n_wtiles, e->tc_words.p);
			LCD_CHECK_LAUNCH(e);
			e->tc_rows = n_rows;
		}
		LCD_CUDA(e, cudaFuncSetAttribute(knn2_tensor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kTcSmemBytes)));
		prof_mark(e, LCD_PROF_NN, s);
		// A CTA walks several (query tile, word split) items with one TMEM allocation and a running pipeline (LCD_NN_PERSIST=0: one CTA
		// per item, as r01).  Unsharded: one CTA per SM takes them all.  Inside the sharded step the search runs beside NCCL kernels that
		// need a few SMs now and then: a grid that holds every SM until the end starves them and then waits for them (measured at 4 ranks:
		// 1.35 -> 1.48 ms), so there a CTA takes only enough items for ~96 word tiles and the grid stays several waves deep.
		static const int nn_persist = env_int("LCD_NN_PERSIST", 1);
		const int n_items = n_qtiles * best_split;
		int grid = n_items;
		if (nn_persist && e->comm)
		{
			const int per_cta = std::max(1, std::min(8, (96 + tps - 1) / std::max(tps, 1))); // items per CTA: 1 / 2 / 4 at 2 / 4 / 8 ranks of C2
			grid = (n_items + per_cta - 1) / per_cta;
		}
		else if (nn_persist)
			grid = std::min(n_items, e->sm_count);
		knn2_tensor_kernel<<<grid, kTcThreads, kTcSmemBytes, s>>>(e->tc_words.p, n_rows, e->row_offset, d_q, nq_total, e->d_partial.p, tps,
		                                                        static_cast<uint32_t>(-32), n_qtiles, best_split);
		prof_mark(e, LCD_PROF_NN, s);
		LCD_CHECK_LAUNCH(e);
		e->nn_last_tensor = 1;
		*n_chunks_out = best_split * kTcEpiGroups;
		return LCD_OK;
	}
	const int max_rows_smem = static_cast<int>((static_cast<size_t>(e->smem_optin) - 16 - 1024) / (e->nw * 4));
	int n_chunks = e->sm_count * e->nn_ctas_per_sm;
	n_chunks = std::min(n_chunks, std::max(1, (n_rows + 31) / 32));
	n_chunks = std::max(n_chunks, (n_rows + max_rows_smem - 1) / max_rows_smem);
	n_chunks = std::max(n_chunks, 1);
	int rows_per_cta = (n_rows + n_chunks - 1) / n_chunks;
	if (rows_per_cta < 1) rows_per_cta = 1;
	n_chunks = std::max(1, (n_rows + rows_per_cta - 1) / rows_per_cta);
	LCD_CUDA(e, e->d_partial.reserve(static_cast<size_t>(n_chunks) * nq_total, 0, false, s));
	int r;
	switch (e->nw)
	{
	case 4: r = launch_knn_nw<4>(e, d_q, nq_total, n_rows, n_chunks, rows_per_cta, e->d_partial.p, s); break;
	case 8: r = launch_knn_nw<8>(e, d_q, nq_total, n_rows, n_chunks, rows_per_cta, e->d_partial.p, s); break;
	case 16: r = launch_knn_nw<16>(e, d_q, nq_total, n_rows, n_chunks, rows_per_cta, e->d_partial.p, s); break;
	default: LCD_FAIL(e, LCD_ERR_INVALID, "unsupported descriptor size %d bytes", e->nw * 4);
	}
	*n_chunks_out = n_chunks;
	return r;
}

int launch_resolve(lcd_engine * e, const ResolveArgs & a, int n_frames, cudaStream_t s)
{
	if (e->f32)
	{
		const size_t smem32 = resolve_l2_smem_bytes(a.nq);
		if (smem32 > 48 * 1024)
		{
			if (e->nw == 64) LCD_CUDA(e, cudaFuncSetAttribute(resolve_l2_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem32)));
			else LCD_CUDA(e, cudaFuncSetAttribute(resolve_l2_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem32)));
		}
		prof_mark(e, LCD_PROF_RESOLVE, s);
		if (e->nw == 64) resolve_l2_kernel<64><<<n_frames, kL2ResolveThreads, smem32, s>>>(a, e->d_partial64.p);
		else resolve_l2_kernel<128><<<n_frames, kL2ResolveThreads, smem32, s>>>(a, e->d_partial64.p);
		prof_mark(e, LCD_PROF_RESOLVE, s);
		LCD_CHECK_LAUNCH(e);
		return LCD_OK;
	}
	const size_t smem = resolve_smem_bytes(a.nq);
#define LCD_RES_CASE(NW_)                                                                                               \
	case NW_:                                                                                                           \
	{                                                                                                                   \
		auto kern = resolve_kernel<NW_>;                                                                                \
		if (smem > 48 * 1024)                                                                                           \
			LCD_CUDA(e, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem))); \
		prof_mark(e, LCD_PROF_RESOLVE, s);                                                                              \
		kern<<<n_frames, kResolveThreads, smem, s>>>(a);                                                                \
		prof_mark(e, LCD_PROF_RESOLVE, s);                                                                              \
		break;                                                                                                          \
	}
	switch (e->nw)
	{
		LCD_RES_CASE(4)
		LCD_RES_CASE(8)
		LCD_RES_CASE(16)
	default: LCD_FAIL(e, LCD_ERR_INVALID, "unsupported descriptor size");
	}
#undef LCD_RES_CASE
	LCD_CHECK_LAUNCH(e);
	return LCD_OK;
}

int ensure_uq(lcd_engine * e, int n_frames, int nq, cudaStream_t s)
{
	LCD_CUDA(e, e->uq_count.reserve(n_frames, 0, false, s));
	LCD_CUDA(e, e->uq_word.reserve(static_cast<size_t>(n_frames) * nq, 0, false, s));
	LCD_CUDA(e, e->uq_prefix.reserve(static_cast<size_t>(n_frames) * (nq + 1), 0, false, s));
	LCD_CUDA(e, e->uq_idf.reserve(static_cast<size_t>(n_frames) * nq, 0, false, s));
	return LCD_OK;
}

void fill_prep(lcd_engine * e, ResolveArgs & a, float n_total, int self_ref)
{
	a.do_prep = 1;
	a.post_len = e->post_len.p;
	a.id_cap = static_cast<int>(e->h_len.size());
	a.n_total = n_total;
	a.self_ref = self_ref;
	a.uq_count = e->uq_count.p;
	a.uq_word = e->uq_word.p;
	a.uq_prefix = e->uq_prefix.p;
	a.uq_idf = e->uq_idf.p;
}

int launch_score(lcd_engine * e, int n_frames, int nq, cudaStream_t s)
{
	ScoreArgs sa;
	sa.nq = nq;
	sa.uq_count = e->uq_count.p;
	sa.uq_word = e->uq_word.p;
	sa.uq_prefix = e->uq_prefix.p;
	sa.uq_idf = e->uq_idf.p;
	sa.post_off = e->post_off.p;
	sa.postings = e->postings.p;
	sa.ni = e->ni.p;
	sa.sig_cap = static_cast<int>(e->h_ni.size());
	sa.acc = e->acc.p;
	sa.acc_stride = e->acc_stride;
	dim3 grid(e->score_blocks, n_frames);
	prof_mark(e, LCD_PROF_SCORE, s);
	score_kernel<<<grid, kScoreThreads, (nq + 1) * sizeof(int), s>>>(sa);
	prof_mark(e, LCD_PROF_SCORE, s);
	LCD_CHECK_LAUNCH(e);
	return LCD_OK;
}

// make the not-indexed tail ascending in id (std::set<int> _notIndexedWords iteration order)
int sort_pending(lcd_engine * e)
{
	if (e->pending_sorted || e->n_pending < 2)
	{
		e->pending_sorted = true;
		return LCD_OK;
	}
	const int base = e->n_indexed, n = e->n_pending;
	std::vector<int> order(n);
	for (int i = 0; i < n; ++i) order[i] = base + i;
	std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return e->h_row_ids[x] < e->h_row_ids[y]; });
	LCD_CUDA(e, e->d_perm.reserve(n, 0, false, e->stream));
	LCD_CUDA(e, cudaMemcpyAsync(e->d_perm.p, order.data(), n * sizeof(int), cudaMemcpyHostToDevice, e->stream));
	LCD_CUDA(e, e->vocab_alt.reserve(static_cast<size_t>(n) * e->nw, 0, false, e->stream));
	const size_t elems = static_cast<size_t>(n) * e->nw;
	gather_rows_kernel<<<static_cast<unsigned>((elems + 255) / 256), 256, 0, e->stream>>>(e->vocab.p, e->d_perm.p, n, e->nw, e->vocab_alt.p);
	LCD_CHECK_LAUNCH(e);
	LCD_CUDA(e, cudaMemcpyAsync(e->vocab.p + static_cast<size_t>(base) * e->nw, e->vocab_alt.p, elems * sizeof(uint32_t),
	                            cudaMemcpyDeviceToDevice, e->stream));
	std::vector<int> ids(n);
	for (int i = 0; i < n; ++i) ids[i] = e->h_row_ids[order[i]];
	for (int i = 0; i < n; ++i)
	{
		e->h_row_ids[base + i] = ids[i];
		e->id2row[ids[i]] = base + i;
	}
	LCD_CUDA(e, cudaMemcpyAsync(e->row_ids.p + base, ids.data(), n * sizeof(int), cudaMemcpyHostToDevice, e->stream));
	LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	e->pending_sorted = true;
	tf_invalidate_from(e, base);
	return LCD_OK;
}

// VWDictionary::addWordRef for the words of one signature (host bookkeeping + device ops)
int add_refs_impl(lcd_engine * e, int sig_id, const int * word_ids, int n)
{
	if (sig_id <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "signature id must be positive");
	LCD_TRY(ensure_sigs(e, sig_id));
	std::vector<int> ids;
	ids.reserve(n);
	for (int i = 0; i < n; ++i)
	{
		if (word_ids[i] > 0) ids.push_back(word_ids[i]);
	}
	std::sort(ids.begin(), ids.end());
	std::vector<RefOp> ops;
	std::vector<MoveOp> moves;
	auto & sw = e->sig_words[sig_id];
	std::vector<std::pair<int, int>> merged;
	merged.reserve(sw.size() + ids.size());
	size_t si = 0;
	size_t extra = 0;
	for (size_t i = 0; i < ids.size();)
	{
		size_t j = i;
		while (j < ids.size() && ids[j] == ids[i]) ++j;
		const int word = ids[i], cnt = static_cast<int>(j - i);
		i = j;
		if (e->id2row.find(word) == e->id2row.end())
		{
			// reference: UWARN("Not found word %d"), VWDictionary.cpp:893
			continue;
		}
		LCD_TRY(ensure_ids(e, word));
		while (si < sw.size() && sw[si].first < word) merged.push_back(sw[si++]);
		RefOp op{word, sig_id, cnt, -1, 0};
		if (si < sw.size() && sw[si].first == word)
		{
			merged.emplace_back(word, sw[si].second + cnt);
			++si;
			op.pos = -1;
			op.newlen = e->h_len[word];
		}
		else
		{
			merged.emplace_back(word, cnt);
			if (e->h_len[word] == e->h_cap[word])
			{
				const int ncap = std::max(4, e->h_cap[word] * 2);
				MoveOp mv{word, e->h_off[word], static_cast<uint32_t>(e->post_used + extra), e->h_len[word]};
				extra += ncap;
				e->h_off[word] = mv.new_off;
				e->h_cap[word] = ncap;
				moves.push_back(mv);
			}
			op.pos = e->h_len[word];
			op.newlen = ++e->h_len[word];
		}
		e->total_refs += cnt;
		ops.push_back(op);
	}
	while (si < sw.size()) merged.push_back(sw[si++]);
	sw.swap(merged);
	e->h_ni[sig_id] += n;
	LCD_CUDA(e, cudaMemcpyAsync(e->ni.p + sig_id, &e->h_ni[sig_id], sizeof(int), cudaMemcpyHostToDevice, e->stream));
	if (extra)
	{
		LCD_TRY(ensure_postings(e, extra));
		e->post_used += extra;
	}
	if (!moves.empty())
	{
		LCD_CUDA(e, e->d_moves.reserve(moves.size(), 0, false, e->stream));
		LCD_CUDA(e, cudaMemcpyAsync(e->d_moves.p, moves.data(), moves.size() * sizeof(MoveOp), cudaMemcpyHostToDevice, e->stream));
		const int nm = static_cast<int>(moves.size());
		index_move_kernel<<<(nm * 32 + 255) / 256, 256, 0, e->stream>>>(e->d_moves.p, nm, e->post_off.p, e->postings.p);
		LCD_CHECK_LAUNCH(e);
	}
	if (!ops.empty())
	{
		LCD_CUDA(e, e->d_ops.reserve(ops.size(), 0, false, e->stream));
		LCD_CUDA(e, cudaMemcpyAsync(e->d_ops.p, ops.data(), ops.size() * sizeof(RefOp), cudaMemcpyHostToDevice, e->stream));
		const int no = static_cast<int>(ops.size());
		index_apply_kernel<<<(no + 255) / 256, 256, 0, e->stream>>>(e->d_ops.p, no, e->post_off.p, e->post_len.p, e->postings.p);
		LCD_CHECK_LAUNCH(e);
	}
	// the op vectors are pageable: make sure the copies completed before they go out of scope
	LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	return LCD_OK;
}

int require_binary(lcd_engine * e, const char * what)
{
	if (e->f32) LCD_FAIL(e, LCD_ERR_INVALID, "%s works on binary descriptors only (this engine holds float descriptors)", what);
	return LCD_OK;
}

// entry points that translate local rows through e->row_ids are only valid on an unsharded engine
int require_unsharded(lcd_engine * e, const char * what)
{
	if (e->row_offset != 0)
		LCD_FAIL(e, LCD_ERR_STATE, "%s needs an unsharded engine (lcd_shard_set_row_offset(%d) is set: use the lcd_shard_* calls)", what, e->row_offset);
	return LCD_OK;
}

int check_queries(lcd_engine * e, const void * q, int nq)
{
	if (!q || nq <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "Descriptors size is null!");
	if (nq > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "at most %d descriptors per frame", kMaxFrameQueries);
	return LCD_OK;
}

// quantise + score of n_frames independent frames on device buffers, no mutation
int localize_dev(lcd_engine * e, const uint32_t * d_q, int n_frames, int nq, int incremental, float nndr, int cmp_new,
                 const int * d_sig_ids, int ns, int n_total, int * d_word_ids_out, float * d_like_out, cudaStream_t s,
                 const int * d_nq_frame = nullptr)
{
	if (e->n_indexed == 0 && !incremental) LCD_FAIL(e, LCD_ERR_STATE, "Dictionary mode is set to fixed but no words are in it!");
	LCD_TRY(require_unsharded(e, "localisation on one engine"));
	const int nq_total = n_frames * nq;
	int n_chunks = 0;
	LCD_TRY(run_knn(e, d_q, nq_total, e->n_indexed, &n_chunks, s));
	const bool score = d_like_out != nullptr && ns > 0;
	ResolveArgs a{};
	a.queries = d_q;
	a.nq = nq;
	a.nq_frame = d_nq_frame;
	a.nq_total = nq_total;
	a.partial = e->d_partial.p;
	a.n_chunks = n_chunks;
	a.row_ids = e->row_ids.p;
	a.incremental = incremental;
	a.nndr = nndr;
	a.cmp_new = cmp_new;
	a.last_word_id = e->last_word_id;
	a.word_ids_out = d_word_ids_out;
	a.n_new_out = nullptr;
	a.pending_desc = nullptr;
	a.pending_ids = nullptr;
	if (score)
	{
		LCD_TRY(ensure_uq(e, n_frames, nq, s));
		LCD_TRY(ensure_acc(e, n_frames));
		LCD_CUDA(e, zero_fill_async(e->acc.p, static_cast<size_t>(e->acc_stride) * n_frames * sizeof(long long), s));
		fill_prep(e, a, static_cast<float>(n_total), 1);
	}
	LCD_TRY(launch_resolve(e, a, n_frames, s));
	if (score)
	{
		LCD_TRY(launch_score(e, n_frames, nq, s));
		dim3 grid((ns + 255) / 256, n_frames);
		gather_likelihood_kernel<<<grid, 256, 0, s>>>(e->acc.p, e->acc_stride, static_cast<int>(e->h_ni.size()), d_sig_ids, ns, d_like_out);
		LCD_CHECK_LAUNCH(e);
	}
	return LCD_OK;
}

} // namespace

// ============================================================================ C ABI ====
extern "C" {

int lcd_abi_version(void) { return 2; }
const char * lcd_build_arch(void) { return "sm_100a"; }

const char * lcd_last_error(const lcd_engine * e) { return e ? e->err.c_str() : g_create_error.c_str(); }
long long lcd_launch_count(const lcd_engine * e) { return e ? e->launches.load() : 0; }

int lcd_nn_select(lcd_engine * e, int kernel)
{
	if (!e) return LCD_ERR_INVALID;
	if (kernel != 0 && kernel != 1) LCD_FAIL(e, LCD_ERR_INVALID, "kernel must be 0 (popcount / exact L2 on the CUDA cores) or 1 (tensor)");
	if (e->f32) e->nn_f32_tensor = kernel;
	else e->nn_tensor = kernel;
	return LCD_OK;
}

int lcd_nn_f32_stats(lcd_engine * e, int nq, int * n_fallback, long long * n_candidates, long long * rows_converted)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (n_fallback) *n_fallback = 0;
	if (n_candidates) *n_candidates = 0;
	if (rows_converted) *rows_converted = e->tf_img_builds;
	if (!e->f32 || !e->tf_flags.p || !e->tf_cand_count.p || nq <= 0) return LCD_OK;
	LCD_CUDA(e, cudaDeviceSynchronize());
	int fb = 0;
	LCD_CUDA(e, cudaMemcpy(&fb, e->tf_flags.p, sizeof(int), cudaMemcpyDeviceToHost));
	std::vector<int> cnt(std::min<size_t>(nq, e->tf_cand_count.cap));
	LCD_CUDA(e, cudaMemcpy(cnt.data(), e->tf_cand_count.p, cnt.size() * sizeof(int), cudaMemcpyDeviceToHost));
	long long tot = 0;
	for (int c : cnt) tot += std::min(c, kTfCandCap);
	if (n_fallback) *n_fallback = fb;
	if (n_candidates) *n_candidates = tot;
	return LCD_OK;
}

int lcd_nn_last_kernel(const lcd_engine * e) { return e ? (e->f32 ? e->nn_last_f32_tensor : e->nn_last_tensor) : LCD_ERR_INVALID; }
void * lcd_stream(lcd_engine * e) { return e ? static_cast<void *>(e->stream) : nullptr; }

lcd_engine * lcd_create(const lcd_config * cfg)
{
	if (!cfg)
	{
		g_create_error = "null config";
		return nullptr;
	}
	if (cfg->desc_type != LCD_DESC_U8 && cfg->desc_type != LCD_DESC_F32)
	{
		g_create_error = "desc_type must be LCD_DESC_U8 (binary, Hamming) or LCD_DESC_F32 (float, squared L2)";
		return nullptr;
	}
	if (cfg->desc_type == LCD_DESC_U8 && cfg->desc_dim != 16 && cfg->desc_dim != 32 && cfg->desc_dim != 64)
	{
		g_create_error = "binary descriptor size must be 16, 32 or 64 bytes";
		return nullptr;
	}
	if (cfg->desc_type == LCD_DESC_F32 && cfg->desc_dim != 64 && cfg->desc_dim != 128)
	{
		g_create_error = "float descriptors must have 64 or 128 dimensions (SURF-64, SURF-128 / SIFT)";
		return nullptr;
	}
	int ndev = 0;
	cudaError_t err = cudaGetDeviceCount(&ndev);
	if (err != cudaSuccess || ndev <= cfg->device || cfg->device < 0)
	{
		g_create_error = std::string("no usable CUDA device: ") + (err != cudaSuccess ? cudaGetErrorString(err) : "device ordinal out of range");
		return nullptr;
	}
	lcd_engine * e = new lcd_engine();
	e->cfg = *cfg;
	e->f32 = cfg->desc_type == LCD_DESC_F32;
	e->nw = e->f32 ? cfg->desc_dim : cfg->desc_dim / 4; // 32-bit words per descriptor row
	if ((err = cudaSetDevice(cfg->device)) != cudaSuccess || (err = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking)) != cudaSuccess ||
	    (err = cudaStreamCreateWithFlags(&e->orb_stream, cudaStreamNonBlocking)) != cudaSuccess)
	{
		g_create_error = std::string("CUDA init failed: ") + cudaGetErrorString(err);
		delete e;
		return nullptr;
	}
	cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, cfg->device);
	cudaDeviceGetAttribute(&e->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, cfg->device);
	e->nn_ctas_per_sm = std::max(1, env_int("LCD_NN_CTAS_PER_SM", e->nn_ctas_per_sm));
	e->nn_tq = env_int("LCD_NN_TQ", e->nn_tq);
	e->nn_variant = env_int("LCD_NN_VARIANT", e->nn_variant);
	e->nn_tensor = env_int("LCD_NN_TENSOR", e->nn_tensor);
	e->nn_f32_tensor = env_int("LCD_NN_F32_TENSOR", e->nn_f32_tensor);
	e->score_blocks = std::max(1, env_int("LCD_SCORE_BLOCKS", e->score_blocks));
	if (ensure_rows(e, std::max(cfg->max_words, 1024)) != LCD_OK || ensure_ids(e, std::max(cfg->max_words, 1024)) != LCD_OK ||
	    ensure_sigs(e, std::max(cfg->max_signatures, 1024)) != LCD_OK)
	{
		g_create_error = e->err;
		lcd_destroy(e);
		return nullptr;
	}
	return e;
}

void lcd_destroy(lcd_engine * e)
{
	if (!e) return;
	cudaSetDevice(e->cfg.device);
	if (e->stream)
	{
		cudaStreamSynchronize(e->stream);
		for (auto & ms : e->map_slots)
			if (ms.done) cudaEventDestroy(ms.done);
		if (e->comm && e->comm_owned && nccl_api().ok) nccl_api().CommDestroy(e->comm);
		if (e->comm_stream) cudaStreamDestroy(e->comm_stream);
		for (auto & half : e->sh_ev)
			for (cudaEvent_t ev : half)
				if (ev) cudaEventDestroy(ev);
		for (cudaEvent_t ev : e->sh_tr)
			if (ev) cudaEventDestroy(ev);
		for (cudaEvent_t ev : e->sh_ring)
			if (ev) cudaEventDestroy(ev);
		if (e->orb_stream)
		{
			cudaStreamSynchronize(e->orb_stream);
			cudaStreamDestroy(e->orb_stream);
		}
		if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
		for (cudaEvent_t ev : e->copy_events) cudaEventDestroy(ev);
		if (e->copy_fence) cudaEventDestroy(e->copy_fence);
		for (int i = 0; i < 4; ++i)
		{
			if (e->aux_stream[i]) cudaStreamDestroy(e->aux_stream[i]);
			if (e->aux_join[i]) cudaEventDestroy(e->aux_join[i]);
		}
		if (e->aux_fork) cudaEventDestroy(e->aux_fork);
		if (e->aux_blur_done) cudaEventDestroy(e->aux_blur_done);
		for (auto & f : e->flights)
		{
			if (f.uploaded) cudaEventDestroy(f.uploaded);
			if (f.done) cudaEventDestroy(f.done);
		}
		cudaStreamDestroy(e->stream);
	}
	for (auto & p : e->prof)
		for (auto ev : p.ev) cudaEventDestroy(ev);
	delete e;
}

int lcd_profile_enable(lcd_engine * e, int on)
{
	if (!e) return LCD_ERR_INVALID;
	e->prof_on = on != 0;
	return LCD_OK;
}

int lcd_profile_reset(lcd_engine * e)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	LCD_CUDA(e, cudaDeviceSynchronize());
	for (auto & p : e->prof) p.used = 0;
	return LCD_OK;
}

int lcd_profile_read(lcd_engine * e, int which, double * total_ms, long long * launches)
{
	if (!e || which < 0 || which > 5) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	LCD_CUDA(e, cudaDeviceSynchronize());
	auto & p = e->prof[which];
	double tot = 0.0;
	for (size_t i = 0; i + 1 < p.used; i += 2)
	{
		float ms = 0.f;
		LCD_CUDA(e, cudaEventElapsedTime(&ms, p.ev[i], p.ev[i + 1]));
		tot += ms;
	}
	if (total_ms) *total_ms = tot;
	if (launches) *launches = static_cast<long long>(p.used / 2);
	return LCD_OK;
}

int lcd_synchronize(lcd_engine * e)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	return LCD_OK;
}

// ---- dictionary ---------------------------------------------------------------------------
int lcd_dict_add_words(lcd_engine * e, const int * ids, const void * desc, int n)
{
	if (!e) return LCD_ERR_INVALID;
	if (n <= 0) return LCD_OK;
	if (!ids || !desc) LCD_FAIL(e, LCD_ERR_INVALID, "null ids/descriptors");
	LCD_TRY(set_device(e));
	int max_id = 0;
	for (int i = 0; i < n; ++i)
	{
		if (ids[i] <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "word ids must be positive (got %d)", ids[i]);
		if (e->id2row.count(ids[i])) LCD_FAIL(e, LCD_ERR_INVALID, "word %d already in the dictionary", ids[i]);
		max_id = std::max(max_id, ids[i]);
	}
	const int base = total_rows(e);
	LCD_TRY(ensure_rows(e, base + n));
	LCD_TRY(ensure_ids(e, max_id));
	LCD_CUDA(e, cudaMemcpyAsync(e->vocab.p + static_cast<size_t>(base) * e->nw, desc, static_cast<size_t>(n) * e->nw * 4, cudaMemcpyHostToDevice, e->stream));
	LCD_CUDA(e, cudaMemcpyAsync(e->row_ids.p + base, ids, static_cast<size_t>(n) * sizeof(int), cudaMemcpyHostToDevice, e->stream));
	LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	for (int i = 0; i < n; ++i)
	{
		if (!e->h_row_ids.empty() && e->n_pending + i > 0 && ids[i] < e->h_row_ids.back()) e->pending_sorted = false;
		e->h_row_ids.push_back(ids[i]);
		e->id2row[ids[i]] = base + i;
	}
	e->n_pending += n;
	// the reference does not touch _lastWordId in addWord; the caller sets it (Memory.cpp:431)
	return LCD_OK;
}

int lcd_dict_remove_words(lcd_engine * e, const int * ids, int n)
{
	if (!e) return LCD_ERR_INVALID;
	if (n <= 0) return LCD_OK;
	LCD_TRY(set_device(e));
	bool pending_hit = false;
	std::vector<int> zero_ids;
	for (int i = 0; i < n; ++i)
	{
		auto it = e->id2row.find(ids[i]);
		if (it == e->id2row.end()) continue;
		const int row = it->second;
		if (row < e->n_indexed) e->removed_rows.insert(row);
		else pending_hit = true;
		e->id2row.erase(it);
		if (ids[i] < static_cast<int>(e->h_len.size()) && e->h_len[ids[i]] > 0)
		{
			// The reference only removes unused words (VWDictionary::deleteUnusedWords, VWDictionary.cpp:1595-1607); a word that still
			// has references takes them with it here: its posting list is read back once so that the per-signature word lists and
			// the reference total stay consistent with the device (a later lcd_index_remove_sig must not count them again).
			const int len = e->h_len[ids[i]];
			std::vector<int2> post(len);
			LCD_CUDA(e, cudaMemcpyAsync(post.data(), e->postings.p + e->h_off[ids[i]], len * sizeof(int2), cudaMemcpyDeviceToHost, e->stream));
			LCD_CUDA(e, cudaStreamSynchronize(e->stream));
			for (const int2 & pc : post)
			{
				e->total_refs -= pc.y;
				auto sw = e->sig_words.find(pc.x);
				if (sw == e->sig_words.end()) continue;
				auto & v = sw->second;
				auto pos = std::lower_bound(v.begin(), v.end(), std::make_pair(ids[i], 0));
				if (pos != v.end() && pos->first == ids[i]) v.erase(pos);
			}
			e->h_len[ids[i]] = 0;
			zero_ids.push_back(ids[i]);
		}
	}
	for (int id : zero_ids)
	{
		LCD_CUDA(e, cudaMemsetAsync(e->post_len.p + id, 0, sizeof(int), e->stream));
	}
	if (pending_hit)
	{
		// compact the not-indexed tail on the spot (it is small)
		const int base = e->n_indexed, np = e->n_pending;
		std::vector<int> keep;
		for (int r = base; r < base + np; ++r)
		{
			auto it = e->id2row.find(e->h_row_ids[r]);
			if (it != e->id2row.end() && it->second == r) keep.push_back(r);
		}
		const int nk = static_cast<int>(keep.size());
		if (nk)
		{
			LCD_CUDA(e, e->d_perm.reserve(nk, 0, false, e->stream));
			LCD_CUDA(e, cudaMemcpyAsync(e->d_perm.p, keep.data(), nk * sizeof(int), cudaMemcpyHostToDevice, e->stream));
			LCD_CUDA(e, e->vocab_alt.reserve(static_cast<size_t>(nk) * e->nw, 0, false, e->stream));
			const size_t elems = static_cast<size_t>(nk) * e->nw;
			gather_rows_kernel<<<static_cast<unsigned>((elems + 255) / 256), 256, 0, e->stream>>>(e->vocab.p, e->d_perm.p, nk, e->nw, e->vocab_alt.p);
			LCD_CHECK_LAUNCH(e);
			LCD_CUDA(e, cudaMemcpyAsync(e->vocab.p + static_cast<size_t>(base) * e->nw, e->vocab_alt.p, elems * 4, cudaMemcpyDeviceToDevice, e->stream));
		}
		std::vector<int> kid(nk);
		for (int i = 0; i < nk; ++i) kid[i] = e->h_row_ids[keep[i]];
		e->h_row_ids.resize(base);
		for (int i = 0; i < nk; ++i)
		{
			e->h_row_ids.push_back(kid[i]);
			e->id2row[kid[i]] = base + i;
		}
		if (nk) LCD_CUDA(e, cudaMemcpyAsync(e->row_ids.p + base, kid.data(), nk * sizeof(int), cudaMemcpyHostToDevice, e->stream));
		e->n_pending = nk;
		tf_invalidate_from(e, base);
	}
	LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	return LCD_OK;
}

int lcd_dict_update(lcd_engine * e)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	LCD_TRY(sort_pending(e));
	if (!e->removed_rows.empty())
	{
		const int tot = total_rows(e);
		std::vector<int> keep;
		keep.reserve(tot);
		int kept_indexed = 0;
		for (int r = 0; r < tot; ++r)
		{
			if (r < e->n_indexed && e->removed_rows.count(r)) continue;
			keep.push_back(r);
			if (r < e->n_indexed) ++kept_indexed;
		}
		const int nk = static_cast<int>(keep.size());
		LCD_CUDA(e, e->vocab_alt.reserve(std::max<size_t>(e->vocab.cap, 1), 0, false, e->stream));
		LCD_CUDA(e, e->row_ids_alt.reserve(std::max<size_t>(e->row_ids.cap, 1), 0, false, e->stream));
		std::vector<int> kid(nk);
		for (int i = 0; i < nk; ++i) kid[i] = e->h_row_ids[keep[i]];
		if (nk)
		{
			LCD_CUDA(e, e->d_perm.reserve(nk, 0, false, e->stream));
			LCD_CUDA(e, cudaMemcpyAsync(e->d_perm.p, keep.data(), nk * sizeof(int), cudaMemcpyHostToDevice, e->stream));
			const size_t elems = static_cast<size_t>(nk) * e->nw;
			gather_rows_kernel<<<static_cast<unsigned>((elems + 255) / 256), 256, 0, e->stream>>>(e->vocab.p, e->d_perm.p, nk, e->nw, e->vocab_alt.p);
			LCD_CHECK_LAUNCH(e);
			LCD_CUDA(e, cudaMemcpyAsync(e->row_ids_alt.p, kid.data(), nk * sizeof(int), cudaMemcpyHostToDevice, e->stream));
		}
		LCD_CUDA(e, cudaStreamSynchronize(e->stream));
		std::swap(e->vocab.p, e->vocab_alt.p);
		std::swap(e->vocab.cap, e->vocab_alt.cap);
		std::swap(e->row_ids.p, e->row_ids_alt.p);
		std::swap(e->row_ids.cap, e->row_ids_alt.cap);
		e->h_row_ids.swap(kid);
		e->id2row.clear();
		for (int i = 0; i < nk; ++i) e->id2row[e->h_row_ids[i]] = i;
		e->n_pending = nk - kept_indexed;
		e->n_indexed = kept_indexed;
		e->removed_rows.clear();
		tf_invalidate_from(e, 0); // rows moved: the fp16 image is rebuilt at the next search
	}
	e->n_indexed += e->n_pending;
	e->n_pending = 0;
	e->pending_sorted = true;
	return LCD_OK;
}

int lcd_dict_clear(lcd_engine * e)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	e->h_row_ids.clear();
	e->id2row.clear();
	e->removed_rows.clear();
	e->n_indexed = e->n_pending = 0;
	e->pending_sorted = true;
	e->last_word_id = 0;
	std::fill(e->h_off.begin(), e->h_off.end(), 0u);
	std::fill(e->h_len.begin(), e->h_len.end(), 0);
	std::fill(e->h_cap.begin(), e->h_cap.end(), 0);
	std::fill(e->h_ni.begin(), e->h_ni.end(), 0);
	if (e->post_len.p) LCD_CUDA(e, cudaMemsetAsync(e->post_len.p, 0, e->post_len.cap * sizeof(int), e->stream));
	if (e->post_off.p) LCD_CUDA(e, cudaMemsetAsync(e->post_off.p, 0, e->post_off.cap * sizeof(uint32_t), e->stream));
	if (e->ni.p) LCD_CUDA(e, cudaMemsetAsync(e->ni.p, 0, e->ni.cap * sizeof(int), e->stream));
	e->post_used = 0;
	e->sig_words.clear();
	e->total_refs = 0;
	e->tf_rows = 0;
	e->tc_rows = 0;
	e->tf_disabled = false;
	if (e->tf_wmax2.p) LCD_CUDA(e, cudaMemsetAsync(e->tf_wmax2.p, 0, sizeof(uint32_t), e->stream));
	if (e->tf_flags.p) LCD_CUDA(e, cudaMemsetAsync(e->tf_flags.p, 0, 4 * sizeof(int), e->stream));
	LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	return LCD_OK;
}

int lcd_dict_size(const lcd_engine * e) { return e ? static_cast<int>(e->id2row.size()) : 0; }
int lcd_dict_indexed_size(const lcd_engine * e) { return e ? e->n_indexed : 0; }
int lcd_dict_not_indexed_size(const lcd_engine * e) { return e ? e->n_pending : 0; }
int lcd_dict_last_word_id(const lcd_engine * e) { return e ? e->last_word_id : 0; }
int lcd_dict_set_last_word_id(lcd_engine * e, int id)
{
	if (!e || id < 0) return LCD_ERR_INVALID;
	e->last_word_id = id;
	return LCD_OK;
}

int lcd_dict_has_word(const lcd_engine * e, int word_id) { return e && e->id2row.count(word_id) ? 1 : 0; }

int lcd_dict_get_indexed(lcd_engine * e, int * ids, void * desc, int cap_rows)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	const int n = std::min(cap_rows, e->n_indexed);
	if (n <= 0) return 0;
	if (ids) memcpy(ids, e->h_row_ids.data(), n * sizeof(int));
	if (desc)
	{
		LCD_CUDA(e, cudaMemcpyAsync(desc, e->vocab.p, static_cast<size_t>(n) * e->nw * 4, cudaMemcpyDeviceToHost, e->stream));
		LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	}
	return n;
}

int lcd_dict_knn2(lcd_engine * e, const void * queries, int nq, int * id1, float * d1, int * id2, float * d2)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!queries || nq <= 0 || !id1 || !d1 || !id2 || !d2) LCD_FAIL(e, LCD_ERR_INVALID, "null argument");
	LCD_TRY(require_unsharded(e, "lcd_dict_knn2"));
	cudaStream_t s = e->stream;
	LCD_CUDA(e, e->d_queries.reserve(static_cast<size_t>(nq) * e->nw, 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->d_queries.p, queries, static_cast<size_t>(nq) * e->nw * 4, cudaMemcpyHostToDevice, s));
	int n_chunks = 0;
	LCD_TRY(run_knn(e, e->d_queries.p, nq, e->n_indexed, &n_chunks, s));
	LCD_CUDA(e, e->d_i1.reserve(nq, 0, false, s));
	LCD_CUDA(e, e->d_i2.reserve(nq, 0, false, s));
	LCD_CUDA(e, e->d_f1.reserve(nq, 0, false, s));
	LCD_CUDA(e, e->d_f2.reserve(nq, 0, false, s));
	if (e->f32)
	{
		knn2_l2_decode_kernel<<<(nq + 255) / 256, 256, 0, s>>>(e->d_partial64.p, n_chunks, nq, e->row_ids.p, e->d_i1.p, e->d_f1.p, e->d_i2.p, e->d_f2.p);
		LCD_CHECK_LAUNCH(e);
	}
	else
	{
		LCD_CUDA(e, e->d_keys.reserve(2 * static_cast<size_t>(nq), 0, false, s));
		knn2_merge_kernel<<<(nq + 255) / 256, 256, 0, s>>>(e->d_partial.p, n_chunks, nq, e->d_keys.p);
		LCD_CHECK_LAUNCH(e);
		knn2_decode_kernel<<<(nq + 255) / 256, 256, 0, s>>>(e->d_keys.p, nq, e->row_ids.p, e->d_i1.p, e->d_f1.p, e->d_i2.p, e->d_f2.p);
		LCD_CHECK_LAUNCH(e);
	}
	LCD_CUDA(e, cudaMemcpyAsync(id1, e->d_i1.p, nq * sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaMemcpyAsync(id2, e->d_i2.p, nq * sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaMemcpyAsync(d1, e->d_f1.p, nq * sizeof(float), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaMemcpyAsync(d2, e->d_f2.p, nq * sizeof(float), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	return LCD_OK;
}

} // extern "C"

// VWDictionary::addNewWords on descriptors that are already on the device: d_q holds `rows` descriptor rows of which the first
// n_valid (host value, or the device counter d_n_valid when n_valid < 0) are real.  Word ids of all rows -> word_ids_out (host),
// *n_new_out = words created, *n_valid_out = the device counter's value.
static int quantize_dev(lcd_engine * e, const uint32_t * d_q, int rows, int n_valid, const int * d_n_valid, int sig_id, int incremental, float nndr,
                        int cmp_new, int * word_ids_out, int * n_new_out, int * n_valid_out, cudaStream_t s)
{
	if (!incremental && e->id2row.empty()) LCD_FAIL(e, LCD_ERR_STATE, "Dictionary mode is set to fixed but no words are in it!");
	LCD_TRY(require_unsharded(e, "lcd_dict_quantize"));
	const int rows0 = total_rows(e);
	LCD_TRY(ensure_rows(e, rows0 + rows));
	int n_chunks = 0;
	LCD_TRY(run_knn(e, d_q, rows, e->n_indexed, &n_chunks, s));
	LCD_CUDA(e, e->d_word_ids.reserve(rows, 0, false, s));
	LCD_CUDA(e, e->d_n_new.reserve(1, 0, false, s));
	ResolveArgs a{};
	a.queries = d_q;
	a.nq = rows;
	a.nq_total = rows;
	a.nq_frame = n_valid < 0 ? d_n_valid : nullptr;
	a.partial = e->d_partial.p;
	a.n_chunks = n_chunks;
	a.row_ids = e->row_ids.p;
	a.incremental = incremental;
	a.nndr = nndr;
	a.cmp_new = cmp_new;
	a.last_word_id = e->last_word_id;
	a.word_ids_out = e->d_word_ids.p;
	a.n_new_out = e->d_n_new.p;
	a.pending_desc = e->vocab.p + static_cast<size_t>(rows0) * e->nw;
	a.pending_ids = e->row_ids.p + rows0;
	a.do_prep = 0;
	LCD_TRY(launch_resolve(e, a, 1, s));
	int n_new = 0, nv = n_valid;
	LCD_CUDA(e, cudaMemcpyAsync(word_ids_out, e->d_word_ids.p, rows * sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaMemcpyAsync(&n_new, e->d_n_new.p, sizeof(int), cudaMemcpyDeviceToHost, s));
	if (n_valid < 0) LCD_CUDA(e, cudaMemcpyAsync(&nv, d_n_valid, sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	if (n_new > 0)
	{
		LCD_TRY(ensure_ids(e, e->last_word_id + n_new));
		for (int k = 0; k < n_new; ++k)
		{
			const int id = e->last_word_id + 1 + k;
			e->h_row_ids.push_back(id);
			e->id2row[id] = rows0 + k;
		}
		e->n_pending += n_new;
		e->last_word_id += n_new;
	}
	if (n_new_out) *n_new_out = n_new;
	if (n_valid_out) *n_valid_out = nv;
	if (sig_id > 0) LCD_TRY(add_refs_impl(e, sig_id, word_ids_out, std::min(std::max(nv, 0), rows)));
	return LCD_OK;
}

extern "C" {

int lcd_dict_quantize(lcd_engine * e, const void * queries, int nq, int sig_id, int incremental, float nndr,
                      int new_words_compared_together, int * word_ids_out, int * n_new_out)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	LCD_TRY(check_queries(e, queries, nq));
	if (!word_ids_out) LCD_FAIL(e, LCD_ERR_INVALID, "null output");
	cudaStream_t s = e->stream;
	LCD_CUDA(e, e->d_queries.reserve(static_cast<size_t>(nq) * e->nw, 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->d_queries.p, queries, static_cast<size_t>(nq) * e->nw * 4, cudaMemcpyHostToDevice, s));
	return quantize_dev(e, e->d_queries.p, nq, nq, nullptr, sig_id, incremental, nndr, new_words_compared_together, word_ids_out, n_new_out, nullptr, s);
}

int lcd_dict_find_nn(lcd_engine * e, const void * queries, int nq, int incremental, float nndr, int * word_ids_out)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	LCD_TRY(check_queries(e, queries, nq));
	if (!word_ids_out) LCD_FAIL(e, LCD_ERR_INVALID, "null output");
	if (e->id2row.empty())
	{
		memset(word_ids_out, 0, nq * sizeof(int));
		return LCD_OK;
	}
	LCD_TRY(require_unsharded(e, "lcd_dict_find_nn"));
	LCD_TRY(sort_pending(e));
	cudaStream_t s = e->stream;
	LCD_CUDA(e, e->d_queries.reserve(static_cast<size_t>(nq) * e->nw, 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->d_queries.p, queries, static_cast<size_t>(nq) * e->nw * 4, cudaMemcpyHostToDevice, s));
	int n_chunks = 0;
	// index rows first, then the not-indexed tail: (dist,row) order = index hits before
	// not-indexed hits at equal distance, as the multimap insertion order (VWDictionary.cpp:1476-1517)
	LCD_TRY(run_knn(e, e->d_queries.p, nq, total_rows(e), &n_chunks, s));
	LCD_CUDA(e, e->d_word_ids.reserve(nq, 0, false, s));
	LCD_CUDA(e, e->d_n_new.reserve(1, 0, false, s));
	ResolveArgs a{};
	a.queries = e->d_queries.p;
	a.nq = nq;
	a.nq_total = nq;
	a.partial = e->d_partial.p;
	a.n_chunks = n_chunks;
	a.row_ids = e->row_ids.p;
	a.incremental = incremental;
	a.nndr = nndr;
	a.cmp_new = 0;
	a.last_word_id = e->last_word_id;
	a.find_only = 1;
	a.word_ids_out = e->d_word_ids.p;
	a.n_new_out = e->d_n_new.p;
	LCD_TRY(launch_resolve(e, a, 1, s));
	LCD_CUDA(e, cudaMemcpyAsync(word_ids_out, e->d_word_ids.p, nq * sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	return LCD_OK;
}

// ---- inverted index ---------------------------------------------------------------------
int lcd_index_add_refs(lcd_engine * e, int sig_id, const int * word_ids, int n)
{
	if (!e) return LCD_ERR_INVALID;
	if (n < 0 || (n > 0 && !word_ids)) LCD_FAIL(e, LCD_ERR_INVALID, "bad word list");
	LCD_TRY(set_device(e));
	return add_refs_impl(e, sig_id, word_ids, n);
}

int lcd_index_remove_sig(lcd_engine * e, int sig_id)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	auto it = e->sig_words.find(sig_id);
	if (it == e->sig_words.end()) return LCD_OK;
	std::vector<RefOp> ops;
	for (auto & wc : it->second)
	{
		const int word = wc.first;
		if (e->id2row.find(word) == e->id2row.end() || e->h_len[word] == 0) continue;
		ops.push_back(RefOp{word, sig_id, wc.second, -1, 0});
		--e->h_len[word];
		e->total_refs -= wc.second;
	}
	e->sig_words.erase(it);
	if (sig_id < static_cast<int>(e->h_ni.size()))
	{
		e->h_ni[sig_id] = 0;
		LCD_CUDA(e, cudaMemsetAsync(e->ni.p + sig_id, 0, sizeof(int), e->stream));
	}
	if (!ops.empty())
	{
		const int no = static_cast<int>(ops.size());
		LCD_CUDA(e, e->d_ops.reserve(no, 0, false, e->stream));
		LCD_CUDA(e, cudaMemcpyAsync(e->d_ops.p, ops.data(), no * sizeof(RefOp), cudaMemcpyHostToDevice, e->stream));
		index_remove_kernel<<<(no * 32 + 255) / 256, 256, 0, e->stream>>>(e->d_ops.p, no, e->post_off.p, e->post_len.p, e->postings.p);
		LCD_CHECK_LAUNCH(e);
	}
	LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	return LCD_OK;
}

int lcd_index_set_ni(lcd_engine * e, const int * sig_ids, const int * ni, int n)
{
	if (!e) return LCD_ERR_INVALID;
	if (n <= 0) return LCD_OK;
	LCD_TRY(set_device(e));
	int mx = 0;
	for (int i = 0; i < n; ++i)
	{
		if (sig_ids[i] <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "signature id must be positive");
		mx = std::max(mx, sig_ids[i]);
	}
	LCD_TRY(ensure_sigs(e, mx));
	for (int i = 0; i < n; ++i) e->h_ni[sig_ids[i]] = ni[i];
	LCD_CUDA(e, cudaMemcpyAsync(e->ni.p, e->h_ni.data(), (static_cast<size_t>(mx) + 1) * sizeof(int), cudaMemcpyHostToDevice, e->stream));
	LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	return LCD_OK;
}

int lcd_index_load_csr(lcd_engine * e, const int * word_ids, int nw, const int64_t * row_ptr, const int * sig, const int * cnt)
{
	if (!e) return LCD_ERR_INVALID;
	if (nw <= 0) return LCD_OK;
	if (!word_ids || !row_ptr || !sig || !cnt) LCD_FAIL(e, LCD_ERR_INVALID, "null argument");
	LCD_TRY(set_device(e));
	const int64_t total = row_ptr[nw] - row_ptr[0];
	int max_word = 0, max_sig = 0;
	// the whole input is validated before any state changes
	if (total < 0) LCD_FAIL(e, LCD_ERR_INVALID, "row_ptr must be non-decreasing");
	for (int k = 0; k < nw; ++k)
	{
		if (e->id2row.find(word_ids[k]) == e->id2row.end()) LCD_FAIL(e, LCD_ERR_INVALID, "word %d is not in the dictionary", word_ids[k]);
		if (row_ptr[k + 1] < row_ptr[k]) LCD_FAIL(e, LCD_ERR_INVALID, "row_ptr must be non-decreasing");
		if (word_ids[k] < static_cast<int>(e->h_len.size()) && e->h_len[word_ids[k]] != 0)
			LCD_FAIL(e, LCD_ERR_STATE, "word %d already has references; bulk load needs empty lists", word_ids[k]);
		max_word = std::max(max_word, word_ids[k]);
	}
	{
		std::unordered_set<int> seen;
		for (int k = 0; k < nw; ++k)
			if (!seen.insert(word_ids[k]).second) LCD_FAIL(e, LCD_ERR_INVALID, "word %d appears twice in the table", word_ids[k]);
	}
	for (int64_t p = row_ptr[0]; p < row_ptr[nw]; ++p)
	{
		if (sig[p] <= 0 || cnt[p] <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "postings need positive signature ids and counts");
		max_sig = std::max(max_sig, sig[p]);
	}
	LCD_TRY(ensure_ids(e, max_word));
	LCD_TRY(ensure_sigs(e, max_sig));
	LCD_TRY(ensure_postings(e, static_cast<size_t>(total)));
	std::vector<int2> buf(static_cast<size_t>(total));
	size_t w = 0;
	for (int k = 0; k < nw; ++k)
	{
		const int word = word_ids[k];
		const int len = static_cast<int>(row_ptr[k + 1] - row_ptr[k]);
		e->h_off[word] = static_cast<uint32_t>(e->post_used + w);
		e->h_len[word] = len;
		e->h_cap[word] = len;
		for (int64_t p = row_ptr[k]; p < row_ptr[k + 1]; ++p)
		{
			buf[w++] = make_int2(sig[p], cnt[p]);
			e->sig_words[sig[p]].emplace_back(word, cnt[p]);
			e->h_ni[sig[p]] += cnt[p];
			e->total_refs += cnt[p];
		}
	}
	// keep the per-signature word lists sorted by word id (add_refs_impl merges against them)
	for (auto & kv : e->sig_words) std::sort(kv.second.begin(), kv.second.end());
	LCD_CUDA(e, cudaMemcpyAsync(e->postings.p + e->post_used, buf.data(), buf.size() * sizeof(int2), cudaMemcpyHostToDevice, e->stream));
	e->post_used += static_cast<size_t>(total);
	LCD_CUDA(e, cudaMemcpyAsync(e->post_off.p, e->h_off.data(), (static_cast<size_t>(max_word) + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
	LCD_CUDA(e, cudaMemcpyAsync(e->post_len.p, e->h_len.data(), (static_cast<size_t>(max_word) + 1) * sizeof(int), cudaMemcpyHostToDevice, e->stream));
	LCD_CUDA(e, cudaMemcpyAsync(e->ni.p, e->h_ni.data(), (static_cast<size_t>(max_sig) + 1) * sizeof(int), cudaMemcpyHostToDevice, e->stream));
	LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	return LCD_OK;
}

int lcd_index_word_nw(lcd_engine * e, int word_id)
{
	if (!e) return LCD_ERR_INVALID;
	if (word_id <= 0 || word_id >= static_cast<int>(e->h_len.size()) || !e->id2row.count(word_id)) return 0;
	return e->h_len[word_id];
}

long long lcd_index_total_refs(const lcd_engine * e) { return e ? e->total_refs : 0; }

int lcd_index_get_refs(lcd_engine * e, int word_id, int * sig, int * cnt, int cap)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (word_id <= 0 || word_id >= static_cast<int>(e->h_len.size()) || !e->id2row.count(word_id)) return 0;
	const int len = e->h_len[word_id];
	if (len == 0) return 0;
	std::vector<int2> buf(len);
	LCD_CUDA(e, cudaMemcpyAsync(buf.data(), e->postings.p + e->h_off[word_id], len * sizeof(int2), cudaMemcpyDeviceToHost, e->stream));
	LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	std::sort(buf.begin(), buf.end(), [](const int2 & x, const int2 & y) { return x.x < y.x; });
	for (int i = 0; i < len && i < cap; ++i)
	{
		if (sig) sig[i] = buf[i].x;
		if (cnt) cnt[i] = buf[i].y;
	}
	return len;
}

int lcd_index_score(lcd_engine * e, const int * query_word_ids, int nq, const int * sig_ids, int ns, int n_total, float * likelihood_out)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!query_word_ids || nq <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "The signature is null");
	if (!sig_ids || ns <= 0 || !likelihood_out) LCD_FAIL(e, LCD_ERR_INVALID, "ids list is empty");
	if (nq > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "at most %d words per signature", kMaxFrameQueries);
	cudaStream_t s = e->stream;
	LCD_CUDA(e, e->d_in_ids.reserve(nq, 0, false, s));
	LCD_CUDA(e, e->d_sig_ids.reserve(ns, 0, false, s));
	LCD_CUDA(e, e->d_like.reserve(ns, 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->d_in_ids.p, query_word_ids, nq * sizeof(int), cudaMemcpyHostToDevice, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->d_sig_ids.p, sig_ids, ns * sizeof(int), cudaMemcpyHostToDevice, s));
	LCD_TRY(ensure_uq(e, 1, nq, s));
	LCD_TRY(ensure_acc(e, 1));
	LCD_CUDA(e, cudaMemsetAsync(e->acc.p, 0, static_cast<size_t>(e->acc_stride) * sizeof(long long), s));
	ResolveArgs a{};
	a.nq = nq;
	fill_prep(e, a, static_cast<float>(n_total), 0);
	int nq_pad = 32;
	while (nq_pad < nq) nq_pad <<= 1;
	prep_from_ids_kernel<<<1, kResolveThreads, nq_pad * sizeof(uint32_t), s>>>(e->d_in_ids.p, a);
	LCD_CHECK_LAUNCH(e);
	LCD_TRY(launch_score(e, 1, nq, s));
	gather_likelihood_kernel<<<dim3((ns + 255) / 256, 1), 256, 0, s>>>(e->acc.p, e->acc_stride, static_cast<int>(e->h_ni.size()), e->d_sig_ids.p, ns, e->d_like.p);
	LCD_CHECK_LAUNCH(e);
	LCD_CUDA(e, cudaMemcpyAsync(likelihood_out, e->d_like.p, ns * sizeof(float), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	return LCD_OK;
}

int lcd_adjust_likelihood_dev(lcd_engine * e, const float * d_likelihood, int n_frames, int ns, int virtual_place_ratio, float * d_adjusted_out,
                              void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!d_likelihood || !d_adjusted_out || n_frames <= 0 || ns <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "likelihood is empty");
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	adjust_likelihood_kernel<<<n_frames, kAdjustThreads, 0, s>>>(d_likelihood, ns, virtual_place_ratio, d_adjusted_out);
	LCD_CHECK_LAUNCH(e);
	return LCD_OK;
}

int lcd_adjust_likelihood(lcd_engine * e, const float * likelihood, int n_frames, int ns, int virtual_place_ratio, float * adjusted_out)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!likelihood || !adjusted_out || n_frames <= 0 || ns <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "likelihood is empty");
	cudaStream_t s = e->stream;
	const size_t n_in = static_cast<size_t>(n_frames) * ns, n_out = static_cast<size_t>(n_frames) * (ns + 1);
	LCD_CUDA(e, e->d_f1.reserve(n_in, 0, false, s));
	LCD_CUDA(e, e->d_f2.reserve(n_out, 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->d_f1.p, likelihood, n_in * sizeof(float), cudaMemcpyHostToDevice, s));
	LCD_TRY(lcd_adjust_likelihood_dev(e, e->d_f1.p, n_frames, ns, virtual_place_ratio, e->d_f2.p, s));
	LCD_CUDA(e, cudaMemcpyAsync(adjusted_out, e->d_f2.p, n_out * sizeof(float), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	return LCD_OK;
}

// ---- Bayes filter over the loop-closure hypotheses ----------------------------------------------------
int lcd_bayes_reset(lcd_engine * e)
{
	if (!e) return LCD_ERR_INVALID;
	e->by_n_state = 0;
	return LCD_OK;
}

int lcd_bayes_compute_posterior(lcd_engine * e, const int * ids, const float * likelihood, int n, const int64_t * col_ptr, const int * nbr_row,
                                const int * nbr_level, const double * prediction_lc, int n_lc, float virtual_place_prior, float * posterior_out)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!ids || !likelihood || n <= 0 || !posterior_out) LCD_FAIL(e, LCD_ERR_INVALID, "likelihood is empty!");
	if (!prediction_lc || n_lc < 2) LCD_FAIL(e, LCD_ERR_INVALID, "Prediction is not valid!");
	if (!col_ptr) LCD_FAIL(e, LCD_ERR_INVALID, "null neighbour table");
	if (!(virtual_place_prior >= 0.f && virtual_place_prior <= 1.f)) LCD_FAIL(e, LCD_ERR_INVALID, "Bayes/VirtualPlacePriorThr must be in [0, 1]");
	for (int i = 1; i < n; ++i)
		if (ids[i] <= ids[i - 1] || ids[i] <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "ids must ascend and only ids[0] may be the (negative) virtual place");
	if (ids[0] == 0) LCD_FAIL(e, LCD_ERR_INVALID, "id 0 is invalid");
	const int64_t nnz = col_ptr[n];
	if (col_ptr[0] != 0 || nnz < 0 || nnz > 0x7FFFFFFF) LCD_FAIL(e, LCD_ERR_INVALID, "bad neighbour table");
	std::vector<int> cp(n + 1), ecol(static_cast<size_t>(nnz));
	for (int c = 0; c < n; ++c)
	{
		if (col_ptr[c + 1] < col_ptr[c]) LCD_FAIL(e, LCD_ERR_INVALID, "col_ptr must be non-decreasing");
		cp[c] = static_cast<int>(col_ptr[c]);
		bool diag = ids[c] < 0;
		for (int64_t k = col_ptr[c]; k < col_ptr[c + 1]; ++k)
		{
			if (nbr_row[k] < 0 || nbr_row[k] >= n || nbr_level[k] < 0 || nbr_level[k] + 1 >= n_lc)
				LCD_FAIL(e, LCD_ERR_INVALID, "neighbour %lld of column %d is out of range", static_cast<long long>(k - col_ptr[c]), c);
			if (k > col_ptr[c] && nbr_row[k] <= nbr_row[k - 1]) LCD_FAIL(e, LCD_ERR_INVALID, "neighbours of a column must ascend");
			diag = diag || nbr_row[k] == c;
			ecol[static_cast<size_t>(k)] = c;
		}
		// generatePrediction: "No 0 margin neighbor for signature" is fatal in the reference (BayesFilter.cpp:371-374)
		if (!diag) LCD_FAIL(e, LCD_ERR_INVALID, "column %d (place %d) does not list the place itself", c, ids[c]);
	}
	cp[n] = static_cast<int>(nnz);
	// _totalPredictionLCValues / _predictionEpsilon as setPredictionLC computes them (float sum of the doubles, smallest value)
	float total = 0.f;
	double eps = prediction_lc[0];
	for (int j = 0; j < n_lc; ++j)
	{
		if (prediction_lc[j] < 0.0 || prediction_lc[j] > 1.0) LCD_FAIL(e, LCD_ERR_INVALID, "The prediction is not valid (values must be between >0 && <=1)");
		if (prediction_lc[j] < eps) eps = prediction_lc[j];
	}
	total = 0.f;
	for (int j = 0; j < n_lc; ++j) total = static_cast<float>(static_cast<double>(total) + prediction_lc[j]); // float += double
	cudaStream_t s = e->stream;
	const size_t nz = static_cast<size_t>(std::max<int64_t>(nnz, 1));
	LCD_CUDA(e, e->by_ids.reserve(n, 0, false, s));
	LCD_CUDA(e, e->by_like.reserve(n, 0, false, s));
	LCD_CUDA(e, e->by_colptr.reserve(n + 1, 0, false, s));
	LCD_CUDA(e, e->by_row.reserve(nz, 0, false, s));
	LCD_CUDA(e, e->by_level.reserve(nz, 0, false, s));
	LCD_CUDA(e, e->by_entry_col.reserve(nz, 0, false, s));
	LCD_CUDA(e, e->by_lc.reserve(n_lc, 0, false, s));
	LCD_CUDA(e, e->by_last.reserve(n, 0, false, s));
	LCD_CUDA(e, e->by_u.reserve(n, 0, false, s));
	LCD_CUDA(e, e->by_scale.reserve(n, 0, false, s));
	LCD_CUDA(e, e->by_delta.reserve(n, 0, false, s));
	LCD_CUDA(e, e->by_post.reserve(n, 0, false, s));
	LCD_CUDA(e, e->by_prior.reserve(n, 0, false, s));
	LCD_CUDA(e, e->by_sums.reserve(4, 0, false, s));
	// the previous state is read while the new one is written: double-buffer by size (state arrays hold max(n, n_state) entries twice)
	const size_t st_need = static_cast<size_t>(std::max(n, e->by_n_state)) * 2;
	LCD_CUDA(e, e->by_state_ids.reserve(st_need, static_cast<size_t>(e->by_n_state), false, s));
	LCD_CUDA(e, e->by_state_post.reserve(st_need, static_cast<size_t>(e->by_n_state), false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->by_ids.p, ids, n * sizeof(int), cudaMemcpyHostToDevice, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->by_like.p, likelihood, n * sizeof(float), cudaMemcpyHostToDevice, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->by_colptr.p, cp.data(), (n + 1) * sizeof(int), cudaMemcpyHostToDevice, s));
	if (nnz)
	{
		LCD_CUDA(e, cudaMemcpyAsync(e->by_row.p, nbr_row, nnz * sizeof(int), cudaMemcpyHostToDevice, s));
		LCD_CUDA(e, cudaMemcpyAsync(e->by_level.p, nbr_level, nnz * sizeof(int), cudaMemcpyHostToDevice, s));
		LCD_CUDA(e, cudaMemcpyAsync(e->by_entry_col.p, ecol.data(), nnz * sizeof(int), cudaMemcpyHostToDevice, s));
	}
	LCD_CUDA(e, cudaMemcpyAsync(e->by_lc.p, prediction_lc, n_lc * sizeof(double), cudaMemcpyHostToDevice, s));
	BayesArgs a{};
	a.n = n;
	a.vp_used = ids[0] < 0 ? 1 : 0;
	a.ids = e->by_ids.p;
	a.like = e->by_like.p;
	a.col_ptr = e->by_colptr.p;
	a.nbr_row = e->by_row.p;
	a.nbr_level = e->by_level.p;
	a.lc = e->by_lc.p;
	a.n_lc = n_lc;
	a.total = total;
	a.eps = static_cast<float>(eps);
	a.vpp = virtual_place_prior;
	// the state lives in the first half of the state arrays, the new one is written to the second half and copied down
	a.prev_ids = e->by_state_ids.p;
	a.prev_post = e->by_state_post.p;
	a.n_prev = e->by_n_state;
	a.last = e->by_last.p;
	a.col_u = e->by_u.p;
	a.col_scale = e->by_scale.p;
	a.col_delta = e->by_delta.p;
	a.prior = e->by_prior.p;
	a.sums = e->by_sums.p;
	a.post = e->by_post.p;
	const int nb = (n + 255) / 256;
	bayes_last_kernel<<<nb, 256, 0, s>>>(a);
	LCD_CHECK_LAUNCH(e);
	bayes_columns_kernel<<<nb, 256, 0, s>>>(a);
	LCD_CHECK_LAUNCH(e);
	if (nnz)
	{
		bayes_scatter_kernel<<<static_cast<unsigned>((nnz + 255) / 256), 256, 0, s>>>(a, static_cast<int>(nnz), e->by_entry_col.p);
		LCD_CHECK_LAUNCH(e);
	}
	bayes_update_kernel<<<nb, 256, 0, s>>>(a);
	LCD_CHECK_LAUNCH(e);
	int * st_i = e->by_state_ids.p + std::max(n, e->by_n_state);
	float * st_p = e->by_state_post.p + std::max(n, e->by_n_state);
	bayes_normalize_kernel<<<nb, 256, 0, s>>>(a, st_i, st_p);
	LCD_CHECK_LAUNCH(e);
	LCD_CUDA(e, cudaMemcpyAsync(e->by_state_ids.p, st_i, n * sizeof(int), cudaMemcpyDeviceToDevice, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->by_state_post.p, st_p, n * sizeof(float), cudaMemcpyDeviceToDevice, s));
	LCD_CUDA(e, cudaMemcpyAsync(posterior_out, e->by_post.p, n * sizeof(float), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	e->by_n_state = n;
	return LCD_OK;
}

// ---- batched localisation ------------------------------------------------------------------
int lcd_localize_batch_dev(lcd_engine * e, const void * d_queries, int n_frames, int nq_per_frame, int incremental, float nndr,
                           int new_words_compared_together, const int * d_sig_ids, int ns, int n_total,
                           int * d_word_ids_out, float * d_likelihood_out, void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!d_queries || n_frames <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "Descriptors size is null!");
	if (nq_per_frame <= 0 || nq_per_frame > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "1..%d descriptors per frame", kMaxFrameQueries);
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	return localize_dev(e, static_cast<const uint32_t *>(d_queries), n_frames, nq_per_frame, incremental, nndr, new_words_compared_together,
	                    d_sig_ids, ns, n_total, d_word_ids_out, d_likelihood_out, s);
}

int lcd_localize_batch(lcd_engine * e, const void * queries, int n_frames, int nq_per_frame, int incremental, float nndr,
                       int new_words_compared_together, const int * sig_ids, int ns, int n_total,
                       int * word_ids_out, float * likelihood_out)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!queries || n_frames <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "Descriptors size is null!");
	if (nq_per_frame <= 0 || nq_per_frame > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "1..%d descriptors per frame", kMaxFrameQueries);
	if (likelihood_out && (!sig_ids || ns <= 0)) LCD_FAIL(e, LCD_ERR_INVALID, "ids list is empty");
	cudaStream_t s = e->stream;
	const size_t nq_total = static_cast<size_t>(n_frames) * nq_per_frame;
	LCD_CUDA(e, e->d_queries.reserve(nq_total * e->nw, 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->d_queries.p, queries, nq_total * e->nw * 4, cudaMemcpyHostToDevice, s));
	if (word_ids_out) LCD_CUDA(e, e->d_word_ids.reserve(nq_total, 0, false, s));
	if (likelihood_out)
	{
		LCD_CUDA(e, e->d_sig_ids.reserve(ns, 0, false, s));
		LCD_CUDA(e, e->d_like.reserve(static_cast<size_t>(n_frames) * ns, 0, false, s));
		LCD_CUDA(e, cudaMemcpyAsync(e->d_sig_ids.p, sig_ids, ns * sizeof(int), cudaMemcpyHostToDevice, s));
	}
	LCD_TRY(localize_dev(e, e->d_queries.p, n_frames, nq_per_frame, incremental, nndr, new_words_compared_together,
	                     e->d_sig_ids.p, likelihood_out ? ns : 0, n_total, word_ids_out ? e->d_word_ids.p : nullptr,
	                     likelihood_out ? e->d_like.p : nullptr, s));
	if (word_ids_out) LCD_CUDA(e, cudaMemcpyAsync(word_ids_out, e->d_word_ids.p, nq_total * sizeof(int), cudaMemcpyDeviceToHost, s));
	if (likelihood_out)
		LCD_CUDA(e, cudaMemcpyAsync(likelihood_out, e->d_like.p, static_cast<size_t>(n_frames) * ns * sizeof(float), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	return LCD_OK;
}

// ---- detect (ORB) ------------------------------------------------------------------------------
static int orb_geometry(lcd_engine * e, int width, int height, const lcd_orb_params * p, OrbGeom & g)
{
	if (!p) LCD_FAIL(e, LCD_ERR_INVALID, "null ORB parameters");
	if (p->n_levels < 1 || p->n_levels > kOrbMaxLevels) LCD_FAIL(e, LCD_ERR_INVALID, "ORB/NLevels must be 1..%d", kOrbMaxLevels);
	if (p->scale_factor != 2.0f) LCD_FAIL(e, LCD_ERR_INVALID, "only ORB/ScaleFactor=2 is implemented");
	if (p->patch_size != 31) LCD_FAIL(e, LCD_ERR_INVALID, "only ORB/PatchSize=31 is implemented");
	if (width <= 0 || height <= 0 || (width % (1 << (p->n_levels - 1))) || (height % (1 << (p->n_levels - 1))))
		LCD_FAIL(e, LCD_ERR_INVALID, "image size must be a multiple of 2^(levels-1)");
	if (static_cast<long long>(width) * height >= (1 << 24)) LCD_FAIL(e, LCD_ERR_CAPACITY, "image too large");
	if (p->n_features <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "Kp/MaxFeatures must be positive");
	g.n_levels = p->n_levels;
	int off = 0;
	for (int l = 0; l < p->n_levels; ++l)
	{
		g.w[l] = width >> l;
		g.h[l] = height >> l;
		g.off[l] = off;
		off += g.w[l] * g.h[l];
	}
	g.frame_stride = off;
	g.edge = p->edge_threshold;
	g.fast_thr = p->fast_threshold;
	g.patch = p->patch_size;
	// ORB computeKeyPoints: features per level (float arithmetic as in OpenCV)
	const float factor = static_cast<float>(1.0 / static_cast<double>(p->scale_factor));
	float nd = p->n_features * (1 - factor) / (1 - static_cast<float>(pow(static_cast<double>(factor), static_cast<double>(p->n_levels))));
	int sum = 0;
	for (int l = 0; l < p->n_levels - 1; ++l)
	{
		g.n_per_level[l] = static_cast<int>(nearbyint(nd));
		sum += g.n_per_level[l];
		nd *= factor;
	}
	g.n_per_level[p->n_levels - 1] = std::max(p->n_features - sum, 0);
	return LCD_OK;
}

// GFTT/ORB: one pyramid level (ORB::compute describes provided keypoints on level 0 only), no divisibility requirement
static int gftt_geometry(lcd_engine * e, int width, int height, const lcd_orb_params * p, OrbGeom & g)
{
	if (!p) LCD_FAIL(e, LCD_ERR_INVALID, "null ORB parameters");
	if (p->patch_size != 31) LCD_FAIL(e, LCD_ERR_INVALID, "only ORB/PatchSize=31 is implemented");
	if (width < 8 || height < 8) LCD_FAIL(e, LCD_ERR_INVALID, "image must be at least 8x8");
	if (static_cast<long long>(width) * height >= (1 << 24)) LCD_FAIL(e, LCD_ERR_CAPACITY, "image too large");
	if (p->n_features <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "Kp/MaxFeatures must be positive");
	if (p->edge_threshold < 0) LCD_FAIL(e, LCD_ERR_INVALID, "ORB/EdgeThreshold must be >= 0");
	g.n_levels = 1;
	g.w[0] = width;
	g.h[0] = height;
	g.off[0] = 0;
	g.frame_stride = width * height;
	g.n_per_level[0] = p->n_features;
	g.edge = p->edge_threshold;
	g.fast_thr = p->fast_threshold;
	g.patch = p->patch_size;
	return LCD_OK;
}

// the host entry points' report of a truncated candidate list (o_overflow)
static int detect_overflow(lcd_engine * e)
{
	if (e->detector == LCD_DETECTOR_GFTT_ORB)
		LCD_FAIL(e, LCD_ERR_CAPACITY, "more than %d GFTT candidate corners in a frame: raise GFTT/QualityLevel", kGfttCandCap);
	LCD_FAIL(e, LCD_ERR_CAPACITY, "more than %d FAST corners in pyramid level 0 (half as many per further level): raise FAST/Threshold", kOrbCandCap);
}

// GFTT corners of frames [frame0, frame0 + n_frames) straight into the keypoint rows (d_kp / d_n already offset to frame0):
// eigenvalue stencil, candidates, selection + ORB::compute's border filter.
static int gftt_detect(lcd_engine * e, int n_frames, int frame0, int total_frames, const OrbGeom & g, const uint8_t * w_gray, const uint8_t * w_mask,
                       int max_corners, int cap, OrbKeypoint * d_kp, int * d_n, cudaStream_t s)
{
	const lcd_gftt_params & gp = e->gftt;
	const int w = g.w[0], h = g.h[0];
	const size_t px = static_cast<size_t>(w) * h;
	const int wpr = (w + 31) / 32;
	LCD_CUDA(e, e->g_eig.reserve(static_cast<size_t>(total_frames) * px, 0, false, s));
	LCD_CUDA(e, e->g_max.reserve(total_frames, 0, false, s));
	LCD_CUDA(e, e->g_cand.reserve(static_cast<size_t>(total_frames) * kGfttCandCap, 0, false, s));
	LCD_CUDA(e, e->g_cand_count.reserve(total_frames, 0, false, s));
	if (gp.block_size == 7) LCD_CUDA(e, e->g_rowsum.reserve(static_cast<size_t>(total_frames) * px * 3, 0, false, s));
	// occupancy bitmap of the accepted corners: shared memory beside the sort buffer when it fits
	const size_t occ_bytes = static_cast<size_t>(h) * wpr * 4;
	const size_t sort_bytes = static_cast<size_t>(kGfttSortCap) * sizeof(unsigned long long);
	const bool occ_smem = sort_bytes + occ_bytes <= 200 * 1024;
	if (!occ_smem) LCD_CUDA(e, e->g_occ.reserve(static_cast<size_t>(total_frames) * h * wpr, 0, false, s));
	LCD_CUDA(e, zero_fill_async(e->g_max.p + frame0, n_frames * sizeof(uint32_t), s));
	LCD_CUDA(e, zero_fill_async(e->g_cand_count.p + frame0, n_frames * sizeof(int), s));
	GfttArgs a{};
	a.gray = w_gray;
	a.mask = w_mask;
	a.w = w;
	a.h = h;
	a.frame_stride = g.frame_stride;
	const double scale = 1.0 / (4.0 * gp.block_size * 255.0);
	a.k0 = static_cast<float>(scale);
	a.k1 = static_cast<float>(2.0 * scale);
	a.eig = e->g_eig.p + static_cast<size_t>(frame0) * px;
	a.max_bits = e->g_max.p + frame0;
	a.rowsum = gp.block_size == 7 ? e->g_rowsum.p + static_cast<size_t>(frame0) * px * 3 : nullptr;
	if (gp.block_size == 7)
	{
		gftt_rowsum7_kernel<<<dim3((h + 127) / 128, n_frames), 128, 0, s>>>(a);
		LCD_CHECK_LAUNCH(e);
		gftt_colsum7_kernel<<<dim3((w + 127) / 128, n_frames), 128, 0, s>>>(a);
	}
	else if (gp.block_size == 5)
		gftt_eigen_kernel<5><<<dim3((w + 4 * 28 - 1) / (4 * 28), n_frames), 128, 0, s>>>(a);
	else
		gftt_eigen_kernel<3><<<dim3((w + 4 * 30 - 1) / (4 * 30), n_frames), 128, 0, s>>>(a);
	LCD_CHECK_LAUNCH(e);
	unsigned long long * cand = e->g_cand.p + static_cast<size_t>(frame0) * kGfttCandCap;
	int * cand_count = e->g_cand_count.p + frame0;
	gftt_candidate_kernel<<<dim3((w + 31) / 32, (h + 7) / 8, n_frames), dim3(32, 8), 0, s>>>(a, gp.quality_level, cand, cand_count, e->o_overflow.p);
	LCD_CHECK_LAUNCH(e);
	GfttSelectArgs sa{};
	sa.cand = cand;
	sa.cand_count = cand_count;
	sa.w = w;
	sa.h = h;
	sa.min_distance = gp.min_distance;
	sa.min_distance2 = gp.min_distance * gp.min_distance;
	sa.cell = gp.min_distance >= 1 ? static_cast<int>(std::nearbyint(gp.min_distance)) : 0; // cvRound: half to even
	sa.max_corners = max_corners;
	sa.edge = g.edge;
	sa.block_size = gp.block_size;
	sa.occ_global = occ_smem ? nullptr : e->g_occ.p + static_cast<size_t>(frame0) * h * wpr;
	sa.kp = d_kp;
	sa.n_kp = d_n;
	sa.cap = cap;
	const size_t smem = sort_bytes + (occ_smem ? occ_bytes : 0);
	LCD_CUDA(e, cudaFuncSetAttribute(gftt_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
	gftt_select_kernel<<<n_frames, kGfttSelectThreads, smem, s>>>(sa);
	LCD_CHECK_LAUNCH(e);
	return LCD_OK;
}

int lcd_set_detector(lcd_engine * e, int strategy, const lcd_gftt_params * gftt)
{
	if (!e) return LCD_ERR_INVALID;
	if (strategy == LCD_DETECTOR_ORB)
	{
		e->detector = strategy;
		return LCD_OK;
	}
	if (strategy != LCD_DETECTOR_GFTT_ORB) LCD_FAIL(e, LCD_ERR_INVALID, "Kp/DetectorStrategy %d is not implemented (2 = ORB, 8 = GFTT/ORB)", strategy);
	if (!gftt) LCD_FAIL(e, LCD_ERR_INVALID, "GFTT/ORB needs its GFTT parameters");
	if (!(gftt->quality_level > 0.0) || !std::isfinite(gftt->quality_level)) LCD_FAIL(e, LCD_ERR_INVALID, "GFTT/QualityLevel must be > 0");
	if (!(gftt->min_distance >= 0.0) || !std::isfinite(gftt->min_distance)) LCD_FAIL(e, LCD_ERR_INVALID, "GFTT/MinDistance must be >= 0");
	if (gftt->block_size != 3 && gftt->block_size != 5 && gftt->block_size != 7) LCD_FAIL(e, LCD_ERR_INVALID, "GFTT/BlockSize must be 3, 5 or 7");
	if (gftt->use_harris) LCD_FAIL(e, LCD_ERR_INVALID, "GFTT/UseHarrisDetector=true is not implemented");
	e->gftt = *gftt;
	e->detector = strategy;
	return LCD_OK;
}

// Detect + describe frames [frame0, frame0 + n_frames) of a batch of total_frames (total_frames = 0: the range is the whole
// batch).  Every input, workspace and output pointer addresses frame 0 of the batch; ranges are independent, so the host
// path runs them chunk by chunk while the next chunk's images are still on their way over PCIe.
static int orb_run(lcd_engine * e, int n_frames, const uint8_t * d_images, int width, int height, int channels, const void * d_depth,
                   int depth_type, const lcd_orb_params * p, int cap, OrbKeypoint * d_kp, uint8_t * d_desc, float * d_xyz, float * d_uv,
                   int * d_n, cudaStream_t s, int frame0 = 0, int total_frames = 0)
{
	if (total_frames <= 0) total_frames = frame0 + n_frames;
	const bool gftt = e->detector == LCD_DETECTOR_GFTT_ORB;
	OrbGeom g{};
	LCD_TRY(gftt ? gftt_geometry(e, width, height, p, g) : orb_geometry(e, width, height, p, g));
	if (channels != 1 && channels != 3) LCD_FAIL(e, LCD_ERR_INVALID, "images must be 8UC1 or 8UC3 (BGR)");
	if (cap <= 0 || cap > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "cap must be 1..%d", kMaxFrameQueries);
	if (!d_depth) depth_type = LCD_DEPTH_NONE;
	if (depth_type < LCD_DEPTH_NONE || depth_type > LCD_DEPTH_MASK_U8) LCD_FAIL(e, LCD_ERR_INVALID, "unknown depth type %d", depth_type);
	const bool use_mask = depth_type == LCD_DEPTH_MASK_U8 || (depth_type != LCD_DEPTH_NONE && p->depth_as_mask);
	const size_t pyr = static_cast<size_t>(total_frames) * g.frame_stride;
	LCD_CUDA(e, e->o_gray.reserve(pyr, 0, false, s));
	LCD_CUDA(e, e->o_blur.reserve(pyr, 0, false, s));
	if (use_mask) LCD_CUDA(e, e->o_mask.reserve(pyr, 0, false, s));
	const int slots = n_frames * g.n_levels, total_slots = total_frames * g.n_levels, slot0 = frame0 * g.n_levels;
	int level_cap = 0;
	for (int l = 0; l < g.n_levels; ++l) level_cap = std::max(level_cap, g.n_per_level[l] + 256);
	if (!gftt)
	{
		LCD_CUDA(e, e->o_cand.reserve(static_cast<size_t>(total_slots) * kOrbCandCap, 0, false, s));
		LCD_CUDA(e, e->o_cand_count.reserve(total_slots, 0, false, s));
		LCD_CUDA(e, e->o_level_n.reserve(total_slots, 0, false, s));
		LCD_CUDA(e, e->o_level_kp.reserve(static_cast<size_t>(total_slots) * level_cap, 0, false, s));
	}
	if (frame0 == 0)
	{
		// the "candidate list truncated" flag of this batch: cleared here, read back by the host entry points
		LCD_CUDA(e, e->o_overflow.reserve(1, 0, true, s));
		LCD_CUDA(e, zero_fill_async(e->o_overflow.p, sizeof(int), s));
	}
	if (!d_kp)
	{
		LCD_CUDA(e, e->o_kp.reserve(static_cast<size_t>(total_frames) * cap, 0, false, s));
		d_kp = e->o_kp.p;
	}
	if (!d_n)
	{
		LCD_CUDA(e, e->o_n.reserve(total_frames, 0, false, s));
		d_n = e->o_n.p;
	}
	// pointers of the range
	const size_t px = static_cast<size_t>(width) * height;
	d_images += static_cast<size_t>(frame0) * px * channels;
	if (d_depth) d_depth = static_cast<const unsigned char *>(d_depth) + static_cast<size_t>(frame0) * px * (depth_elem_bytes(depth_type));
	uint8_t * const w_gray = e->o_gray.p + static_cast<size_t>(frame0) * g.frame_stride;
	uint8_t * const w_blur = e->o_blur.p + static_cast<size_t>(frame0) * g.frame_stride;
	uint8_t * const w_mask = use_mask ? e->o_mask.p + static_cast<size_t>(frame0) * g.frame_stride : nullptr;
	uint32_t * const w_cand = gftt ? nullptr : e->o_cand.p + static_cast<size_t>(slot0) * kOrbCandCap;
	int * const w_cand_count = gftt ? nullptr : e->o_cand_count.p + slot0;
	int * const w_level_n = gftt ? nullptr : e->o_level_n.p + slot0;
	OrbKeypoint * const w_level_kp = gftt ? nullptr : e->o_level_kp.p + static_cast<size_t>(slot0) * level_cap;
	d_kp += static_cast<size_t>(frame0) * cap;
	d_n += frame0;
	if (d_desc) d_desc += static_cast<size_t>(frame0) * cap * 32;
	if (d_xyz) d_xyz += static_cast<size_t>(frame0) * cap * 3;
	if (d_uv) d_uv += static_cast<size_t>(frame0) * cap * 2;
	if (e->gauss_sigma_loaded != 2.0f)
	{
		// cv::getGaussianKernel(7, 2, CV_32F): exp(-x^2 / (2 sigma^2)) normalised in double, stored as float
		double t[7], sum = 0;
		for (int i = 0; i < 7; ++i)
		{
			t[i] = exp(-0.5 * (i - 3) * (i - 3) / 4.0);
			sum += t[i];
		}
		float kf[7];
		for (int i = 0; i < 7; ++i) kf[i] = static_cast<float>(t[i] / sum);
		LCD_CUDA(e, cudaMemcpyToSymbolAsync(kOrbGauss7, kf, sizeof(kf), 0, cudaMemcpyHostToDevice, s));
		LCD_CUDA(e, cudaStreamSynchronize(s));
		e->gauss_sigma_loaded = 2.0f;
	}
	prof_mark(e, LCD_PROF_ORB, s);
	if (!gftt) LCD_CUDA(e, zero_fill_async(w_cand_count, slots * sizeof(int), s));
	{
		OrbPrepArgs a{};
		a.images = d_images;
		a.channels = channels;
		a.depth = use_mask ? d_depth : nullptr;
		a.depth_type = depth_type;
		a.min_depth = p->min_depth;
		a.max_depth = p->max_depth;
		a.gray = w_gray;
		a.mask = w_mask;
		a.g = g;
		const bool aligned = ((reinterpret_cast<uintptr_t>(d_images) | reinterpret_cast<uintptr_t>(a.depth) | reinterpret_cast<uintptr_t>(w_gray) |
		                       reinterpret_cast<uintptr_t>(w_mask)) & 15u) == 0 && g.frame_stride % 16 == 0;
		e->orb_path = 0;
		if (width % 8 == 0 && height % 2 == 0 && aligned && env_int("LCD_ORB_PREP_VEC", 1) != 0)
		{
			e->orb_path |= 4;
			dim3 blk(16, 16), grd((width / 8 + 15) / 16, (height / 2 + 15) / 16, n_frames);
			orb_prepare_vec_kernel<<<grd, blk, 0, s>>>(a);
		}
		else
		{
			dim3 blk(32, 8), grd(((width + 1) / 2 + 31) / 32, ((height + 1) / 2 + 7) / 8, n_frames);
			orb_prepare_kernel<<<grd, blk, 0, s>>>(a);
		}
		LCD_CHECK_LAUNCH(e);
	}
	for (int l = 2; l < g.n_levels; ++l)
	{
		dim3 blk(32, 8), grd((g.w[l] + 31) / 32, (g.h[l] + 7) / 8, n_frames);
		orb_down_kernel<<<grd, blk, 0, s>>>(w_gray, w_mask, g, l);
		LCD_CHECK_LAUNCH(e);
	}
	if (!e->aux_fork)
	{
		LCD_CUDA(e, cudaEventCreateWithFlags(&e->aux_fork, cudaEventDisableTiming));
		LCD_CUDA(e, cudaEventCreateWithFlags(&e->aux_blur_done, cudaEventDisableTiming));
		for (int i = 0; i < 4; ++i)
		{
			LCD_CUDA(e, cudaStreamCreateWithFlags(&e->aux_stream[i], cudaStreamNonBlocking));
			LCD_CUDA(e, cudaEventCreateWithFlags(&e->aux_join[i], cudaEventDisableTiming));
		}
	}
	// one tensor map per pyramid level ([frame][y][x], 96 x 40 boxes): shared by the FAST and the blur kernels
	const int orb_tma = env_int("LCD_ORB_TMA", 1);
	OrbTensorMap tmaps[kOrbMaxLevels];
	bool tma_ok = orb_tma != 0;
	for (int l = 0; l < g.n_levels && tma_ok; ++l)
		tma_ok = make_plane_tensor_map(&tmaps[l], w_gray + g.off[l], g.w[l], g.h[l], n_frames, static_cast<size_t>(g.frame_stride), kFastTmaGW, kFastTmaGH);
	e->orb_tma_used = tma_ok ? 1 : 0;
	if (tma_ok) e->orb_path |= 1;
	LCD_CUDA(e, cudaEventRecord(e->aux_fork, s));
	if (d_desc)
	{
		// the blurred pyramid only feeds the descriptors: it runs on a side stream under FAST and the (latency-bound) selection
		cudaStream_t bs = e->aux_stream[3];
		LCD_CUDA(e, cudaStreamWaitEvent(bs, e->aux_fork, 0));
		for (int l = 0; l < g.n_levels; ++l)
		{
			if (tma_ok)
			{
				dim3 grd((g.w[l] + kFastTmaTW - 1) / kFastTmaTW, (g.h[l] + kFastTmaTH - 1) / kFastTmaTH, n_frames);
				orb_blur_tma_kernel<<<grd, 256, 0, bs>>>(tmaps[l], w_blur, g, l);
			}
			else
			{
				dim3 grd((g.w[l] + kBlurTW - 1) / kBlurTW, (g.h[l] + kBlurTH - 1) / kBlurTH, n_frames);
				orb_blur_kernel<<<grd, 256, 0, bs>>>(w_gray, w_blur, g, l);
			}
			LCD_CHECK_LAUNCH(e);
		}
		LCD_CUDA(e, cudaEventRecord(e->aux_blur_done, bs));
	}
	if (gftt)
		LCD_TRY(gftt_detect(e, n_frames, frame0, total_frames, g, w_gray, w_mask, p->n_features, cap, d_kp, d_n, s));
	else
	{
		OrbSelectArgs a{};
		a.gray = w_gray;
		a.g = g;
		a.cand = w_cand;
		a.cand_count = w_cand_count;
		a.level_kp = w_level_kp;
		a.level_n = w_level_n;
		a.level_cap = level_cap;
		a.overflow = e->o_overflow.p;
		// The levels are independent: level 0 (the long one) stays on the caller's stream, the coarser ones run FAST + selection on side
		// streams beside it and join before the merge.  Selection is one CTA per (frame, level), latency-bound: level l holds at most
		// kOrbCandCap >> l candidates in shared memory (192 KB, 96 KB, 48 KB, ...), so the FAST / blur CTAs of other levels share its SMs.
		LCD_CUDA(e, cudaFuncSetAttribute(orb_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
		                                 static_cast<int>(static_cast<size_t>(kOrbCandCap) * (4 + 4 + 2 + 2))));
		for (int l = g.n_levels - 1; l >= 0; --l)
		{
			cudaStream_t ls = s;
			if (l > 0)
			{
				ls = e->aux_stream[(l - 1) % 3];
				LCD_CUDA(e, cudaStreamWaitEvent(ls, e->aux_fork, 0));
			}
			if (tma_ok)
			{
				// gray tile + halo staged by the TMA engine (one cp.async.bulk.tensor per CTA), byte-SIMD compass test and suppression
				dim3 grd((g.w[l] + kFastTmaTW - 1) / kFastTmaTW, (g.h[l] + kFastTmaTH - 1) / kFastTmaTH, n_frames);
				orb_fast_tma_kernel<<<grd, 256, 0, ls>>>(tmaps[l], w_mask, g, l, w_cand, w_cand_count);
			}
			else
			{
				dim3 grd((g.w[l] + kFastTW - 1) / kFastTW, (g.h[l] + kFastTH - 1) / kFastTH, n_frames);
				orb_fast_kernel<<<grd, 256, 0, ls>>>(w_gray, w_mask, g, l, w_cand, w_cand_count);
			}
			LCD_CHECK_LAUNCH(e);
			a.level = l;
			a.cand_cap = std::max(2048, kOrbCandCap >> l);
			const size_t smem = static_cast<size_t>(a.cand_cap) * (4 + 4 + 2 + 2);
			orb_select_kernel<<<n_frames, kOrbSelectThreads, smem, ls>>>(a);
			LCD_CHECK_LAUNCH(e);
			if (l > 0 && l <= 3) LCD_CUDA(e, cudaEventRecord(e->aux_join[l - 1], ls));
		}
		for (int l = 1; l < g.n_levels && l <= 3; ++l) LCD_CUDA(e, cudaStreamWaitEvent(s, e->aux_join[l - 1], 0));
		int pad = 1;
		while (pad < g.n_levels * level_cap) pad <<= 1;
		orb_merge_kernel<<<n_frames, 1024, pad * sizeof(unsigned long long), s>>>(w_level_kp, w_level_n, g.n_levels, level_cap, p->n_features,
		                                                                          d_kp, d_n, cap);
		LCD_CHECK_LAUNCH(e);
	}
	if (d_desc)
	{
		LCD_CUDA(e, cudaStreamWaitEvent(s, e->aux_blur_done, 0));
		dim3 grd((cap + kOrbDescribeKp - 1) / kOrbDescribeKp, n_frames);
		bool patch_ok = g.edge >= kOrbPatchR && env_int("LCD_ORB_PATCH", 1) != 0;
		for (int l = 0; l < g.n_levels; ++l) patch_ok = patch_ok && g.w[l] % 4 == 0;
		if (patch_ok) e->orb_path |= 2;
		if (patch_ok)
			orb_describe_patch_kernel<<<grd, 256, 0, s>>>(w_blur, g, d_kp, d_n, cap, d_desc);
		else
			orb_describe_kernel<<<grd, 256, 0, s>>>(w_gray, w_blur, g, d_kp, d_n, cap, d_desc);
		LCD_CHECK_LAUNCH(e);
	}
	if (d_xyz || d_uv)
	{
		if (d_xyz)
		{
			OrbXyzArgs a{};
			a.depth = (depth_type != LCD_DEPTH_NONE && depth_type != LCD_DEPTH_MASK_U8) ? d_depth : nullptr;
			a.depth_type = depth_type;
			a.w = width;
			a.h = height;
			a.fx = p->fx;
			a.fy = p->fy;
			a.cx = p->cx;
			a.cy = p->cy;
			a.min_depth = p->min_depth;
			a.max_depth = p->max_depth;
			a.kps = d_kp;
			a.n_kp = d_n;
			a.cap = cap;
			a.xyz = d_xyz;
			dim3 grd((cap + 255) / 256, n_frames);
			orb_xyz_kernel<<<grd, 256, 0, s>>>(a);
			LCD_CHECK_LAUNCH(e);
		}
		if (d_uv)
		{
			dim3 grd((cap + 255) / 256, n_frames);
			orb_uv_kernel<<<grd, 256, 0, s>>>(d_kp, d_n, cap, d_uv);
			LCD_CHECK_LAUNCH(e);
		}
	}
	prof_mark(e, LCD_PROF_ORB, s);
	return LCD_OK;
}

int lcd_orb_detect_describe_dev(lcd_engine * e, int n_frames, const uint8_t * d_images, int width, int height, int channels, const void * d_depth,
                                int depth_type, const lcd_orb_params * params, int cap, lcd_keypoint * d_kp_out, uint8_t * d_desc_out,
                                float * d_xyz_out, float * d_uv_out, int * d_n_out, void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!d_images || n_frames <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "null image");
	static_assert(sizeof(lcd_keypoint) == sizeof(OrbKeypoint), "keypoint layout");
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	return orb_run(e, n_frames, d_images, width, height, channels, d_depth, depth_type, params, cap, reinterpret_cast<OrbKeypoint *>(d_kp_out),
	               d_desc_out, d_xyz_out, d_uv_out, d_n_out, s);
}

int lcd_orb_detect_describe(lcd_engine * e, int n_frames, const uint8_t * images, int width, int height, int channels, const void * depth,
                            int depth_type, const lcd_orb_params * params, int cap, lcd_keypoint * kp_out, uint8_t * desc_out, float * xyz_out,
                            int * n_out)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!images || n_frames <= 0 || width <= 0 || height <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "null image");
	if (cap <= 0 || cap > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "cap must be 1..%d", kMaxFrameQueries);
	cudaStream_t s = e->orb_stream; // not the dictionary's stream: this call may overlap lcd_dict_update (Memory.cpp:5284)
	const size_t px = static_cast<size_t>(n_frames) * width * height;
	LCD_CUDA(e, e->o_img.reserve(px * channels, 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->o_img.p, images, px * channels, cudaMemcpyHostToDevice, s));
	if (!depth) depth_type = LCD_DEPTH_NONE;
	const size_t dbytes = depth_elem_bytes(depth_type);
	if (depth_type != LCD_DEPTH_NONE)
	{
		LCD_CUDA(e, e->o_depth.reserve(px * dbytes, 0, false, s));
		LCD_CUDA(e, cudaMemcpyAsync(e->o_depth.p, depth, px * dbytes, cudaMemcpyHostToDevice, s));
	}
	const size_t rows = static_cast<size_t>(n_frames) * cap;
	LCD_CUDA(e, e->o_kp.reserve(rows, 0, false, s));
	LCD_CUDA(e, e->o_desc.reserve(rows * 32, 0, false, s));
	LCD_CUDA(e, e->o_xyz.reserve(rows * 3, 0, false, s));
	LCD_CUDA(e, e->o_n.reserve(n_frames, 0, false, s));
	LCD_TRY(orb_run(e, n_frames, e->o_img.p, width, height, channels, depth_type != LCD_DEPTH_NONE ? e->o_depth.p : nullptr, depth_type, params, cap,
	                e->o_kp.p, desc_out ? e->o_desc.p : nullptr, xyz_out ? e->o_xyz.p : nullptr, nullptr, e->o_n.p, s));
	if (kp_out) LCD_CUDA(e, cudaMemcpyAsync(kp_out, e->o_kp.p, rows * sizeof(OrbKeypoint), cudaMemcpyDeviceToHost, s));
	if (desc_out) LCD_CUDA(e, cudaMemcpyAsync(desc_out, e->o_desc.p, rows * 32, cudaMemcpyDeviceToHost, s));
	if (xyz_out) LCD_CUDA(e, cudaMemcpyAsync(xyz_out, e->o_xyz.p, rows * 3 * sizeof(float), cudaMemcpyDeviceToHost, s));
	if (n_out) LCD_CUDA(e, cudaMemcpyAsync(n_out, e->o_n.p, n_frames * sizeof(int), cudaMemcpyDeviceToHost, s));
	int overflow = 0;
	LCD_CUDA(e, cudaMemcpyAsync(&overflow, e->o_overflow.p, sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	if (overflow) return detect_overflow(e);
	return LCD_OK;
}

int lcd_orb_overflow(lcd_engine * e)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!e->o_overflow.p) return 0;
	int flag = 0;
	LCD_CUDA(e, cudaDeviceSynchronize());
	LCD_CUDA(e, cudaMemcpy(&flag, e->o_overflow.p, sizeof(int), cudaMemcpyDeviceToHost));
	return flag ? 1 : 0;
}

int lcd_orb_last_path(const lcd_engine * e)
{
	return e ? e->orb_path : LCD_ERR_INVALID;
}

long long lcd_debug_orb_buffer(lcd_engine * e, int which, void * out, long long cap_bytes)
{
	if (!e || !out) return LCD_ERR_INVALID;
	if (set_device(e) != LCD_OK) return LCD_ERR_CUDA;
	const void * src = nullptr;
	size_t bytes = 0;
	switch (which)
	{
	case 0: src = e->o_gray.p; bytes = e->o_gray.cap; break;
	case 1: src = e->o_mask.p; bytes = e->o_mask.cap; break;
	case 2: src = e->o_blur.p; bytes = e->o_blur.cap; break;
	case 3: src = e->o_cand.p; bytes = e->o_cand.cap * sizeof(uint32_t); break;
	case 4: src = e->o_cand_count.p; bytes = e->o_cand_count.cap * sizeof(int); break;
	case 5: src = e->o_level_n.p; bytes = e->o_level_n.cap * sizeof(int); break;
	case 10: src = e->g_eig.p; bytes = e->g_eig.cap * sizeof(float); break;
	case 7: src = e->v_clk.p; bytes = e->v_clk.cap * sizeof(long long); break;
#ifdef LCD_DEBUG_PHASES
	case 9:
	{
		void * sym = nullptr;
		if (cudaGetSymbolAddress(&sym, g_match_dbg) != cudaSuccess) return LCD_ERR_CUDA;
		src = sym;
		bytes = sizeof(long long) * 8;
		break;
	}
#endif
	case 8:
	{
		void * sym = nullptr;
		if (cudaGetSymbolAddress(&sym, g_pnp_dbg) != cudaSuccess) return LCD_ERR_CUDA;
		src = sym;
		bytes = sizeof(long long) * 8;
		break;
	}
	default: return LCD_ERR_INVALID;
	}
	if (!src) return 0;
	bytes = std::min<size_t>(bytes, static_cast<size_t>(cap_bytes));
	if (cudaMemcpy(out, src, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) return LCD_ERR_CUDA;
	return static_cast<long long>(bytes);
}

// ---- geometric verification ------------------------------------------------------------------
static int verify_upload(lcd_engine * e, int n_pairs, int cap, const void * desc_from, const float * xyz_from, const int * n_from,
                         const void * desc_to, const float * uv_to, const int * n_to, cudaStream_t s, const float * xyz_to = nullptr)
{
	const size_t rows = static_cast<size_t>(n_pairs) * cap;
	LCD_CUDA(e, e->v_df.reserve(rows * e->nw, 0, false, s));
	LCD_CUDA(e, e->v_dt.reserve(rows * e->nw, 0, false, s));
	LCD_CUDA(e, e->v_xyz.reserve(rows * 3, 0, false, s));
	LCD_CUDA(e, e->v_uv.reserve(rows * 2, 0, false, s));
	LCD_CUDA(e, e->v_nf.reserve(n_pairs, 0, false, s));
	LCD_CUDA(e, e->v_nt.reserve(n_pairs, 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->v_df.p, desc_from, rows * e->nw * 4, cudaMemcpyHostToDevice, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->v_dt.p, desc_to, rows * e->nw * 4, cudaMemcpyHostToDevice, s));
	if (xyz_from) LCD_CUDA(e, cudaMemcpyAsync(e->v_xyz.p, xyz_from, rows * 3 * sizeof(float), cudaMemcpyHostToDevice, s));
	else LCD_CUDA(e, cudaMemsetAsync(e->v_xyz.p, 0, rows * 3 * sizeof(float), s));
	if (uv_to) LCD_CUDA(e, cudaMemcpyAsync(e->v_uv.p, uv_to, rows * 2 * sizeof(float), cudaMemcpyHostToDevice, s));
	else LCD_CUDA(e, cudaMemsetAsync(e->v_uv.p, 0, rows * 2 * sizeof(float), s));
	LCD_CUDA(e, cudaMemcpyAsync(e->v_nf.p, n_from, n_pairs * sizeof(int), cudaMemcpyHostToDevice, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->v_nt.p, n_to, n_pairs * sizeof(int), cudaMemcpyHostToDevice, s));
	if (xyz_to)
	{
		LCD_CUDA(e, e->v_xyz_to.reserve(rows * 3, 0, false, s));
		LCD_CUDA(e, cudaMemcpyAsync(e->v_xyz_to.p, xyz_to, rows * 3 * sizeof(float), cudaMemcpyHostToDevice, s));
	}
	return LCD_OK;
}

struct MatchSrc
{
	const uint32_t * desc_from;
	const float * xyz_from;
	const int * n_from;
	const int * from_slot;
	int cap_from;
	const uint32_t * desc_to;
	const float * uv_to;
	const int * n_to;
	int n_to_all;
	int cap_to;
	const float * xyz_to; // 3-D points of the TO side (words3B) or nullptr
};

static int launch_match(lcd_engine * e, int n_pairs, int cap, float nndr, bool want_ids, cudaStream_t s, const MatchSrc * src = nullptr)
{
	const size_t rows = static_cast<size_t>(n_pairs) * cap;
	LCD_CUDA(e, e->v_obj.reserve(rows * 3, 0, false, s));
	LCD_CUDA(e, e->v_img.reserve(rows * 2, 0, false, s));
	LCD_CUDA(e, e->v_mid.reserve(rows, 0, false, s));
	LCD_CUDA(e, e->v_mfrom.reserve(rows, 0, false, s));
	LCD_CUDA(e, e->v_mto.reserve(rows, 0, false, s));
	LCD_CUDA(e, e->v_nm.reserve(n_pairs, 0, false, s));
	if (want_ids)
	{
		LCD_CUDA(e, e->v_fid.reserve(rows, 0, false, s));
		LCD_CUDA(e, e->v_tid.reserve(rows, 0, false, s));
	}
	MatchArgs a{};
	if (src)
	{
		a.desc_from = src->desc_from;
		a.xyz_from = src->xyz_from;
		a.n_from = src->n_from;
		a.from_slot = src->from_slot;
		a.cap_from = src->cap_from;
		a.desc_to = src->desc_to;
		a.uv_to = src->uv_to;
		a.n_to = src->n_to;
		a.n_to_all = src->n_to_all;
		a.cap_to = src->cap_to;
		a.xyz_to = src->xyz_to;
	}
	else
	{
		a.desc_from = e->v_df.p;
		a.xyz_from = e->v_xyz.p;
		a.n_from = e->v_nf.p;
		a.from_slot = nullptr;
		a.cap_from = cap;
		a.desc_to = e->v_dt.p;
		a.uv_to = e->v_uv.p;
		a.n_to = e->v_nt.p;
		a.n_to_all = 0;
		a.cap_to = cap;
		a.xyz_to = e->match_has_xyz_to ? e->v_xyz_to.p : nullptr;
	}
	if (a.xyz_to) LCD_CUDA(e, e->v_obj_to.reserve(rows * 3, 0, false, s));
	a.obj_to = a.xyz_to ? e->v_obj_to.p : nullptr;
	e->pnp_has_obj_to = a.xyz_to != nullptr;
	a.cap = cap;
	a.nndr = nndr;
	a.obj = e->v_obj.p;
	a.img = e->v_img.p;
	a.match_id = e->v_mid.p;
	a.match_from = e->v_mfrom.p;
	a.match_to = e->v_mto.p;
	a.n_match = e->v_nm.p;
	a.from_ids = want_ids ? e->v_fid.p : nullptr;
	a.to_ids = want_ids ? e->v_tid.p : nullptr;
	const size_t smem = match_smem_bytes(cap, e->nw);
	if (smem > static_cast<size_t>(e->smem_optin)) LCD_FAIL(e, LCD_ERR_CAPACITY, "cap %d needs %zu B of shared memory", cap, smem);
#define LCD_MATCH_CASE(NW_)                                                                                             \
	case NW_:                                                                                                           \
	{                                                                                                                   \
		auto kern = pair_match_kernel<NW_>;                                                                             \
		if (smem > 48 * 1024)                                                                                           \
			LCD_CUDA(e, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem))); \
		prof_mark(e, LCD_PROF_MATCH, s);                                                                                \
		kern<<<n_pairs, kResolveThreads, smem, s>>>(a);                                                                 \
		prof_mark(e, LCD_PROF_MATCH, s);                                                                                \
		break;                                                                                                          \
	}
	switch (e->nw)
	{
		LCD_MATCH_CASE(4)
		LCD_MATCH_CASE(8)
		LCD_MATCH_CASE(16)
	default: LCD_FAIL(e, LCD_ERR_INVALID, "unsupported descriptor size");
	}
#undef LCD_MATCH_CASE
	LCD_CHECK_LAUNCH(e);
	return LCD_OK;
}

static int launch_pnp(lcd_engine * e, int n_pairs, int cap, const lcd_verify_params * p, cudaStream_t s, bool gate_min_matches = true,
                      bool want_cov = true)
{
	const size_t rows = static_cast<size_t>(n_pairs) * cap;
	if (want_cov && p->var_median_ratio <= 1) LCD_FAIL(e, LCD_ERR_INVALID, "Vis/PnPVarianceMedianRatio must be > 1 (UASSERT in estimateMotion3DTo2D)");
	LCD_CUDA(e, e->v_cov6.reserve(n_pairs * 6, 0, false, s));
	LCD_CUDA(e, e->v_rvec.reserve(n_pairs * 3, 0, false, s));
	LCD_CUDA(e, e->v_tvec.reserve(n_pairs * 3, 0, false, s));
	LCD_CUDA(e, e->v_inl.reserve(rows, 0, false, s));
	LCD_CUDA(e, e->v_ninl.reserve(n_pairs, 0, false, s));
	LCD_CUDA(e, e->v_iters.reserve(n_pairs, 0, false, s));
	LCD_CUDA(e, e->v_ok.reserve(n_pairs, 0, false, s));
	LCD_CUDA(e, e->v_T.reserve(n_pairs * 12, 0, false, s));
	LCD_CUDA(e, e->v_clk.reserve(n_pairs * 16, 0, false, s));
	PnpArgs a{};
	a.obj = e->v_obj.p;
	a.img = e->v_img.p;
	a.n_pts = e->v_nm.p;
	a.cap = cap;
	a.cam = CamK{p->fx, p->fy, p->cx, p->cy};
	a.iterations = p->iterations;
	a.reproj = p->reproj_error;
	a.min_inliers = p->min_inliers;
	a.refine_iterations = p->refine_iterations;
	a.refine_sigma = p->refine_sigma;
	a.gate_min_matches = gate_min_matches ? 1 : 0;
	a.obj_to = (want_cov && e->pnp_has_obj_to) ? e->v_obj_to.p : nullptr;
	a.var_median_ratio = p->var_median_ratio;
	a.max_variance = p->max_variance;
	a.split_linear = p->split_linear_cov;
	a.img_w = p->image_width;
	a.img_h = p->image_height;
	a.cov6 = want_cov ? e->v_cov6.p : nullptr;
	a.rvec = e->v_rvec.p;
	a.tvec = e->v_tvec.p;
	a.inliers = e->v_inl.p;
	a.n_inliers = e->v_ninl.p;
	a.iters_run = e->v_iters.p;
	a.ok = e->v_ok.p;
	a.transform = e->v_T.p;
	static const int pnp_clocks = env_int("LCD_PNP_CLOCKS", 0); // diagnostics: phase clocks of the RANSAC kernel (lcd_debug_orb_buffer 7)
	a.phase_clk = pnp_clocks ? e->v_clk.p : nullptr;
	const size_t smem = pnp_smem_bytes(cap);
	if (smem > static_cast<size_t>(e->smem_optin)) LCD_FAIL(e, LCD_ERR_CAPACITY, "cap %d needs %zu B of shared memory", cap, smem);
	if (smem > 48 * 1024)
		LCD_CUDA(e, cudaFuncSetAttribute(pnp_ransac_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
	prof_mark(e, LCD_PROF_PNP, s);
	pnp_ransac_kernel<<<n_pairs, kVerifyThreads, smem, s>>>(a);
	prof_mark(e, LCD_PROF_PNP, s);
	LCD_CHECK_LAUNCH(e);
	return LCD_OK;
}

// Reg/RepeatOnce: the second registration pass of the pairs whose first pass succeeded (guess_match_kernel), then PnP again on all pairs
// (pairs that keep their first-pass correspondences reproduce their first-pass result).  src as in launch_match.
static int launch_second_pass(lcd_engine * e, int n_pairs, int cap, const lcd_verify_params * p, cudaStream_t s, const MatchSrc * src)
{
	if (!p->repeat_once || p->guess_win_size <= 0 || p->image_width <= 0 || p->image_height <= 0) return LCD_OK;
	GuessMatchArgs a{};
	if (src)
	{
		a.desc_from = src->desc_from;
		a.xyz_from = src->xyz_from;
		a.n_from = src->n_from;
		a.from_slot = src->from_slot;
		a.cap_from = src->cap_from;
		a.desc_to = src->desc_to;
		a.uv_to = src->uv_to;
		a.xyz_to = src->xyz_to;
		a.n_to = src->n_to;
		a.n_to_all = src->n_to_all;
		a.cap_to = src->cap_to;
	}
	else
	{
		a.desc_from = e->v_df.p;
		a.xyz_from = e->v_xyz.p;
		a.n_from = e->v_nf.p;
		a.from_slot = nullptr;
		a.cap_from = cap;
		a.desc_to = e->v_dt.p;
		a.uv_to = e->v_uv.p;
		a.xyz_to = e->match_has_xyz_to ? e->v_xyz_to.p : nullptr;
		a.n_to = e->v_nt.p;
		a.n_to_all = 0;
		a.cap_to = cap;
	}
	a.cap = cap;
	a.ok1 = e->v_ok.p;
	a.rvec = e->v_rvec.p;
	a.tvec = e->v_tvec.p;
	a.cam = CamK{p->fx, p->fy, p->cx, p->cy};
	a.img_w = p->image_width;
	a.img_h = p->image_height;
	a.win = static_cast<float>(p->guess_win_size);
	a.nndr = p->nndr;
	a.obj = e->v_obj.p;
	a.img = e->v_img.p;
	a.obj_to = e->pnp_has_obj_to ? e->v_obj_to.p : nullptr;
	a.match_id = e->v_mid.p;
	a.match_from = e->v_mfrom.p;
	a.match_to = e->v_mto.p;
	a.n_match = e->v_nm.p;
	const size_t smem = guess_smem_bytes(cap);
	if (smem > static_cast<size_t>(e->smem_optin)) LCD_FAIL(e, LCD_ERR_CAPACITY, "cap %d needs %zu B of shared memory", cap, smem);
#define LCD_GUESS_CASE(NW_)                                                                                              \
	case NW_:                                                                                                            \
	{                                                                                                                    \
		auto kern = guess_match_kernel<NW_>;                                                                             \
		if (smem > 48 * 1024)                                                                                            \
			LCD_CUDA(e, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem))); \
		prof_mark(e, LCD_PROF_MATCH, s);                                                                                 \
		kern<<<n_pairs, 256, smem, s>>>(a);                                                                              \
		prof_mark(e, LCD_PROF_MATCH, s);                                                                                 \
		break;                                                                                                           \
	}
	switch (e->nw)
	{
		LCD_GUESS_CASE(4)
		LCD_GUESS_CASE(8)
		LCD_GUESS_CASE(16)
	default: LCD_FAIL(e, LCD_ERR_INVALID, "unsupported descriptor size");
	}
#undef LCD_GUESS_CASE
	LCD_CHECK_LAUNCH(e);
	return launch_pnp(e, n_pairs, cap, p, s);
}

// copy the per-pair verification outputs back (cap = 0: skip the id arrays)
static int verify_download(lcd_engine * e, int n_pairs, int cap, lcd_verify_result * results, int * match_ids, int * inlier_ids, cudaStream_t s)
{
	const size_t rows = static_cast<size_t>(n_pairs) * cap;
	if (cap > 0 && inlier_ids)
	{
		LCD_CUDA(e, e->v_inl_ids.reserve(rows, 0, false, s));
		gather_by_index_kernel<<<dim3((cap + 255) / 256, n_pairs), 256, 0, s>>>(e->v_mid.p, e->v_inl.p, e->v_ninl.p, cap, e->v_inl_ids.p);
		LCD_CHECK_LAUNCH(e);
	}
	LCD_CUDA(e, e->v_packed.reserve(n_pairs, 0, false, s));
	LCD_CUDA(e, e->h_packed.reserve(n_pairs));
	pack_verify_results_kernel<<<(n_pairs + 127) / 128, 128, 0, s>>>(n_pairs, e->v_ok.p, e->v_nm.p, e->v_ninl.p, e->v_iters.p, e->v_rvec.p, e->v_tvec.p,
	                                                                e->v_T.p, e->v_cov6.p, e->v_packed.p);
	LCD_CHECK_LAUNCH(e);
	LCD_CUDA(e, cudaMemcpyAsync(e->h_packed.p, e->v_packed.p, n_pairs * sizeof(PackedVerifyResult), cudaMemcpyDeviceToHost, s));
	if (cap > 0 && match_ids) LCD_CUDA(e, cudaMemcpyAsync(match_ids, e->v_mid.p, rows * sizeof(int), cudaMemcpyDeviceToHost, s));
	if (cap > 0 && inlier_ids) LCD_CUDA(e, cudaMemcpyAsync(inlier_ids, e->v_inl_ids.p, rows * sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	static_assert(sizeof(PackedVerifyResult) == sizeof(lcd_verify_result), "PackedVerifyResult must mirror lcd_verify_result");
	memcpy(results, e->h_packed.p, n_pairs * sizeof(lcd_verify_result));
	return LCD_OK;
}

static int check_verify_args(lcd_engine * e, int n_pairs, int cap, const void * a, const void * b, const int * na, const int * nb)
{
	if (n_pairs <= 0 || cap <= 0 || !a || !b || !na || !nb) LCD_FAIL(e, LCD_ERR_INVALID, "null or empty verification input");
	if (cap > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "at most %d features per signature", kMaxFrameQueries);
	return LCD_OK;
}

int lcd_match_pairs(lcd_engine * e, int n_pairs, int cap, const void * desc_from, const int * n_from, const void * desc_to,
                    const int * n_to, float nndr, int * from_ids, int * to_ids)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(require_binary(e, "lcd_match_pairs"));
	LCD_TRY(set_device(e));
	LCD_TRY(check_verify_args(e, n_pairs, cap, desc_from, desc_to, n_from, n_to));
	cudaStream_t s = e->stream;
	LCD_TRY(verify_upload(e, n_pairs, cap, desc_from, nullptr, n_from, desc_to, nullptr, n_to, s));
	e->match_has_xyz_to = false;
	LCD_TRY(launch_match(e, n_pairs, cap, nndr, true, s));
	const size_t rows = static_cast<size_t>(n_pairs) * cap;
	if (from_ids) LCD_CUDA(e, cudaMemcpyAsync(from_ids, e->v_fid.p, rows * sizeof(int), cudaMemcpyDeviceToHost, s));
	if (to_ids) LCD_CUDA(e, cudaMemcpyAsync(to_ids, e->v_tid.p, rows * sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	return LCD_OK;
}

int lcd_verify_batch(lcd_engine * e, int n_pairs, int cap, const void * desc_from, const float * xyz_from, const int * n_from,
                     const void * desc_to, const float * uv_to, const float * xyz_to, const int * n_to, const lcd_verify_params * params,
                     lcd_verify_result * results, int * match_ids, int * inlier_ids)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(require_binary(e, "lcd_verify_batch"));
	LCD_TRY(set_device(e));
	LCD_TRY(check_verify_args(e, n_pairs, cap, desc_from, desc_to, n_from, n_to));
	if (!xyz_from || !uv_to || !params || !results) LCD_FAIL(e, LCD_ERR_INVALID, "null verification argument");
	if (params->iterations > kMaxRansacIters) LCD_FAIL(e, LCD_ERR_CAPACITY, "Vis/Iterations > %d", kMaxRansacIters);
	cudaStream_t s = e->stream;
	LCD_TRY(verify_upload(e, n_pairs, cap, desc_from, xyz_from, n_from, desc_to, uv_to, n_to, s, xyz_to));
	e->match_has_xyz_to = xyz_to != nullptr;
	LCD_TRY(launch_match(e, n_pairs, cap, params->nndr, false, s));
	LCD_TRY(launch_pnp(e, n_pairs, cap, params, s));
	LCD_TRY(launch_second_pass(e, n_pairs, cap, params, s, nullptr));
	return verify_download(e, n_pairs, cap, results, match_ids, inlier_ids, s);
}

// ---- stand-alone PnP RANSAC: util3d::solvePnPRansac ------------------------------------------------
static int check_pnp_camera(lcd_engine * e, const double K[9], const double * dist_coeffs, int n_dist, int flags)
{
	if (!K) LCD_FAIL(e, LCD_ERR_INVALID, "null camera matrix");
	if (K[1] != 0.0 || K[3] != 0.0 || K[6] != 0.0 || K[7] != 0.0 || K[8] != 1.0 || !(K[0] > 0.0) || !(K[4] > 0.0))
		LCD_FAIL(e, LCD_ERR_INVALID, "camera matrix must be [fx 0 cx; 0 fy cy; 0 0 1]");
	for (int i = 0; i < n_dist; ++i)
		if (dist_coeffs && dist_coeffs[i] != 0.0)
			LCD_FAIL(e, LCD_ERR_INVALID, "distortion coefficients are not supported: rectify first (CameraModel::D() is zero for rectified images, CameraModel.h:111)");
	if (flags != 0) LCD_FAIL(e, LCD_ERR_INVALID, "Vis/PnPFlags=%d is not implemented (0 = cv::SOLVEPNP_ITERATIVE only)", flags);
	return LCD_OK;
}

int lcd_pnp_ransac_batch(lcd_engine * e, int n_sets, int cap, const float * object_points, const float * image_points, const int * n_points,
                         const double K[9], const double * dist_coeffs, int n_dist, double * rvec, double * tvec, int use_extrinsic_guess,
                         int iterations, float reproj_error, int min_inliers, int flags, int refine_iterations, float refine_sigma,
                         int * inliers_out, int * n_inliers_out, int * iterations_run_out)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (n_sets <= 0 || cap <= 0 || !object_points || !image_points || !n_points || !rvec || !tvec) LCD_FAIL(e, LCD_ERR_INVALID, "null or empty PnP input");
	if (cap > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "at most %d correspondences per set", kMaxFrameQueries);
	LCD_TRY(check_pnp_camera(e, K, dist_coeffs, n_dist, flags));
	if (iterations > kMaxRansacIters) LCD_FAIL(e, LCD_ERR_CAPACITY, "iterationsCount > %d", kMaxRansacIters);
	for (int i = 0; i < n_sets; ++i)
	{
		if (n_points[i] < 0 || n_points[i] > cap) LCD_FAIL(e, LCD_ERR_INVALID, "set %d has %d points (cap %d)", i, n_points[i], cap);
		// cv3::solvePnPRansac switches to P3P on exactly four points (opencv/solvepnp.cpp:150-154): not implemented
		if (n_points[i] == 4) LCD_FAIL(e, LCD_ERR_INVALID, "set %d has exactly 4 points: the reference solves it with P3P, which is not implemented", i);
	}
	(void)use_extrinsic_guess; // the RANSAC kernel is EPnP on 6 points, which ignores the guess; on failure rvec / tvec are left untouched
	cudaStream_t s = e->stream;
	const size_t rows = static_cast<size_t>(n_sets) * cap;
	LCD_CUDA(e, e->v_obj.reserve(rows * 3, 0, false, s));
	LCD_CUDA(e, e->v_img.reserve(rows * 2, 0, false, s));
	LCD_CUDA(e, e->v_nm.reserve(n_sets, 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->v_obj.p, object_points, rows * 3 * sizeof(float), cudaMemcpyHostToDevice, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->v_img.p, image_points, rows * 2 * sizeof(float), cudaMemcpyHostToDevice, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->v_nm.p, n_points, n_sets * sizeof(int), cudaMemcpyHostToDevice, s));
	lcd_verify_params vp{};
	vp.min_inliers = min_inliers;
	vp.iterations = iterations;
	vp.reproj_error = reproj_error;
	vp.refine_iterations = refine_iterations;
	vp.refine_sigma = refine_sigma;
	vp.fx = K[0];
	vp.fy = K[4];
	vp.cx = K[2];
	vp.cy = K[5];
	vp.var_median_ratio = 2;
	LCD_TRY(launch_pnp(e, n_sets, cap, &vp, s, false, false));
	std::vector<double> hr(static_cast<size_t>(n_sets) * 3), ht(static_cast<size_t>(n_sets) * 3);
	std::vector<int> hn(n_sets), hit(n_sets);
	LCD_CUDA(e, cudaMemcpyAsync(hr.data(), e->v_rvec.p, hr.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaMemcpyAsync(ht.data(), e->v_tvec.p, ht.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaMemcpyAsync(hn.data(), e->v_ninl.p, n_sets * sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaMemcpyAsync(hit.data(), e->v_iters.p, n_sets * sizeof(int), cudaMemcpyDeviceToHost, s));
	if (inliers_out) LCD_CUDA(e, cudaMemcpyAsync(inliers_out, e->v_inl.p, rows * sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	for (int i = 0; i < n_sets; ++i)
	{
		// a model was found (the kernel zeroes the pose first and writes the final model last): rvec / tvec of the (refined) model;
		// otherwise the caller's values stay, as when cv3::solvePnPRansac returns false (solvepnp.cpp:183-192)
		bool found = hn[i] > 0;
		for (int k = 0; k < 3; ++k) found = found || hr[3 * i + k] != 0.0 || ht[3 * i + k] != 0.0;
		if (found)
		{
			for (int k = 0; k < 3; ++k)
			{
				rvec[3 * i + k] = hr[3 * i + k];
				tvec[3 * i + k] = ht[3 * i + k];
			}
		}
		if (n_inliers_out) n_inliers_out[i] = hn[i];
		if (iterations_run_out) iterations_run_out[i] = hit[i];
	}
	return LCD_OK;
}

int lcd_pnp_ransac(lcd_engine * e, const float * object_points, const float * image_points, int n, const double K[9], const double * dist_coeffs,
                   int n_dist, double rvec[3], double tvec[3], int use_extrinsic_guess, int iterations, float reproj_error, int min_inliers,
                   int flags, int refine_iterations, float refine_sigma, int * inliers_out, int * n_inliers_out)
{
	if (!e) return LCD_ERR_INVALID;
	if (n <= 0)
	{
		if (n_inliers_out) *n_inliers_out = 0;
		return LCD_OK;
	}
	return lcd_pnp_ransac_batch(e, 1, n, object_points, image_points, &n, K, dist_coeffs, n_dist, rvec, tvec, use_extrinsic_guess, iterations,
	                            reproj_error, min_inliers, flags, refine_iterations, refine_sigma, inliers_out, n_inliers_out, nullptr);
}

// ---- brute-force matching of two descriptor sets: cv::BFMatcher ----------------------------------------
} // extern "C"
template <int NW, bool F32>
static int launch_bf(lcd_engine * e, int n_pairs, int cap, const uint32_t * A, const int * nA, const uint32_t * B, const int * nB, ulonglong2 * keys,
                     cudaStream_t s)
{
	dim3 grid((cap + kBfThreads - 1) / kBfThreads, n_pairs);
	prof_mark(e, LCD_PROF_MATCH, s);
	bf_knn2_kernel<NW, F32><<<grid, kBfThreads, 0, s>>>(A, nA, B, nB, cap, keys);
	prof_mark(e, LCD_PROF_MATCH, s);
	LCD_CHECK_LAUNCH(e);
	return LCD_OK;
}

static int launch_bf_any(lcd_engine * e, int n_pairs, int cap, const uint32_t * A, const int * nA, const uint32_t * B, const int * nB,
                         ulonglong2 * keys, cudaStream_t s)
{
	if (e->f32) return e->nw == 64 ? launch_bf<64, true>(e, n_pairs, cap, A, nA, B, nB, keys, s) : launch_bf<128, true>(e, n_pairs, cap, A, nA, B, nB, keys, s);
	switch (e->nw)
	{
	case 4: return launch_bf<4, false>(e, n_pairs, cap, A, nA, B, nB, keys, s);
	case 8: return launch_bf<8, false>(e, n_pairs, cap, A, nA, B, nB, keys, s);
	case 16: return launch_bf<16, false>(e, n_pairs, cap, A, nA, B, nB, keys, s);
	default: LCD_FAIL(e, LCD_ERR_INVALID, "unsupported descriptor size");
	}
}

extern "C" {
int lcd_match_bf(lcd_engine * e, int n_pairs, int cap, const void * desc_query, const int * n_query, const void * desc_train, const int * n_train,
                 int mode, int * idx1, float * dist1, int * idx2, float * dist2)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	LCD_TRY(check_verify_args(e, n_pairs, cap, desc_query, desc_train, n_query, n_train));
	if (mode != LCD_MATCH_KNN2 && mode != LCD_MATCH_CROSSCHECK) LCD_FAIL(e, LCD_ERR_INVALID, "mode must be LCD_MATCH_KNN2 or LCD_MATCH_CROSSCHECK");
	if (!idx1 || !dist1 || (mode == LCD_MATCH_KNN2 && (!idx2 || !dist2))) LCD_FAIL(e, LCD_ERR_INVALID, "null output");
	cudaStream_t s = e->stream;
	const size_t rows = static_cast<size_t>(n_pairs) * cap;
	// FROM buffers hold the train side, TO buffers the query side (cv::BFMatcher::match(queryDescriptors = TO, trainDescriptors = FROM))
	LCD_TRY(verify_upload(e, n_pairs, cap, desc_train, nullptr, n_train, desc_query, nullptr, n_query, s));
	LCD_CUDA(e, e->bf_keys_a.reserve(rows, 0, false, s));
	LCD_CUDA(e, e->d_i1.reserve(rows, 0, false, s));
	LCD_CUDA(e, e->d_f1.reserve(rows, 0, false, s));
	const int nb = static_cast<int>((rows + 255) / 256);
	if (mode == LCD_MATCH_KNN2)
	{
		LCD_TRY(launch_bf_any(e, n_pairs, cap, e->v_dt.p, e->v_nt.p, e->v_df.p, e->v_nf.p, e->bf_keys_a.p, s));
		LCD_CUDA(e, e->d_i2.reserve(rows, 0, false, s));
		LCD_CUDA(e, e->d_f2.reserve(rows, 0, false, s));
		const unsigned long long * k = reinterpret_cast<const unsigned long long *>(e->bf_keys_a.p);
		if (e->f32)
		{
			bf_decode_kernel<true><<<nb, 256, 0, s>>>(k, 2, 0, static_cast<int>(rows), e->d_i1.p, e->d_f1.p);
			bf_decode_kernel<true><<<nb, 256, 0, s>>>(k, 2, 1, static_cast<int>(rows), e->d_i2.p, e->d_f2.p);
		}
		else
		{
			bf_decode_kernel<false><<<nb, 256, 0, s>>>(k, 2, 0, static_cast<int>(rows), e->d_i1.p, e->d_f1.p);
			bf_decode_kernel<false><<<nb, 256, 0, s>>>(k, 2, 1, static_cast<int>(rows), e->d_i2.p, e->d_f2.p);
		}
		LCD_CHECK_LAUNCH(e);
		++e->launches;
		LCD_CUDA(e, cudaMemcpyAsync(idx2, e->d_i2.p, rows * sizeof(int), cudaMemcpyDeviceToHost, s));
		LCD_CUDA(e, cudaMemcpyAsync(dist2, e->d_f2.p, rows * sizeof(float), cudaMemcpyDeviceToHost, s));
	}
	else
	{
		// nearest train row of every query, nearest query of every train row, then the mutual test
		LCD_TRY(launch_bf_any(e, n_pairs, cap, e->v_dt.p, e->v_nt.p, e->v_df.p, e->v_nf.p, e->bf_keys_a.p, s));
		LCD_CUDA(e, e->bf_keys_b.reserve(rows, 0, false, s));
		LCD_TRY(launch_bf_any(e, n_pairs, cap, e->v_df.p, e->v_nf.p, e->v_dt.p, e->v_nt.p, e->bf_keys_b.p, s));
		LCD_CUDA(e, e->bf_best.reserve(rows, 0, false, s));
		bf_cross_kernel<<<dim3((cap + 255) / 256, n_pairs), 256, 0, s>>>(e->bf_keys_a.p, e->bf_keys_b.p, e->v_nt.p, cap, e->bf_best.p);
		LCD_CHECK_LAUNCH(e);
		if (e->f32) bf_decode_kernel<true><<<nb, 256, 0, s>>>(e->bf_best.p, 1, 0, static_cast<int>(rows), e->d_i1.p, e->d_f1.p);
		else bf_decode_kernel<false><<<nb, 256, 0, s>>>(e->bf_best.p, 1, 0, static_cast<int>(rows), e->d_i1.p, e->d_f1.p);
		LCD_CHECK_LAUNCH(e);
	}
	LCD_CUDA(e, cudaMemcpyAsync(idx1, e->d_i1.p, rows * sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaMemcpyAsync(dist1, e->d_f1.p, rows * sizeof(float), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	if (mode == LCD_MATCH_KNN2)
	{
		// rows past a pair's query count were not written by the kernel: report them as "no match"
		for (int p = 0; p < n_pairs; ++p)
			for (int i = std::max(0, std::min(n_query[p], cap)); i < cap; ++i)
			{
				const size_t r = static_cast<size_t>(p) * cap + i;
				idx1[r] = idx2[r] = -1;
				dist1[r] = dist2[r] = -1.0f;
			}
	}
	return LCD_OK;
}

// ---- signature store + fused query -------------------------------------------------------------
int lcd_sig_count(const lcd_engine * e) { return e ? e->st_slots - static_cast<int>(e->free_slots.size()) : 0; }
int lcd_sig_slots(const lcd_engine * e) { return e ? e->st_slots : 0; }

int lcd_sig_add_batch(lcd_engine * e, const int * sig_ids, int n_sigs, int cap, const void * desc, const float * xyz, const int * n)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(require_binary(e, "lcd_sig_add_batch"));
	if (n_sigs <= 0) return LCD_OK;
	if (!sig_ids || !desc || !xyz || !n || cap <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "null signature data");
	if (cap > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "at most %d features per signature", kMaxFrameQueries);
	LCD_TRY(set_device(e));
	cudaStream_t s = e->stream;
	if (e->st_cap == 0) e->st_cap = cap;
	if (cap != e->st_cap) LCD_FAIL(e, LCD_ERR_INVALID, "signature store was created with %d rows per signature, got %d", e->st_cap, cap);
	int max_id = 0;
	for (int i = 0; i < n_sigs; ++i)
	{
		if (sig_ids[i] <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "signature id must be positive");
		max_id = std::max(max_id, sig_ids[i]);
	}
	if (static_cast<size_t>(max_id) + 1 > e->h_slot_of_sig.size())
	{
		const size_t old = e->h_slot_of_sig.size();
		const size_t ncap = std::max<size_t>(max_id + 1, old + old / 2 + 1024);
		e->h_slot_of_sig.resize(ncap, -1);
	}
	// slots: freed slots are reused first (one add + one remove per frame is what the WM -> LTM transfer produces: the store must
	// not grow); the bulk copy is used when the slots happen to be consecutive
	const size_t prev_slots = static_cast<size_t>(e->st_slots);
	std::vector<int> slots(n_sigs);
	bool contiguous = true;
	for (int i = 0; i < n_sigs; ++i)
	{
		int slot = e->h_slot_of_sig[sig_ids[i]];
		if (slot < 0)
		{
			if (!e->free_slots.empty())
			{
				slot = e->free_slots.back();
				e->free_slots.pop_back();
			}
			else slot = e->st_slots++;
		}
		slots[i] = slot;
		if (i > 0 && slots[i] != slots[i - 1] + 1) contiguous = false;
		e->h_slot_of_sig[sig_ids[i]] = slot;
	}
	LCD_CUDA(e, e->st_desc.reserve(static_cast<size_t>(e->st_slots) * cap * e->nw, prev_slots * cap * e->nw, false, s));
	LCD_CUDA(e, e->st_xyz.reserve(static_cast<size_t>(e->st_slots) * cap * 3, prev_slots * cap * 3, false, s));
	LCD_CUDA(e, e->st_n.reserve(static_cast<size_t>(e->st_slots), prev_slots, true, s));
	const size_t drow = static_cast<size_t>(cap) * e->nw * 4, xrow = static_cast<size_t>(cap) * 3 * sizeof(float);
	if (contiguous)
	{
		LCD_CUDA(e, cudaMemcpyAsync(e->st_desc.p + static_cast<size_t>(slots[0]) * cap * e->nw, desc, drow * n_sigs, cudaMemcpyHostToDevice, s));
		LCD_CUDA(e, cudaMemcpyAsync(e->st_xyz.p + static_cast<size_t>(slots[0]) * cap * 3, xyz, xrow * n_sigs, cudaMemcpyHostToDevice, s));
		LCD_CUDA(e, cudaMemcpyAsync(e->st_n.p + slots[0], n, n_sigs * sizeof(int), cudaMemcpyHostToDevice, s));
	}
	else
	{
		for (int i = 0; i < n_sigs; ++i)
		{
			LCD_CUDA(e, cudaMemcpyAsync(e->st_desc.p + static_cast<size_t>(slots[i]) * cap * e->nw, static_cast<const char *>(desc) + drow * i, drow, cudaMemcpyHostToDevice, s));
			LCD_CUDA(e, cudaMemcpyAsync(e->st_xyz.p + static_cast<size_t>(slots[i]) * cap * 3, xyz + static_cast<size_t>(i) * cap * 3, xrow, cudaMemcpyHostToDevice, s));
			LCD_CUDA(e, cudaMemcpyAsync(e->st_n.p + slots[i], n + i, sizeof(int), cudaMemcpyHostToDevice, s));
		}
	}
	LCD_CUDA(e, e->st_slot_of_sig.reserve(e->h_slot_of_sig.size(), 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->st_slot_of_sig.p, e->h_slot_of_sig.data(), e->h_slot_of_sig.size() * sizeof(int), cudaMemcpyHostToDevice, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	return LCD_OK;
}

int lcd_sig_remove(lcd_engine * e, int sig_id)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (sig_id <= 0 || sig_id >= static_cast<int>(e->h_slot_of_sig.size()) || e->h_slot_of_sig[sig_id] < 0) return LCD_OK;
	const int slot = e->h_slot_of_sig[sig_id];
	e->h_slot_of_sig[sig_id] = -1;
	e->free_slots.push_back(slot);
	const int minus1 = -1;
	LCD_CUDA(e, cudaMemcpyAsync(e->st_slot_of_sig.p + sig_id, &minus1, sizeof(int), cudaMemcpyHostToDevice, e->stream));
	LCD_CUDA(e, cudaMemsetAsync(e->st_n.p + slot, 0, sizeof(int), e->stream));
	LCD_CUDA(e, cudaStreamSynchronize(e->stream));
	return LCD_OK;
}

static int verify_top_dev(lcd_engine * e, const uint32_t * d_q, const float * d_uv, int n_frames, int nq, const float * d_like,
                          const int * d_sig_ids, int ns, const lcd_verify_params * vp, cudaStream_t s, const int * d_nq_frame = nullptr,
                          const float * d_xyz_to = nullptr);

static int process_dev(lcd_engine * e, const uint32_t * d_q, const float * d_uv, int n_frames, int nq, int incremental, float nndr, int cmp_new,
                       const int * d_sig_ids, int ns, int n_total, const lcd_verify_params * vp, int * d_words, float * d_like, cudaStream_t s)
{
	if (!vp) LCD_FAIL(e, LCD_ERR_INVALID, "null verification parameters");
	if (vp->iterations > kMaxRansacIters) LCD_FAIL(e, LCD_ERR_CAPACITY, "Vis/Iterations > %d", kMaxRansacIters);
	if (e->st_cap == 0) LCD_FAIL(e, LCD_ERR_STATE, "the signature store is empty: nothing to verify against");
	if (!d_sig_ids || ns <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "ids list is empty");
	if (!d_like)
	{
		LCD_CUDA(e, e->d_like.reserve(static_cast<size_t>(n_frames) * ns, 0, false, s));
		d_like = e->d_like.p;
	}
	LCD_TRY(localize_dev(e, d_q, n_frames, nq, incremental, nndr, cmp_new, d_sig_ids, ns, n_total, d_words, d_like, s));
	return verify_top_dev(e, d_q, d_uv, n_frames, nq, d_like, d_sig_ids, ns, vp, s);
}

static int verify_top_dev(lcd_engine * e, const uint32_t * d_q, const float * d_uv, int n_frames, int nq, const float * d_like,
                          const int * d_sig_ids, int ns, const lcd_verify_params * vp, cudaStream_t s, const int * d_nq_frame, const float * d_xyz_to)
{
	if (!vp) LCD_FAIL(e, LCD_ERR_INVALID, "null verification parameters");
	if (vp->iterations > kMaxRansacIters) LCD_FAIL(e, LCD_ERR_CAPACITY, "Vis/Iterations > %d", kMaxRansacIters);
	if (e->st_cap == 0) LCD_FAIL(e, LCD_ERR_STATE, "the signature store is empty: nothing to verify against");
	LCD_CUDA(e, e->d_hyp_id.reserve(n_frames, 0, false, s));
	LCD_CUDA(e, e->d_hyp_slot.reserve(n_frames, 0, false, s));
	argmax_hypothesis_kernel<<<n_frames, 256, 0, s>>>(d_like, ns, d_sig_ids, e->st_slot_of_sig.p, static_cast<int>(e->h_slot_of_sig.size()),
	                                                  e->d_hyp_id.p, e->d_hyp_slot.p);
	LCD_CHECK_LAUNCH(e);
	const int cap = std::max(e->st_cap, nq);
	MatchSrc src{e->st_desc.p, e->st_xyz.p, e->st_n.p, e->d_hyp_slot.p, e->st_cap, d_q, d_uv, d_nq_frame, nq, nq, d_xyz_to};
	LCD_TRY(launch_match(e, n_frames, cap, vp->nndr, false, s, &src));
	LCD_TRY(launch_pnp(e, n_frames, cap, vp, s));
	return launch_second_pass(e, n_frames, cap, vp, s, &src);
}

int lcd_process_batch_dev(lcd_engine * e, const void * d_queries, const float * d_uv, int n_frames, int nq_per_frame, int incremental, float nndr,
                          int new_words_compared_together, const int * d_sig_ids, int ns, int n_total, const lcd_verify_params * vp,
                          int * d_word_ids_out, float * d_likelihood_out, void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(require_binary(e, "lcd_process_batch_dev"));
	LCD_TRY(set_device(e));
	if (!d_queries || !d_uv || n_frames <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "Descriptors size is null!");
	if (nq_per_frame <= 0 || nq_per_frame > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "1..%d descriptors per frame", kMaxFrameQueries);
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	return process_dev(e, static_cast<const uint32_t *>(d_queries), d_uv, n_frames, nq_per_frame, incremental, nndr, new_words_compared_together,
	                   d_sig_ids, ns, n_total, vp, d_word_ids_out, d_likelihood_out, s);
}

// images -> detect -> quantise -> score -> verify, all on device buffers
static int process_frames_dev(lcd_engine * e, int n_frames, const uint8_t * d_images, int width, int height, int channels, const void * d_depth,
                              int depth_type, const lcd_orb_params * op, int incremental, float nndr, int cmp_new, const int * d_sig_ids, int ns,
                              int n_total, const lcd_verify_params * vp, int * d_words, float * d_like, cudaStream_t s,
                              const uint8_t * h_images = nullptr, const void * h_depth = nullptr)
{
	if (!op) LCD_FAIL(e, LCD_ERR_INVALID, "null ORB parameters");
	if (e->cfg.desc_type != LCD_DESC_U8 || e->cfg.desc_dim != 32) LCD_FAIL(e, LCD_ERR_INVALID, "ORB descriptors need an engine with 32-byte binary descriptors");
	const int cap = op->n_features;
	if (cap <= 0 || cap > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "Kp/MaxFeatures must be 1..%d", kMaxFrameQueries);
	const size_t rows = static_cast<size_t>(n_frames) * cap;
	LCD_CUDA(e, e->o_kp.reserve(rows, 0, false, s));
	LCD_CUDA(e, e->o_desc.reserve(rows * 32, 0, false, s));
	LCD_CUDA(e, e->o_xyz.reserve(rows * 3, 0, false, s));
	LCD_CUDA(e, e->o_uv.reserve(rows * 2, 0, false, s));
	LCD_CUDA(e, e->o_n.reserve(n_frames, 0, false, s));
	// padding rows of short frames must hold defined bytes for the NN kernel
	LCD_CUDA(e, zero_fill_async(e->o_desc.p, rows * 32, s));
	if (!h_images)
	{
		LCD_TRY(orb_run(e, n_frames, d_images, width, height, channels, d_depth, depth_type, op, cap, e->o_kp.p, e->o_desc.p, e->o_xyz.p, e->o_uv.p,
		                e->o_n.p, s));
	}
	else
	{
		// host frames: upload in chunks on the copy stream and run detect + describe on each chunk as soon as it has
		// landed, so that the PCIe transfer of chunk c+1 hides behind the ORB kernels of chunk c
		if (!e->copy_stream)
		{
			LCD_CUDA(e, cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
			LCD_CUDA(e, cudaEventCreateWithFlags(&e->copy_fence, cudaEventDisableTiming));
		}
		const int chunk_env = env_int("LCD_UPLOAD_CHUNK", 0); // 0: one chunk (per-chunk ORB launches are latency-bound, measured: chunking only pays for very large batches)
		const int chunk = chunk_env > 0 ? chunk_env : n_frames;
		const int n_chunks = (n_frames + chunk - 1) / chunk;
		while (static_cast<int>(e->copy_events.size()) < n_chunks)
		{
			cudaEvent_t ev;
			LCD_CUDA(e, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
			e->copy_events.push_back(ev);
		}
		const size_t px = static_cast<size_t>(width) * height;
		const size_t dbytes = depth_elem_bytes(depth_type);
		// the device staging buffers may still be read by work queued on s (a previous call): order the copies after it
		LCD_CUDA(e, cudaEventRecord(e->copy_fence, s));
		LCD_CUDA(e, cudaStreamWaitEvent(e->copy_stream, e->copy_fence, 0));
		for (int c = 0; c < n_chunks; ++c)
		{
			const int f0 = c * chunk, nf = std::min(chunk, n_frames - f0);
			LCD_CUDA(e, cudaMemcpyAsync(const_cast<uint8_t *>(d_images) + f0 * px * channels, h_images + f0 * px * channels, nf * px * channels,
			                            cudaMemcpyHostToDevice, e->copy_stream));
			if (h_depth && d_depth)
				LCD_CUDA(e, cudaMemcpyAsync(static_cast<unsigned char *>(const_cast<void *>(d_depth)) + f0 * px * dbytes,
				                            static_cast<const unsigned char *>(h_depth) + f0 * px * dbytes, nf * px * dbytes, cudaMemcpyHostToDevice,
				                            e->copy_stream));
			LCD_CUDA(e, cudaEventRecord(e->copy_events[c], e->copy_stream));
		}
		for (int c = 0; c < n_chunks; ++c)
		{
			const int f0 = c * chunk, nf = std::min(chunk, n_frames - f0);
			LCD_CUDA(e, cudaStreamWaitEvent(s, e->copy_events[c], 0));
			LCD_TRY(orb_run(e, nf, d_images, width, height, channels, d_depth, depth_type, op, cap, e->o_kp.p, e->o_desc.p, e->o_xyz.p, e->o_uv.p,
			                e->o_n.p, s, f0, n_frames));
		}
	}
	if (!d_like)
	{
		LCD_CUDA(e, e->d_like.reserve(static_cast<size_t>(n_frames) * ns, 0, false, s));
		d_like = e->d_like.p;
	}
	const uint32_t * d_q = reinterpret_cast<const uint32_t *>(e->o_desc.p);
	LCD_TRY(localize_dev(e, d_q, n_frames, cap, incremental, nndr, cmp_new, d_sig_ids, ns, n_total, d_words, d_like, s, e->o_n.p));
	if (vp) LCD_TRY(verify_top_dev(e, d_q, e->o_uv.p, n_frames, cap, d_like, d_sig_ids, ns, vp, s, e->o_n.p, e->o_xyz.p));
	return LCD_OK;
}

int lcd_process_frames_dev(lcd_engine * e, int n_frames, const uint8_t * d_images, int width, int height, int channels, const void * d_depth,
                           int depth_type, const lcd_orb_params * op, int incremental, float nndr, int new_words_compared_together,
                           const int * d_sig_ids, int ns, int n_total, const lcd_verify_params * vp, int * d_word_ids_out,
                           float * d_likelihood_out, void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!d_images || n_frames <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "null image");
	if (!d_sig_ids || ns <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "ids list is empty");
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	return process_frames_dev(e, n_frames, d_images, width, height, channels, d_depth, depth_type, op, incremental, nndr, new_words_compared_together,
	                          d_sig_ids, ns, n_total, vp, d_word_ids_out, d_likelihood_out, s);
}

int lcd_process_frames(lcd_engine * e, int n_frames, const uint8_t * images, int width, int height, int channels, const void * depth, int depth_type,
                       const lcd_orb_params * op, int incremental, float nndr, int new_words_compared_together, const int * sig_ids, int ns,
                       int n_total, const lcd_verify_params * vp, int * n_kp_out, int * word_ids_out, float * likelihood_out, int * hypothesis_out,
                       lcd_verify_result * results)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!images || n_frames <= 0 || width <= 0 || height <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "null image");
	if (!sig_ids || ns <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "ids list is empty");
	if (!op) LCD_FAIL(e, LCD_ERR_INVALID, "null ORB parameters");
	cudaStream_t s = e->stream;
	const size_t px = static_cast<size_t>(n_frames) * width * height;
	LCD_CUDA(e, e->o_img.reserve(px * channels, 0, false, s));
	if (!depth) depth_type = LCD_DEPTH_NONE;
	if (depth_type != LCD_DEPTH_NONE)
	{
		const size_t dbytes = depth_elem_bytes(depth_type);
		LCD_CUDA(e, e->o_depth.reserve(px * dbytes, 0, false, s));
	}
	// the frames themselves are uploaded chunk by chunk inside process_frames_dev, overlapped with detect + describe
	const int cap = op->n_features;
	const size_t rows = static_cast<size_t>(n_frames) * std::max(cap, 1);
	LCD_CUDA(e, e->d_sig_ids.reserve(ns, 0, false, s));
	LCD_CUDA(e, e->d_like.reserve(static_cast<size_t>(n_frames) * ns, 0, false, s));
	LCD_CUDA(e, e->d_word_ids.reserve(rows, 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->d_sig_ids.p, sig_ids, ns * sizeof(int), cudaMemcpyHostToDevice, s));
	LCD_TRY(process_frames_dev(e, n_frames, e->o_img.p, width, height, channels, depth_type != LCD_DEPTH_NONE ? e->o_depth.p : nullptr, depth_type, op,
	                           incremental, nndr, new_words_compared_together, e->d_sig_ids.p, ns, n_total, vp, e->d_word_ids.p, e->d_like.p, s, images,
	                           depth_type != LCD_DEPTH_NONE ? depth : nullptr));
	if (n_kp_out) LCD_CUDA(e, cudaMemcpyAsync(n_kp_out, e->o_n.p, n_frames * sizeof(int), cudaMemcpyDeviceToHost, s));
	if (word_ids_out) LCD_CUDA(e, cudaMemcpyAsync(word_ids_out, e->d_word_ids.p, rows * sizeof(int), cudaMemcpyDeviceToHost, s));
	if (likelihood_out)
		LCD_CUDA(e, cudaMemcpyAsync(likelihood_out, e->d_like.p, static_cast<size_t>(n_frames) * ns * sizeof(float), cudaMemcpyDeviceToHost, s));
	if (vp && hypothesis_out) LCD_CUDA(e, cudaMemcpyAsync(hypothesis_out, e->d_hyp_id.p, n_frames * sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, e->h_overflow.reserve(1));
	LCD_CUDA(e, cudaMemcpyAsync(e->h_overflow.p, e->o_overflow.p, sizeof(int), cudaMemcpyDeviceToHost, s));
	if (vp && results) LCD_TRY(verify_download(e, n_frames, 0, results, nullptr, nullptr, s));
	LCD_CUDA(e, cudaStreamSynchronize(s));
	if (*e->h_overflow.p) return detect_overflow(e);
	return LCD_OK;
}

// ---- pipelined host path: two batches in flight ------------------------------------------------------------
int lcd_process_frames_submit(lcd_engine * e, int n_frames, const uint8_t * images, int width, int height, int channels, const void * depth,
                              int depth_type, const lcd_orb_params * op, int incremental, float nndr, int new_words_compared_together,
                              const int * sig_ids, int ns, int n_total, const lcd_verify_params * vp, int * n_kp_out, int * word_ids_out,
                              float * likelihood_out, int * hypothesis_out, lcd_verify_result * results)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!images || n_frames <= 0 || width <= 0 || height <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "null image");
	if (!sig_ids || ns <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "ids list is empty");
	if (!op) LCD_FAIL(e, LCD_ERR_INVALID, "null ORB parameters");
	if (e->flights_busy >= 2) LCD_FAIL(e, LCD_ERR_INVALID, "two batches are already in flight: call lcd_process_frames_wait first");
	cudaStream_t s = e->stream;
	const int slot = (e->flight_head + e->flights_busy) & 1;
	lcd_engine::Flight & f = e->flights[slot];
	if (!e->copy_stream)
	{
		LCD_CUDA(e, cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
		LCD_CUDA(e, cudaEventCreateWithFlags(&e->copy_fence, cudaEventDisableTiming));
	}
	if (!f.uploaded)
	{
		LCD_CUDA(e, cudaEventCreateWithFlags(&f.uploaded, cudaEventDisableTiming));
		LCD_CUDA(e, cudaEventCreateWithFlags(&f.done, cudaEventDisableTiming));
	}
	const size_t px = static_cast<size_t>(n_frames) * width * height;
	if (!depth) depth_type = LCD_DEPTH_NONE;
	const size_t dbytes = depth_elem_bytes(depth_type);
	// upload on the copy stream: the slot's previous batch was waited for, so its staging buffers are free
	static const int dbg_tl = env_int("LCD_DEBUG_TIMELINE", 0); // diagnostics: print each batch's upload / compute window at _wait
	if (dbg_tl && !f.t_h0)
	{
		cudaEventCreate(&f.t_h0);
		cudaEventCreate(&f.t_h1);
		cudaEventCreate(&f.t_c0);
		cudaEventCreate(&f.t_c1);
		if (!e->t_base)
		{
			cudaEventCreate(&e->t_base);
			cudaEventRecord(e->t_base, e->copy_stream);
		}
	}
	if (dbg_tl) cudaEventRecord(f.t_h0, e->copy_stream);
	LCD_CUDA(e, f.img.reserve(px * channels, 0, false, e->copy_stream));
	LCD_CUDA(e, cudaMemcpyAsync(f.img.p, images, px * channels, cudaMemcpyHostToDevice, e->copy_stream));
	if (depth_type != LCD_DEPTH_NONE)
	{
		LCD_CUDA(e, f.depth.reserve(px * dbytes, 0, false, e->copy_stream));
		LCD_CUDA(e, cudaMemcpyAsync(f.depth.p, depth, px * dbytes, cudaMemcpyHostToDevice, e->copy_stream));
	}
	// the signature id list rides on the copy stream too: a host -> device copy queued on the compute stream would sit in the
	// same copy-engine queue as the next batch's images and serialise the two batches (measured)
	LCD_CUDA(e, f.sig_ids.reserve(ns, 0, false, e->copy_stream));
	LCD_CUDA(e, cudaMemcpyAsync(f.sig_ids.p, sig_ids, ns * sizeof(int), cudaMemcpyHostToDevice, e->copy_stream));
	if (dbg_tl) cudaEventRecord(f.t_h1, e->copy_stream);
	LCD_CUDA(e, cudaEventRecord(f.uploaded, e->copy_stream));
	// compute on the engine stream, behind the previous batch
	const int cap = op->n_features;
	const size_t rows = static_cast<size_t>(n_frames) * std::max(cap, 1);
	LCD_CUDA(e, e->d_like.reserve(static_cast<size_t>(n_frames) * ns, 0, false, s));
	LCD_CUDA(e, e->d_word_ids.reserve(rows, 0, false, s));
	LCD_CUDA(e, cudaStreamWaitEvent(s, f.uploaded, 0));
	if (dbg_tl) cudaEventRecord(f.t_c0, s);
	LCD_TRY(process_frames_dev(e, n_frames, f.img.p, width, height, channels, depth_type != LCD_DEPTH_NONE ? f.depth.p : nullptr, depth_type, op,
	                           incremental, nndr, new_words_compared_together, f.sig_ids.p, ns, n_total, vp, e->d_word_ids.p, e->d_like.p, s));
	if (n_kp_out) LCD_CUDA(e, cudaMemcpyAsync(n_kp_out, e->o_n.p, n_frames * sizeof(int), cudaMemcpyDeviceToHost, s));
	if (word_ids_out) LCD_CUDA(e, cudaMemcpyAsync(word_ids_out, e->d_word_ids.p, rows * sizeof(int), cudaMemcpyDeviceToHost, s));
	if (likelihood_out)
		LCD_CUDA(e, cudaMemcpyAsync(likelihood_out, e->d_like.p, static_cast<size_t>(n_frames) * ns * sizeof(float), cudaMemcpyDeviceToHost, s));
	if (vp && hypothesis_out) LCD_CUDA(e, cudaMemcpyAsync(hypothesis_out, e->d_hyp_id.p, n_frames * sizeof(int), cudaMemcpyDeviceToHost, s));
	f.user_results = nullptr;
	if (vp && results)
	{
		LCD_CUDA(e, e->v_packed.reserve(n_frames, 0, false, s));
		LCD_CUDA(e, f.res.reserve(n_frames));
		pack_verify_results_kernel<<<(n_frames + 127) / 128, 128, 0, s>>>(n_frames, e->v_ok.p, e->v_nm.p, e->v_ninl.p, e->v_iters.p, e->v_rvec.p,
		                                                                 e->v_tvec.p, e->v_T.p, e->v_cov6.p, e->v_packed.p);
		LCD_CHECK_LAUNCH(e);
		LCD_CUDA(e, cudaMemcpyAsync(f.res.p, e->v_packed.p, n_frames * sizeof(PackedVerifyResult), cudaMemcpyDeviceToHost, s));
		f.user_results = results;
	}
	f.n_frames = n_frames;
	LCD_CUDA(e, f.overflow.reserve(1));
	LCD_CUDA(e, cudaMemcpyAsync(f.overflow.p, e->o_overflow.p, sizeof(int), cudaMemcpyDeviceToHost, s));
	if (dbg_tl) cudaEventRecord(f.t_c1, s);
	LCD_CUDA(e, cudaEventRecord(f.done, s));
	++e->flights_busy;
	return LCD_OK;
}

int lcd_process_frames_wait(lcd_engine * e)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (e->flights_busy <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "no batch in flight");
	lcd_engine::Flight & f = e->flights[e->flight_head];
	LCD_CUDA(e, cudaEventSynchronize(f.done));
	if (f.t_h0 && e->t_base)
	{
		float a = 0, b = 0, c = 0, d = 0;
		cudaEventElapsedTime(&a, e->t_base, f.t_h0);
		cudaEventElapsedTime(&b, e->t_base, f.t_h1);
		cudaEventElapsedTime(&c, e->t_base, f.t_c0);
		cudaEventElapsedTime(&d, e->t_base, f.t_c1);
		fprintf(stderr, "[lcd timeline] upload %.2f..%.2f  compute %.2f..%.2f ms\n", a, b, c, d);
	}
	if (f.user_results) memcpy(f.user_results, f.res.p, f.n_frames * sizeof(lcd_verify_result));
	f.user_results = nullptr;
	e->flight_head ^= 1;
	--e->flights_busy;
	if (f.overflow.p && *f.overflow.p) return detect_overflow(e);
	return LCD_OK;
}

int lcd_verify_top_dev(lcd_engine * e, const void * d_queries, const float * d_uv, int n_frames, int nq_per_frame, const float * d_likelihood,
                       const int * d_sig_ids, int ns, const lcd_verify_params * vp, void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(require_binary(e, "lcd_verify_top_dev"));
	LCD_TRY(set_device(e));
	if (!d_queries || !d_uv || !d_likelihood || !d_sig_ids || n_frames <= 0 || ns <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "null argument");
	if (nq_per_frame <= 0 || nq_per_frame > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "1..%d descriptors per frame", kMaxFrameQueries);
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	return verify_top_dev(e, static_cast<const uint32_t *>(d_queries), d_uv, n_frames, nq_per_frame, d_likelihood, d_sig_ids, ns, vp, s);
}

int lcd_process_fetch(lcd_engine * e, int n_frames, int * hypothesis_out, lcd_verify_result * results)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (n_frames <= 0) return LCD_OK;
	cudaStream_t s = e->stream;
	LCD_CUDA(e, cudaDeviceSynchronize());
	if (hypothesis_out) LCD_CUDA(e, cudaMemcpyAsync(hypothesis_out, e->d_hyp_id.p, n_frames * sizeof(int), cudaMemcpyDeviceToHost, s));
	if (results) return verify_download(e, n_frames, 0, results, nullptr, nullptr, s);
	LCD_CUDA(e, cudaStreamSynchronize(s));
	return LCD_OK;
}

int lcd_process_fetch_async(lcd_engine * e, int n_frames, int * hypothesis_out, lcd_verify_result * results, void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (n_frames <= 0) return LCD_OK;
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	if (hypothesis_out) LCD_CUDA(e, cudaMemcpyAsync(hypothesis_out, e->d_hyp_id.p, n_frames * sizeof(int), cudaMemcpyDeviceToHost, s));
	if (results)
	{
		static_assert(sizeof(PackedVerifyResult) == sizeof(lcd_verify_result), "packed result layout");
		if (!e->v_ok.p || !e->d_hyp_id.p) LCD_FAIL(e, LCD_ERR_STATE, "no verification results on the device: run a step with verify parameters first");
		LCD_CUDA(e, e->v_packed.reserve(n_frames, 0, false, s));
		pack_verify_results_kernel<<<(n_frames + 127) / 128, 128, 0, s>>>(n_frames, e->v_ok.p, e->v_nm.p, e->v_ninl.p, e->v_iters.p, e->v_rvec.p, e->v_tvec.p,
		                                                                 e->v_T.p, e->v_cov6.p, e->v_packed.p);
		LCD_CHECK_LAUNCH(e);
		LCD_CUDA(e, cudaMemcpyAsync(results, e->v_packed.p, n_frames * sizeof(PackedVerifyResult), cudaMemcpyDeviceToHost, s));
	}
	return LCD_OK;
}

int lcd_process_batch(lcd_engine * e, const void * queries, const float * uv, int n_frames, int nq_per_frame, int incremental, float nndr,
                      int new_words_compared_together, const int * sig_ids, int ns, int n_total, const lcd_verify_params * vp,
                      int * word_ids_out, float * likelihood_out, int * hypothesis_out, lcd_verify_result * results)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(require_binary(e, "lcd_process_batch"));
	LCD_TRY(set_device(e));
	if (!queries || !uv || n_frames <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "Descriptors size is null!");
	if (nq_per_frame <= 0 || nq_per_frame > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "1..%d descriptors per frame", kMaxFrameQueries);
	if (!sig_ids || ns <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "ids list is empty");
	cudaStream_t s = e->stream;
	const size_t nq_total = static_cast<size_t>(n_frames) * nq_per_frame;
	LCD_CUDA(e, e->d_queries.reserve(nq_total * e->nw, 0, false, s));
	LCD_CUDA(e, e->d_uv.reserve(nq_total * 2, 0, false, s));
	LCD_CUDA(e, e->d_sig_ids.reserve(ns, 0, false, s));
	LCD_CUDA(e, e->d_like.reserve(static_cast<size_t>(n_frames) * ns, 0, false, s));
	if (word_ids_out) LCD_CUDA(e, e->d_word_ids.reserve(nq_total, 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->d_queries.p, queries, nq_total * e->nw * 4, cudaMemcpyHostToDevice, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->d_uv.p, uv, nq_total * 2 * sizeof(float), cudaMemcpyHostToDevice, s));
	LCD_CUDA(e, cudaMemcpyAsync(e->d_sig_ids.p, sig_ids, ns * sizeof(int), cudaMemcpyHostToDevice, s));
	LCD_TRY(process_dev(e, e->d_queries.p, e->d_uv.p, n_frames, nq_per_frame, incremental, nndr, new_words_compared_together, e->d_sig_ids.p, ns,
	                    n_total, vp, word_ids_out ? e->d_word_ids.p : nullptr, e->d_like.p, s));
	if (word_ids_out) LCD_CUDA(e, cudaMemcpyAsync(word_ids_out, e->d_word_ids.p, nq_total * sizeof(int), cudaMemcpyDeviceToHost, s));
	if (likelihood_out)
		LCD_CUDA(e, cudaMemcpyAsync(likelihood_out, e->d_like.p, static_cast<size_t>(n_frames) * ns * sizeof(float), cudaMemcpyDeviceToHost, s));
	if (hypothesis_out) LCD_CUDA(e, cudaMemcpyAsync(hypothesis_out, e->d_hyp_id.p, n_frames * sizeof(int), cudaMemcpyDeviceToHost, s));
	if (results) return verify_download(e, n_frames, 0, results, nullptr, nullptr, s);
	LCD_CUDA(e, cudaStreamSynchronize(s));
	return LCD_OK;
}

// ---- word-range sharding ---------------------------------------------------------------------
int lcd_shard_set_row_offset(lcd_engine * e, int global_row_offset)
{
	if (!e || global_row_offset < 0) return LCD_ERR_INVALID;
	e->row_offset = global_row_offset;
	return LCD_OK;
}

int lcd_shard_knn2_keys_dev(lcd_engine * e, const void * d_queries, int nq, uint32_t * d_keys_out, void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(require_binary(e, "lcd_shard_knn2_keys_dev"));
	LCD_TRY(set_device(e));
	if (!d_queries || nq <= 0 || !d_keys_out) LCD_FAIL(e, LCD_ERR_INVALID, "null argument");
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	int n_chunks = 0;
	LCD_TRY(run_knn(e, static_cast<const uint32_t *>(d_queries), nq, e->n_indexed, &n_chunks, s));
	knn2_merge_kernel<<<(nq + 255) / 256, 256, 0, s>>>(e->d_partial.p, n_chunks, nq, d_keys_out);
	LCD_CHECK_LAUNCH(e);
	return LCD_OK;
}

int lcd_shard_resolve_score_dev(lcd_engine * e, const void * d_queries, int n_frames, int nq_per_frame,
                                const uint32_t * d_keys_gathered, int n_ranks, const int * d_row_ids, int total_rows_, int last_word_id,
                                int incremental, float nndr, int new_words_compared_together, const int * d_sig_ids, int ns, int n_total,
                                int * d_word_ids_out, long long * d_scores_out, void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(require_binary(e, "lcd_shard_resolve_score_dev"));
	LCD_TRY(set_device(e));
	if (!d_queries || !d_keys_gathered || !d_row_ids || n_frames <= 0 || n_ranks <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "null argument");
	if (nq_per_frame <= 0 || nq_per_frame > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "1..%d descriptors per frame", kMaxFrameQueries);
	(void)total_rows_;
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	const bool score = d_scores_out != nullptr && ns > 0;
	ResolveArgs a{};
	a.queries = static_cast<const uint32_t *>(d_queries);
	a.nq = nq_per_frame;
	a.nq_total = n_frames * nq_per_frame;
	a.partial = reinterpret_cast<const uint2 *>(d_keys_gathered);
	a.n_chunks = n_ranks;
	a.row_ids = d_row_ids;
	a.incremental = incremental;
	a.nndr = nndr;
	a.cmp_new = new_words_compared_together;
	a.last_word_id = last_word_id;
	a.word_ids_out = d_word_ids_out;
	if (score)
	{
		LCD_TRY(ensure_uq(e, n_frames, nq_per_frame, s));
		LCD_TRY(ensure_acc(e, n_frames));
		LCD_CUDA(e, zero_fill_async(e->acc.p, static_cast<size_t>(e->acc_stride) * n_frames * sizeof(long long), s));
		fill_prep(e, a, static_cast<float>(n_total), 1);
	}
	LCD_TRY(launch_resolve(e, a, n_frames, s));
	if (score)
	{
		LCD_TRY(launch_score(e, n_frames, nq_per_frame, s));
		dim3 grid((ns + 255) / 256, n_frames);
		gather_fixed_kernel<<<grid, 256, 0, s>>>(e->acc.p, e->acc_stride, static_cast<int>(e->h_ni.size()), d_sig_ids, ns, d_scores_out);
		LCD_CHECK_LAUNCH(e);
	}
	return LCD_OK;
}

int lcd_shard_resolve_frames_dev(lcd_engine * e, const void * d_queries_all, int frame0, int n_frames, int n_frames_total, int nq_per_frame,
                                 const uint32_t * d_keys_gathered, int n_ranks, const int * d_row_ids, int last_word_id, int incremental,
                                 float nndr, int new_words_compared_together, const int * d_n_per_frame, int * d_word_ids_out, void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(require_binary(e, "lcd_shard_resolve_frames_dev"));
	LCD_TRY(set_device(e));
	if (!d_queries_all || !d_keys_gathered || !d_row_ids || !d_word_ids_out || n_frames <= 0 || n_ranks <= 0 || frame0 < 0 ||
	    frame0 + n_frames > n_frames_total)
		LCD_FAIL(e, LCD_ERR_INVALID, "null argument or frame range outside the job");
	if (nq_per_frame <= 0 || nq_per_frame > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "1..%d descriptors per frame", kMaxFrameQueries);
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	ResolveArgs a{};
	a.queries = static_cast<const uint32_t *>(d_queries_all) + static_cast<size_t>(frame0) * nq_per_frame * e->nw;
	a.nq = nq_per_frame;
	a.nq_total = n_frames_total * nq_per_frame;                                     // stride between the gathered key sets
	a.partial = reinterpret_cast<const uint2 *>(d_keys_gathered) + static_cast<size_t>(frame0) * nq_per_frame;
	a.n_chunks = n_ranks;
	a.row_ids = d_row_ids;
	a.incremental = incremental;
	a.nndr = nndr;
	a.cmp_new = new_words_compared_together;
	a.last_word_id = last_word_id;
	a.word_ids_out = d_word_ids_out;
	a.nq_frame = d_n_per_frame ? d_n_per_frame + frame0 : nullptr;
	return launch_resolve(e, a, n_frames, s);
}

int lcd_shard_score_ids_dev(lcd_engine * e, const int * d_word_ids_all, int n_frames, int nq_per_frame, const int * d_sig_ids, int ns, int n_total,
                            long long * d_scores_out, void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!d_word_ids_all || !d_sig_ids || !d_scores_out || n_frames <= 0 || ns <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "null argument");
	if (nq_per_frame <= 0 || nq_per_frame > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "1..%d words per signature", kMaxFrameQueries);
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	LCD_TRY(ensure_uq(e, n_frames, nq_per_frame, s));
	LCD_TRY(ensure_acc(e, n_frames));
	LCD_CUDA(e, zero_fill_async(e->acc.p, static_cast<size_t>(e->acc_stride) * n_frames * sizeof(long long), s));
	ResolveArgs a{};
	a.nq = nq_per_frame;
	fill_prep(e, a, static_cast<float>(n_total), 1);
	int nq_pad = 32;
	while (nq_pad < nq_per_frame) nq_pad <<= 1;
	prof_mark(e, LCD_PROF_RESOLVE, s);
	prep_from_ids_kernel<<<n_frames, kResolveThreads, nq_pad * sizeof(uint32_t), s>>>(d_word_ids_all, a);
	prof_mark(e, LCD_PROF_RESOLVE, s);
	LCD_CHECK_LAUNCH(e);
	LCD_TRY(launch_score(e, n_frames, nq_per_frame, s));
	dim3 grid((ns + 255) / 256, n_frames);
	gather_fixed_kernel<<<grid, 256, 0, s>>>(e->acc.p, e->acc_stride, static_cast<int>(e->h_ni.size()), d_sig_ids, ns, d_scores_out);
	LCD_CHECK_LAUNCH(e);
	return LCD_OK;
}

// ---- mapping mode: Memory::update for a stream of frames ------------------------------------------------------------------
int lcd_map_detect_async(lcd_engine * e, const uint8_t * image, int width, int height, int channels, const void * depth, int depth_type,
                         const lcd_orb_params * params)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!image || width <= 0 || height <= 0 || !params) LCD_FAIL(e, LCD_ERR_INVALID, "null image");
	if (e->cfg.desc_type != LCD_DESC_U8 || e->cfg.desc_dim != 32) LCD_FAIL(e, LCD_ERR_INVALID, "ORB descriptors need an engine with 32-byte binary descriptors");
	if (e->map_busy >= 2) LCD_FAIL(e, LCD_ERR_STATE, "two detections are already in flight: call lcd_map_frame first");
	const int cap = params->n_features;
	if (cap <= 0 || cap > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "Kp/MaxFeatures must be 1..%d", kMaxFrameQueries);
	lcd_engine::MapSlot & ms = e->map_slots[(e->map_head + e->map_busy) & 1];
	cudaStream_t s = e->orb_stream;
	if (!ms.done) LCD_CUDA(e, cudaEventCreateWithFlags(&ms.done, cudaEventDisableTiming));
	const size_t px = static_cast<size_t>(width) * height;
	if (!depth) depth_type = LCD_DEPTH_NONE;
	LCD_CUDA(e, ms.img.reserve(px * channels, 0, false, s));
	LCD_CUDA(e, cudaMemcpyAsync(ms.img.p, image, px * channels, cudaMemcpyHostToDevice, s));
	if (depth_type != LCD_DEPTH_NONE)
	{
		LCD_CUDA(e, ms.depth.reserve(px * depth_elem_bytes(depth_type), 0, false, s));
		LCD_CUDA(e, cudaMemcpyAsync(ms.depth.p, depth, px * depth_elem_bytes(depth_type), cudaMemcpyHostToDevice, s));
	}
	LCD_CUDA(e, ms.kp.reserve(cap, 0, false, s));
	LCD_CUDA(e, ms.desc.reserve(static_cast<size_t>(cap) * 32, 0, false, s));
	LCD_CUDA(e, ms.xyz.reserve(static_cast<size_t>(cap) * 3, 0, false, s));
	LCD_CUDA(e, ms.n.reserve(1, 0, false, s));
	LCD_CUDA(e, ms.h_n.reserve(1));
	LCD_CUDA(e, ms.h_overflow.reserve(1));
	LCD_CUDA(e, zero_fill_async(ms.desc.p, static_cast<size_t>(cap) * 32, s)); // padding rows feed the NN kernel: defined bytes
	LCD_TRY(orb_run(e, 1, ms.img.p, width, height, channels, depth_type != LCD_DEPTH_NONE ? ms.depth.p : nullptr, depth_type, params, cap, ms.kp.p, ms.desc.p,
	                ms.xyz.p, nullptr, ms.n.p, s));
	LCD_CUDA(e, cudaMemcpyAsync(ms.h_n.p, ms.n.p, sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaMemcpyAsync(ms.h_overflow.p, e->o_overflow.p, sizeof(int), cudaMemcpyDeviceToHost, s));
	LCD_CUDA(e, cudaEventRecord(ms.done, s));
	ms.cap = cap;
	ms.busy = true;
	++e->map_busy;
	return LCD_OK;
}

int lcd_map_frame(lcd_engine * e, int sig_id, int incremental, float nndr, int new_words_compared_together, const int * wm_sig_ids, int ns,
                  int n_total, int * n_kp_out, lcd_keypoint * kp_out, uint8_t * desc_out, float * xyz_out, int * word_ids_out, int * n_new_out,
                  float * likelihood_out)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (e->map_busy <= 0) LCD_FAIL(e, LCD_ERR_STATE, "no detection in flight: call lcd_map_detect_async first");
	if (!word_ids_out) LCD_FAIL(e, LCD_ERR_INVALID, "null output");
	lcd_engine::MapSlot & ms = e->map_slots[e->map_head];
	cudaStream_t s = e->stream;
	// Memory::preUpdate: the words of the previous frame join the index (VWDictionary::update)
	LCD_TRY(lcd_dict_update(e));
	LCD_CUDA(e, cudaStreamWaitEvent(s, ms.done, 0));
	const int cap = ms.cap;
	int n_new = 0, n_kp = 0;
	// Memory::createSignature: quantise the frame's descriptors (they never leave the device), references for sig_id
	int rc = quantize_dev(e, reinterpret_cast<const uint32_t *>(ms.desc.p), cap, -1, ms.n.p, sig_id, incremental, nndr, new_words_compared_together,
	                      word_ids_out, &n_new, &n_kp, s);
	e->map_head ^= 1;
	--e->map_busy;
	ms.busy = false;
	if (rc != LCD_OK) return rc;
	if (*ms.h_overflow.p) return detect_overflow(e);
	if (n_kp_out) *n_kp_out = n_kp;
	if (n_new_out) *n_new_out = n_new;
	if (kp_out) LCD_CUDA(e, cudaMemcpyAsync(kp_out, ms.kp.p, static_cast<size_t>(n_kp) * sizeof(OrbKeypoint), cudaMemcpyDeviceToHost, s));
	if (desc_out) LCD_CUDA(e, cudaMemcpyAsync(desc_out, ms.desc.p, static_cast<size_t>(n_kp) * 32, cudaMemcpyDeviceToHost, s));
	if (xyz_out) LCD_CUDA(e, cudaMemcpyAsync(xyz_out, ms.xyz.p, static_cast<size_t>(n_kp) * 3 * sizeof(float), cudaMemcpyDeviceToHost, s));
	// Memory::computeLikelihood against the working memory
	if (likelihood_out && wm_sig_ids && ns > 0 && n_kp > 0) return lcd_index_score(e, word_ids_out, n_kp, wm_sig_ids, ns, n_total, likelihood_out);
	LCD_CUDA(e, cudaStreamSynchronize(s));
	return LCD_OK;
}

// ---- NCCL inside the library: communicator + the fused sharded step ------------------------------------------------
int lcd_shard_unique_id(char id_out[128])
{
	static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
	if (!id_out) return LCD_ERR_INVALID;
	if (!nccl_api().ok)
	{
		g_create_error = nccl_api().why;
		return LCD_ERR_STATE;
	}
	ncclUniqueId id;
	if (nccl_api().GetUniqueId(&id) != ncclSuccess)
	{
		g_create_error = "ncclGetUniqueId failed";
		return LCD_ERR_CUDA;
	}
	memcpy(id_out, &id, 128);
	return LCD_OK;
}

// LCD_SHARD_TRACE=2: sixteen steps of per-stage events recorded without any synchronisation, printed after the sixteenth
static int shard_record(lcd_engine * e, int h, int k, cudaStream_t st)
{
	LCD_CUDA(e, cudaEventRecord(e->sh_ev[h][k], st));
	if (e->sh_trace == 2 && e->sh_ring_step < 16) LCD_CUDA(e, cudaEventRecord(e->sh_ring[(e->sh_ring_step * 2 + h) * 9 + k], st));
	return LCD_OK;
}

static int shard_comm_common(lcd_engine * e, int rank, int n_ranks)
{
	if (!e->comm_stream) LCD_CUDA(e, cudaStreamCreateWithFlags(&e->comm_stream, cudaStreamNonBlocking));
	e->sh_trace = env_int("LCD_SHARD_TRACE", 0);
	if (e->sh_trace == 2 && e->sh_ring.empty())
	{
		e->sh_ring.assign(16 * 2 * 9, nullptr);
		for (cudaEvent_t & ev : e->sh_ring) LCD_CUDA(e, cudaEventCreate(&ev));
	}
	for (auto & half : e->sh_ev)
		for (cudaEvent_t & ev : half)
			if (!ev) LCD_CUDA(e, cudaEventCreateWithFlags(&ev, e->sh_trace ? cudaEventDefault : cudaEventDisableTiming));
	for (cudaEvent_t & ev : e->sh_tr)
		if (e->sh_trace && !ev) LCD_CUDA(e, cudaEventCreate(&ev));
	e->sh_rank = rank;
	e->sh_ranks = n_ranks;
	return LCD_OK;
}

int lcd_shard_comm_init(lcd_engine * e, const char id[128], int rank, int n_ranks)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!id || n_ranks < 1 || rank < 0 || rank >= n_ranks) LCD_FAIL(e, LCD_ERR_INVALID, "bad rank %d of %d", rank, n_ranks);
	if (!nccl_api().ok) LCD_FAIL(e, LCD_ERR_STATE, "%s", nccl_api().why.c_str());
	if (e->comm) LCD_FAIL(e, LCD_ERR_STATE, "the engine already has a communicator");
	ncclUniqueId uid;
	memcpy(&uid, id, 128);
	LCD_NCCL(e, nccl_api().CommInitRank(&e->comm, n_ranks, uid, rank));
	e->comm_owned = true;
	return shard_comm_common(e, rank, n_ranks);
}

int lcd_shard_comm_adopt(lcd_engine * e, void * nccl_comm, int rank, int n_ranks)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!nccl_comm || n_ranks < 1 || rank < 0 || rank >= n_ranks) LCD_FAIL(e, LCD_ERR_INVALID, "bad communicator / rank");
	if (!nccl_api().ok) LCD_FAIL(e, LCD_ERR_STATE, "%s", nccl_api().why.c_str());
	if (e->comm) LCD_FAIL(e, LCD_ERR_STATE, "the engine already has a communicator");
	e->comm = static_cast<ncclComm_t>(nccl_comm);
	e->comm_owned = false;
	return shard_comm_common(e, rank, n_ranks);
}

int lcd_shard_comm_destroy(lcd_engine * e)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (e->comm)
	{
		LCD_CUDA(e, cudaDeviceSynchronize());
		if (e->comm_owned) nccl_api().CommDestroy(e->comm);
		e->comm = nullptr;
	}
	e->sh_ranks = 1;
	e->sh_rank = 0;
	return LCD_OK;
}

int lcd_shard_process_frames_dev(lcd_engine * e, int n_frames, const uint8_t * d_images, int width, int height, int channels, const void * d_depth,
                                 int depth_type, const lcd_orb_params * op, int incremental, float nndr, int new_words_compared_together,
                                 const int * d_sig_ids, int ns, int n_total, const int * d_row_ids_global, int last_word_id,
                                 const lcd_verify_params * vp, int * d_word_ids_out, float * d_likelihood_out, void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(require_binary(e, "lcd_shard_process_frames_dev"));
	LCD_TRY(set_device(e));
	if (!e->comm) LCD_FAIL(e, LCD_ERR_STATE, "no communicator: call lcd_shard_comm_init first");
	if (!d_images || n_frames <= 0 || !op || !d_sig_ids || ns <= 0 || !d_row_ids_global || !d_likelihood_out)
		LCD_FAIL(e, LCD_ERR_INVALID, "null argument");
	if (e->cfg.desc_dim != 32) LCD_FAIL(e, LCD_ERR_INVALID, "ORB descriptors need an engine with 32-byte binary descriptors");
	const int cap = op->n_features;
	if (cap <= 0 || cap > kMaxFrameQueries) LCD_FAIL(e, LCD_ERR_CAPACITY, "Kp/MaxFeatures must be 1..%d", kMaxFrameQueries);
	const NcclApi & nc = nccl_api();
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	cudaStream_t c = e->comm_stream;
	const int G = e->sh_ranks, R = e->sh_rank;
	// The dictionary search runs on two halves of the local batch, so that the descriptor all-gather of the second half and the key
	// exchange of the first run under a search kernel.  The merge + NNDR stage is a one-CTA-per-frame kernel that takes as long for half a
	// batch as for a whole one, so it runs once on the whole batch and its exchange (word ids) is exposed: measured cheaper than splitting.
	const int n_parts = n_frames >= 2 && env_int("LCD_SHARD_NN_PARTS", 2) >= 2 ? 2 : 1;
	const int part_frames[2] = {n_parts == 2 ? (n_frames + 1) / 2 : n_frames, n_parts == 2 ? n_frames / 2 : 0};
	const int part_f0[2] = {0, part_frames[0]};
	// merge + NNDR always runs on the whole batch; the TF-IDF stage scores G x n_frames frames, so from 4 ranks on it is no longer a
	// single-wave kernel and is split in two halves of every rank's frames: the reduce-scatter of the first half runs under the scoring of
	// the second (LCD_SHARD_SCORE_PARTS=1|2 overrides)
	const int t_parts = 1;
	const int tail_frames[2] = {n_frames, 0};
	const int tail_f0[2] = {0, n_frames};
	const int s_parts_env = env_int("LCD_SHARD_SCORE_PARTS", 0);
	const int s_parts = n_frames >= 2 && (s_parts_env ? s_parts_env >= 2 : G >= 4) ? 2 : 1;
	const int score_frames[2] = {s_parts == 2 ? (n_frames + 1) / 2 : n_frames, s_parts == 2 ? n_frames / 2 : 0};
	const int score_f0[2] = {0, score_frames[0]};
	const size_t rows = static_cast<size_t>(n_frames) * cap;
	LCD_CUDA(e, e->o_kp.reserve(rows, 0, false, s));
	LCD_CUDA(e, e->o_desc.reserve(rows * 32, 0, false, s));
	LCD_CUDA(e, e->o_xyz.reserve(rows * 3, 0, false, s));
	LCD_CUDA(e, e->o_uv.reserve(rows * 2, 0, false, s));
	LCD_CUDA(e, e->o_n.reserve(n_frames, 0, false, s));
	LCD_CUDA(e, e->sh_n_all.reserve(static_cast<size_t>(G) * n_frames, 0, false, s));
	LCD_CUDA(e, e->d_like.reserve(static_cast<size_t>(n_frames) * ns, 0, false, s));
	for (int h = 0; h < n_parts; ++h)
	{
		const size_t pr = static_cast<size_t>(part_frames[h]) * cap; // descriptor rows of this part on one rank
		LCD_CUDA(e, e->sh_desc_all[h].reserve(pr * 32 * G, 0, false, s));
		LCD_CUDA(e, e->sh_keys[h].reserve(pr * 2 * G, 0, false, s));
	}
	LCD_CUDA(e, e->sh_keys_mine[0].reserve(rows * 2 * G, 0, false, s)); // [rank][local frame][feature]: both halves land in one array
	LCD_CUDA(e, e->sh_words_loc[0].reserve(rows, 0, false, s));
	LCD_CUDA(e, e->sh_words_all[0].reserve(rows * G, 0, false, s));
	for (int h = 0; h < s_parts; ++h)
	{
		LCD_CUDA(e, e->sh_scores[h].reserve(static_cast<size_t>(score_frames[h]) * G * ns, 0, false, s));
		LCD_CUDA(e, e->sh_scores_loc[h].reserve(static_cast<size_t>(score_frames[h]) * ns, 0, false, s));
	}
	std::chrono::steady_clock::time_point host_t[6];
	const auto host_begin = std::chrono::steady_clock::now();
	if (e->sh_trace == 1 && e->sh_trace_armed)
	{
		// timeline of the PREVIOUS step, in ms after its first kernel: per half, the end of each compute stage (s) and exchange (c)
		LCD_CUDA(e, cudaEventSynchronize(e->sh_tr[1]));
		LCD_CUDA(e, cudaStreamSynchronize(c));
		static const char * names[8] = {"orb", "ag_desc", "nn", "a2a_keys", "resolve", "ag_words", "score", "rs_scores"};
		float ms = 0.f;
		fprintf(stderr, "[lcd shard trace rank %d]", R);
		for (int h = 0; h < n_parts; ++h)
			for (int k = 0; k < 8; ++k)
				if ((k < 4 || (k < 6 ? h < t_parts : h < s_parts)) && cudaEventElapsedTime(&ms, e->sh_tr[0], e->sh_ev[h][k]) == cudaSuccess) fprintf(stderr, " %s%d=%.3f", names[k], h, ms);
		if (cudaEventElapsedTime(&ms, e->sh_tr[0], e->sh_tr[1]) == cudaSuccess) fprintf(stderr, " end=%.3f", ms);
		fprintf(stderr, "\n");
	}
	LCD_CUDA(e, zero_fill_async(e->o_desc.p, rows * 32, s)); // padding rows of short frames must hold defined bytes
	if (e->sh_trace) LCD_CUDA(e, cudaEventRecord(e->sh_tr[0], s));
	if (e->sh_trace == 2 && e->sh_ring_step < 16) LCD_CUDA(e, cudaEventRecord(e->sh_ring[(e->sh_ring_step * 2 + 0) * 9 + 8], s));
	// the communication stream starts behind everything already queued on the compute stream
	LCD_CUDA(e, cudaEventRecord(e->sh_ev[0][7], s));
	LCD_CUDA(e, cudaStreamWaitEvent(c, e->sh_ev[0][7], 0));

	host_t[0] = std::chrono::steady_clock::now();
	// phase 1: detect + describe the local frames in one pass (splitting detection costs more than the 30-50 us all-gather it would hide),
	// then all-gather the descriptors part by part (and the keypoint counts): the second part's exchange runs under the first part's search
	LCD_TRY(orb_run(e, n_frames, d_images, width, height, channels, d_depth, depth_type, op, cap, e->o_kp.p, e->o_desc.p, e->o_xyz.p, e->o_uv.p, e->o_n.p, s, 0,
	                n_frames));
	for (int h = 0; h < n_parts; ++h)
	{
		LCD_TRY(shard_record(e, h, 0, s));
		LCD_CUDA(e, cudaStreamWaitEvent(c, e->sh_ev[h][0], 0));
		const size_t pr = static_cast<size_t>(part_frames[h]) * cap;
		LCD_NCCL(e, nc.GroupStart());
		LCD_NCCL(e, nc.AllGather(e->o_desc.p + static_cast<size_t>(part_f0[h]) * cap * 32, e->sh_desc_all[h].p, pr * 32, ncclUint8, e->comm, c));
		if (h == n_parts - 1) LCD_NCCL(e, nc.AllGather(e->o_n.p, e->sh_n_all.p, n_frames, ncclInt32, e->comm, c));
		LCD_NCCL(e, nc.GroupEnd());
		LCD_TRY(shard_record(e, h, 1, c));
	}
	host_t[1] = std::chrono::steady_clock::now();
	// phase 2: top-2 keys of every rank's descriptors over the local word range; every rank gets back the keys of ITS frames
	for (int h = 0; h < n_parts; ++h)
	{
		const size_t pr = static_cast<size_t>(part_frames[h]) * cap;
		const int nq_all = static_cast<int>(pr) * G;
		LCD_CUDA(e, cudaStreamWaitEvent(s, e->sh_ev[h][1], 0));
		int n_chunks = 0;
		LCD_TRY(run_knn(e, reinterpret_cast<const uint32_t *>(e->sh_desc_all[h].p), nq_all, e->n_indexed, &n_chunks, s));
		knn2_merge_kernel<<<(nq_all + 255) / 256, 256, 0, s>>>(e->d_partial.p, n_chunks, nq_all, e->sh_keys[h].p);
		LCD_CHECK_LAUNCH(e);
		LCD_TRY(shard_record(e, h, 2, s));
		LCD_CUDA(e, cudaStreamWaitEvent(c, e->sh_ev[h][2], 0));
		LCD_NCCL(e, nc.GroupStart());
		for (int p = 0; p < G; ++p)
		{
			LCD_NCCL(e, nc.Send(e->sh_keys[h].p + static_cast<size_t>(p) * pr * 2, pr * 2, ncclUint32, p, e->comm, c));
			LCD_NCCL(e, nc.Recv(e->sh_keys_mine[0].p + (static_cast<size_t>(p) * rows + static_cast<size_t>(part_f0[h]) * cap) * 2, pr * 2, ncclUint32, p, e->comm, c));
		}
		LCD_NCCL(e, nc.GroupEnd());
		LCD_TRY(shard_record(e, h, 3, c));
	}
	host_t[2] = std::chrono::steady_clock::now();
	// phase 3: merge + NNDR / new-word pass of the local frames, all-gather of their word ids
	for (int h = 0; h < t_parts; ++h)
	{
		const size_t pr = static_cast<size_t>(tail_frames[h]) * cap;
		LCD_CUDA(e, cudaStreamWaitEvent(s, e->sh_ev[t_parts == 2 ? h : n_parts - 1][3], 0));
		ResolveArgs a{};
		a.queries = reinterpret_cast<const uint32_t *>(e->o_desc.p) + static_cast<size_t>(tail_f0[h]) * cap * e->nw;
		a.nq = cap;
		a.nq_total = static_cast<int>(rows);                       // stride between the G key sets
		a.partial = reinterpret_cast<const uint2 *>(e->sh_keys_mine[0].p) + static_cast<size_t>(tail_f0[h]) * cap;
		a.n_chunks = G;
		a.row_ids = d_row_ids_global;
		a.incremental = incremental;
		a.nndr = nndr;
		a.cmp_new = new_words_compared_together;
		a.last_word_id = last_word_id;
		a.word_ids_out = e->sh_words_loc[h].p;
		a.nq_frame = e->o_n.p + tail_f0[h];
		LCD_TRY(launch_resolve(e, a, tail_frames[h], s));
		if (d_word_ids_out)
			LCD_CUDA(e, cudaMemcpyAsync(d_word_ids_out + static_cast<size_t>(tail_f0[h]) * cap, e->sh_words_loc[h].p, pr * sizeof(int), cudaMemcpyDeviceToDevice, s));
		LCD_TRY(shard_record(e, h, 4, s));
		LCD_CUDA(e, cudaStreamWaitEvent(c, e->sh_ev[h][4], 0));
		LCD_NCCL(e, nc.AllGather(e->sh_words_loc[h].p, e->sh_words_all[h].p, pr, ncclInt32, e->comm, c));
		LCD_TRY(shard_record(e, h, 5, c));
	}
	host_t[3] = std::chrono::steady_clock::now();
	// phase 4: TF-IDF of every rank's frames over the local word range, reduce-scatter of the exact fixed-point sums
	for (int h = 0; h < s_parts; ++h)
	{
		const int nf_all = score_frames[h] * G; // frames [score_f0, +score_frames) of every rank, rank-major
		LCD_CUDA(e, cudaStreamWaitEvent(s, e->sh_ev[0][5], 0));
		LCD_TRY(ensure_uq(e, nf_all, cap, s));
		LCD_TRY(ensure_acc(e, nf_all));
		LCD_CUDA(e, zero_fill_async(e->acc.p, static_cast<size_t>(e->acc_stride) * nf_all * sizeof(long long), s));
		ResolveArgs a{};
		a.nq = cap;
		fill_prep(e, a, static_cast<float>(n_total), 1);
		int nq_pad = 32;
		while (nq_pad < cap) nq_pad <<= 1;
		prof_mark(e, LCD_PROF_RESOLVE, s);
		prep_local_ids_kernel<<<nf_all, kResolveThreads, nq_pad * sizeof(uint32_t), s>>>(e->sh_words_all[0].p, a, n_frames, score_f0[h], score_frames[h]);
		prof_mark(e, LCD_PROF_RESOLVE, s);
		LCD_CHECK_LAUNCH(e);
		LCD_TRY(launch_score(e, nf_all, cap, s));
		gather_fixed_kernel<<<dim3((ns + 255) / 256, nf_all), 256, 0, s>>>(e->acc.p, e->acc_stride, static_cast<int>(e->h_ni.size()), d_sig_ids, ns, e->sh_scores[h].p);
		LCD_CHECK_LAUNCH(e);
		LCD_TRY(shard_record(e, h, 6, s));
		LCD_CUDA(e, cudaStreamWaitEvent(c, e->sh_ev[h][6], 0));
		LCD_NCCL(e, nc.ReduceScatter(e->sh_scores[h].p, e->sh_scores_loc[h].p, static_cast<size_t>(score_frames[h]) * ns, ncclInt64, ncclSum, e->comm, c));
		LCD_TRY(shard_record(e, h, 7, c));
	}
	host_t[4] = std::chrono::steady_clock::now();
	// phase 5: likelihood of the local frames, verification of their top hypothesis
	for (int h = 0; h < s_parts; ++h)
	{
		const int n = score_frames[h] * ns;
		LCD_CUDA(e, cudaStreamWaitEvent(s, e->sh_ev[h][7], 0));
		fixed_to_float_kernel<<<(n + 255) / 256, 256, 0, s>>>(e->sh_scores_loc[h].p, n, d_likelihood_out + static_cast<size_t>(score_f0[h]) * ns);
		LCD_CHECK_LAUNCH(e);
	}
	if (vp)
		LCD_TRY(verify_top_dev(e, reinterpret_cast<const uint32_t *>(e->o_desc.p), e->o_uv.p, n_frames, cap, d_likelihood_out, d_sig_ids, ns, vp, s, e->o_n.p,
		                       e->o_xyz.p));
	if (e->sh_trace)
	{
		LCD_CUDA(e, cudaEventRecord(e->sh_tr[1], s));
		e->sh_trace_armed = true;
	}
	host_t[5] = std::chrono::steady_clock::now();
	if (e->sh_trace == 2 && e->sh_ring_step == 9)
	{
		auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
			return std::chrono::duration<double, std::micro>(b - a).count();
		};
		fprintf(stderr, "[lcd shard host rank %d] us: reserve=%.0f orb+ag_desc=%.0f nn+a2a=%.0f resolve+ag_words=%.0f score+rs=%.0f verify=%.0f\n", R,
		        us(host_begin, host_t[0]), us(host_t[0], host_t[1]), us(host_t[1], host_t[2]), us(host_t[2], host_t[3]), us(host_t[3], host_t[4]),
		        us(host_t[4], host_t[5]));
	}
	if (e->sh_trace == 2 && e->sh_ring_step < 16)
	{
		LCD_CUDA(e, cudaEventRecord(e->sh_ring[(e->sh_ring_step * 2 + 1) * 9 + 8], s));
		if (++e->sh_ring_step == 16)
		{
			LCD_CUDA(e, cudaStreamSynchronize(s));
			LCD_CUDA(e, cudaStreamSynchronize(c));
			static const char * names[8] = {"orb", "ag_desc", "nn", "a2a_keys", "resolve", "ag_words", "score", "rs_scores"};
			const cudaEvent_t origin = e->sh_ring[(8 * 2 + 0) * 9 + 8]; // begin of step 8
			for (int st = 8; st < 12; ++st)
			{
				float ms = 0.f;
				fprintf(stderr, "[lcd shard ring rank %d step %d]", R, st);
				if (cudaEventElapsedTime(&ms, origin, e->sh_ring[(st * 2 + 0) * 9 + 8]) == cudaSuccess) fprintf(stderr, " begin=%.3f", ms);
				for (int h = 0; h < n_parts; ++h)
					for (int k = 0; k < 8; ++k)
						if ((k < 4 || (k < 6 ? h < t_parts : h < s_parts)) && cudaEventElapsedTime(&ms, origin, e->sh_ring[(st * 2 + h) * 9 + k]) == cudaSuccess) fprintf(stderr, " %s%d=%.3f", names[k], h, ms);
				if (cudaEventElapsedTime(&ms, origin, e->sh_ring[(st * 2 + 1) * 9 + 8]) == cudaSuccess) fprintf(stderr, " end=%.3f", ms);
				fprintf(stderr, "\n");
			}
		}
	}
	return LCD_OK;
}

int lcd_shard_finalize_dev(lcd_engine * e, const long long * d_scores, int n, float * d_likelihood_out, void * stream)
{
	if (!e) return LCD_ERR_INVALID;
	LCD_TRY(set_device(e));
	if (!d_scores || !d_likelihood_out || n <= 0) LCD_FAIL(e, LCD_ERR_INVALID, "null argument");
	cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : e->stream;
	fixed_to_float_kernel<<<(n + 255) / 256, 256, 0, s>>>(d_scores, n, d_likelihood_out);
	LCD_CHECK_LAUNCH(e);
	return LCD_OK;
}

} // extern "C"
