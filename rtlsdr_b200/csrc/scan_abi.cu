/*
 * scan_abi.cu -- implementation of include/rtlsdr_gpu_scan.h on CUDA (sm_100a).
 *
 * Host responsibilities kept here (no DSP on the CPU):
 *  - host-built tables exactly as the reference builds them
 *    (sine_table rtl_power.c:247-261, window_coefs :985-988),
 *  - the pinned, double-buffered staging ring that submit() copies into
 *    (async buffers are re-armed right after the callback, librtlsdr.c:2705-2707),
 *  - grouping the submitted reads by hop into segments so that one CTA
 *    accumulates many reads of a hop in registers before a single flush,
 *  - tunes[i].samples bookkeeping (rtl_power.c:717, :435): deterministic from
 *    the number of reads, so it is counted on the host.
 */
#include "../../include/rtlsdr_gpu_scan.h"
#include "csv_text.cuh"
#include "scan_host.cuh"
#include "scan_kernels.cuh"
#include "scan_large.cuh"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

using namespace rscan;

namespace {

constexpr int kDescSlots = 4;
constexpr size_t kDefaultRing = 32u << 20;
constexpr size_t kScratchBudget = 512ull << 20; /* device bytes for decimation / large-FFT scratch */
constexpr int kChainMaxPasses = 7;           /* fused fifth_order chain up to 128x decimation */
constexpr int kDecimChunks = 4;              /* only for batches >= kDecimOverlapBytes (measured: a loss below) */
constexpr size_t kDecimOverlapBytes = 1ull << 30;

struct DescSlot {
	void *h = nullptr; /* pinned */
	void *d = nullptr;
	size_t cap = 0;
	cudaEvent_t done = nullptr;
	bool used = false;
};

struct RegularKey {
	const void *base = nullptr;
	int hop_first = -1, hop_count = 0, passes = 0;
	long long pass_stride = 0, hop_stride = 0;
	bool valid = false;
	int n_reads = 0, n_segs = 0;
	bool operator==(const RegularKey &o) const
	{
		return valid && o.valid && base == o.base && hop_first == o.hop_first && hop_count == o.hop_count &&
		       passes == o.passes && pass_stride == o.pass_stride && hop_stride == o.hop_stride;
	}
};

} // namespace

struct rtlsdr_gpu_scan {
	rtlsdr_gpu_scan_cfg_t cfg;
	ScanShape shape;
	int num_sms = 148, ctas_per_sm = 2;

	cudaStream_t own_stream = nullptr, stream = nullptr;
	cudaEvent_t ev_a = nullptr, ev_b = nullptr;

	long long *d_avg = nullptr;     /* [tune_count * N] bins, then [tune_count] sample counters */
	long long *d_smp64 = nullptr;   /* = d_avg + tune_count * N */
	/* RTLSDR_GPU_FLAG_ASYNC_REPORT: a second accumulator set.  collect_device() reports the current set on
	 * report_stream and flips, so the handle's stream runs transform kernels back to back (d_avg / d_smp64
	 * always point at the set the NEXT submits accumulate into) */
	long long *d_avg_other = nullptr;
	cudaStream_t report_stream = nullptr;
	cudaEvent_t ev_scan = nullptr, ev_report[2] = { nullptr, nullptr };
	bool report_pending[2] = { false, false };
	int cur_acc = 0;
	unsigned *d_done = nullptr;     /* [tune_count] epilogue tickets (fused read-and-zero) */
	unsigned long long *d_level = nullptr; /* [tune_count][2] soft-AGC byte counts (optional) */
	std::vector<uint64_t> level_bytes;
	int2 *d_tw = nullptr;
	int2 *d_twc = nullptr;          /* small path: per-stage compact twiddles (shared-memory image); large path: round A's */
	int2 *d_twb = nullptr;          /* large path: round-B twiddles re-ordered [se][plow][ilow] */
	uint16_t *d_win = nullptr;
	double *d_db = nullptr;
	double *d_iir = nullptr;        /* -s iir smoothing state [tune_count][db_count - 1] */
	int *d_samples = nullptr;
	int *h_samples_pinned = nullptr;
	std::vector<int> samples;
	PassTw tw0;

	/* staging ring: two halves, each host pinned + device mirror */
	size_t ring_bytes = 0;
	int ring_reads = 0; /* reads per half */
	uint8_t *h_ring[2] = { nullptr, nullptr };
	uint8_t *d_ring[2] = { nullptr, nullptr };
	cudaEvent_t ring_done[2] = { nullptr, nullptr };
	bool ring_busy[2] = { false, false };
	int cur_half = 0;
	std::vector<int> ring_hops;
	std::vector<uint8_t> hop_shadow; /* RTLSDR_GPU_FLAG_SHORT_READS: [tune_count][buf_len], the reference's tunes[i].buf8 */

	DescSlot desc[kDescSlots];
	int desc_next = 0;
	/* cached descriptors of recent regular (strided) batches, LRU */
	struct RegCache {
		RegularKey key;
		void *d_desc = nullptr;
		size_t cap = 0;
		std::vector<int4> segs;
		uint64_t stamp = 0;
	};
	std::vector<RegCache> reg_cache;
	uint64_t reg_stamp = 0;
	/* submit_batch: H2D copies run on their own stream, chunk by chunk, ahead of the kernels */
	/* decimating path: the (memory-bound) decimators of chunk k+1 overlap the (compute-bound)
	 * transform of chunk k on two auxiliary streams */
	cudaStream_t aux[2] = { nullptr, nullptr };
	cudaEvent_t fork_ev = nullptr, join_ev[2] = { nullptr, nullptr };
	cudaStream_t hb_head_stream = nullptr;  /* -F chain: head tiles beside the streaming kernel */
	cudaEvent_t hb_fork = nullptr, hb_join = nullptr;
	cudaStream_t copy_stream = nullptr;
	cudaEvent_t bulk_free = nullptr;   /* last kernel that reads d_bulk has finished */
	bool bulk_used = false;
	std::vector<cudaEvent_t> chunk_ready;

	/* scratch for decimation and the large-FFT path */
	uint8_t *d_scratch = nullptr;
	size_t scratch_bytes = 0;

	/* bulk H2D staging for submit_batch */
	uint8_t *d_bulk = nullptr;
	size_t bulk_bytes = 0;

	/* CSV rows (csv_text.cuh): column table of set_csv_columns(), per-row slots and lengths, and for
	 * collect_csv() the packed text and its length */
	int2 *d_csv_cols = nullptr;
	int csv_rows = 0;
	double csv_step = 0.0;
	char *d_csv_slots = nullptr;
	size_t csv_slot_bytes = 0;
	int *d_csv_lens = nullptr;
	char *d_csv_text = nullptr;
	size_t csv_text_bytes = 0;
	long long *d_csv_len = nullptr;
	long long *h_csv_len = nullptr; /* pinned */

	/* true while the last operation this handle put on its OWN stream was the report epilogue:
	 * only then may the next transform kernel be launched programmatically dependent (it reads
	 * nothing the epilogue writes before its pdl_wait) */
	bool last_was_epilogue = false;
	bool samples_on_device = false; /* set by merge_device(): collect() reads the counts back from d_smp64 */
	uint64_t launches = 0, h2d = 0, d2h = 0;
	/* timing of the transform kernels */
	std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timed;
	std::vector<cudaEvent_t> ev_pool;
	bool timing = false;
	int timing_every = 1;   /* bracket every k-th transform with events (events between kernels
	                         * prevent programmatic dependent launch, so benchmarks sample) */
	uint64_t timing_count = 0;

	/* debug / A-B switches, read from the environment ONCE at init (never on the launch path):
	 * RTLSDR_GPU_BOXCAR_STREAM = 0|1|2|3|5 forces the narrow-scan kernel variant,
	 * RTLSDR_GPU_NO_FUSED_BOXCAR / RTLSDR_GPU_NO_HB_STREAM fall back to the staged kernels */
	int dbg_boxcar_mode = -1;
	int dbg_stagger_ns = 0;
	bool dbg_no_fused_boxcar = false, dbg_no_hb_stream = false, dbg_rms_warp = false;
	int dbg_large_pipe = 1;

	std::string last_error;
};

namespace {

#define CU(call)                                                                                 \
	do {                                                                                         \
		cudaError_t _e = (call);                                                                 \
		if (_e != cudaSuccess) {                                                                 \
			h->last_error = std::string(#call) + ": " + cudaGetErrorString(_e);                  \
			return RTLSDR_GPU_ERR_CUDA;                                                          \
		}                                                                                        \
	} while (0)

int check_launch(rtlsdr_gpu_scan *h, const char *what)
{
	cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess) {
		h->last_error = std::string(what) + ": " + cudaGetErrorString(e);
		return RTLSDR_GPU_ERR_CUDA;
	}
	h->launches++;
	return 0;
}

/* ---- host tables (reference expressions, see header) ------------------- */

void host_sine_table(int m, int16_t *out)
{
	const int n = 1 << m, count = n * 3 / 4;
	for (int i = 0; i < count; i++) {
		double d = (double)i * 2.0 * M_PI / n;
		out[i] = (int16_t)(int)round(32767 * sin(d));
	}
}

typedef double (*window_fn)(int, int);
double win_rectangle(int, int) { return 1.0; }
double win_hamming(int i, int n)
{
	double a = 25.0 / 46.0, b = 21.0 / 46.0, n1 = (double)(n - 1);
	return a - b * cos(2 * i * M_PI / n1);
}
double win_blackman(int i, int n)
{
	double a0 = 7938.0 / 18608.0, a1 = 9240.0 / 18608.0, a2 = 1430.0 / 18608.0, n1 = (double)(n - 1);
	return a0 - a1 * cos(2 * i * M_PI / n1) + a2 * cos(4 * i * M_PI / n1);
}
double win_blackman_harris(int i, int n)
{
	double a0 = 0.35875, a1 = 0.48829, a2 = 0.14128, a3 = 0.01168, n1 = (double)(n - 1);
	return a0 - a1 * cos(2 * i * M_PI / n1) + a2 * cos(4 * i * M_PI / n1) - a3 * cos(6 * i * M_PI / n1);
}
double win_hann_poisson(int i, int n)
{
	double a = 2.0, n1 = (double)(n - 1);
	return 0.5 * (1 - cos(2 * M_PI * i / n1)) * pow(M_E, (-a * (double)abs((int)(n1 - 1 - 2 * i))) / n1);
}
double win_youssef(int i, int n)
{
	double a = 0.0025, n1 = (double)(n - 1);
	double w = win_blackman_harris(i, n);
	w *= pow(M_E, (-a * (double)abs((int)(n1 - 1 - 2 * i))) / n1);
	return w;
}
double win_bartlett(int i, int n)
{
	double l = (double)n, n1 = l - 1;
	double w = (i - n1 / 2) / (l / 2);
	if (w < 0)
		w = -w;
	return 1 - w;
}

/* cic_9_tables rows (rtl_power.c:219-232), entries [1..5] */
const int kCic9[11][5] = {
	{ 0, 0, 0, 0, 0 },
	{ -156, -97, 2798, -15489, 61019 },
	{ -128, -568, 5593, -24125, 74126 },
	{ -129, -639, 6187, -26281, 77511 },
	{ -122, -612, 6082, -26353, 77818 },
	{ -120, -602, 6015, -26269, 77757 },
	{ -120, -582, 5951, -26128, 77542 },
	{ -119, -580, 5931, -26094, 77505 },
	{ -119, -578, 5921, -26077, 77484 },
	{ -119, -577, 5917, -26067, 77473 },
	{ -199, -362, 5303, -25505, 77489 },
};

/* ---- init ------------------------------------------------------------- */

/* the handle's debug / A-B switches (see rtlsdr_gpu_scan), read from the environment */
int read_debug_switches(rtlsdr_gpu_scan *h)
{
	if (const char *f = getenv("RTLSDR_GPU_BOXCAR_STREAM")) {
		const int m = atoi(f);
		if (m != 0 && m != 1 && m != 2 && m != 3 && m != 5)
			return RTLSDR_GPU_ERR_CONFIG; /* not a kernel variant */
		h->dbg_boxcar_mode = m;
	}
	h->dbg_no_fused_boxcar = getenv("RTLSDR_GPU_NO_FUSED_BOXCAR") != nullptr;
	if (const char *f = getenv("RTLSDR_GPU_STAGGER_NS"))
		h->dbg_stagger_ns = atoi(f);
	h->dbg_no_hb_stream = getenv("RTLSDR_GPU_NO_HB_STREAM") != nullptr;
	if (const char *f = getenv("RTLSDR_GPU_LARGE_PIPE")) /* A/B switch: 0 = one-tile-per-CTA round B for N >= 2^17 */
		h->dbg_large_pipe = atoi(f) != 0;
	h->dbg_rms_warp = getenv("RTLSDR_GPU_RMS_WARP") != nullptr; /* 1-bin hops: warp-per-read kernel instead of CTA-per-read */
	return 0;
}

/* device buffer of `bytes`, each set to `byte` on stream s.  A failed allocation sets *rc. */
template <class T>
bool alloc_fill(T **dst, size_t bytes, int byte, cudaStream_t s, int *rc)
{
	if (cudaMalloc(dst, bytes) != cudaSuccess) {
		*rc = RTLSDR_GPU_ERR_NOMEM;
		return false;
	}
	return cudaMemsetAsync(*dst, byte, bytes, s) == cudaSuccess;
}

/* device copy of a host table; an empty table stays nullptr.  A failed allocation sets *rc. */
template <class T>
bool upload(T **dst, const std::vector<T> &v, int *rc)
{
	if (v.empty())
		return true;
	if (cudaMalloc(dst, v.size() * sizeof(T)) != cudaSuccess) {
		*rc = RTLSDR_GPU_ERR_NOMEM;
		return false;
	}
	return cudaMemcpy(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice) == cudaSuccess;
}

/* ---- events for kernel timing ----------------------------------------- */

cudaEvent_t get_event(rtlsdr_gpu_scan *h)
{
	cudaEvent_t e = nullptr;
	if (!h->ev_pool.empty()) {
		e = h->ev_pool.back();
		h->ev_pool.pop_back();
		return e;
	}
	if (cudaEventCreate(&e) != cudaSuccess)
		return nullptr;
	return e;
}

struct TimedScope {
	rtlsdr_gpu_scan *h;
	cudaEvent_t a = nullptr, b = nullptr;
	explicit TimedScope(rtlsdr_gpu_scan *hh) : h(hh)
	{
		if (!h->timing || (h->timing_count++ % (uint64_t)h->timing_every) != 0)
			return;
		h->last_was_epilogue = false;
		a = get_event(h);
		b = get_event(h);
		if (a && b)
			cudaEventRecord(a, h->stream);
	}
	~TimedScope()
	{
		if (a && b) {
			cudaEventRecord(b, h->stream);
			h->timed.push_back({ a, b });
		}
	}
};

/* ---- descriptor upload ------------------------------------------------- */

int desc_acquire(rtlsdr_gpu_scan *h, size_t bytes, DescSlot **out)
{
	DescSlot &s = h->desc[h->desc_next];
	h->desc_next = (h->desc_next + 1) % kDescSlots;
	if (s.used)
		CU(cudaEventSynchronize(s.done));
	if (s.cap < bytes) {
		size_t cap = std::max(bytes, (size_t)1 << 16);
		if (s.h)
			cudaFreeHost(s.h);
		if (s.d)
			cudaFree(s.d);
		s.h = s.d = nullptr;
		s.cap = 0;
		CU(cudaMallocHost(&s.h, cap));
		CU(cudaMalloc(&s.d, cap));
		s.cap = cap;
	}
	if (!s.done)
		CU(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
	*out = &s;
	return 0;
}

int ensure_scratch(rtlsdr_gpu_scan *h, size_t bytes)
{
	if (h->scratch_bytes >= bytes)
		return 0;
	if (h->d_scratch) {
		CU(cudaStreamSynchronize(h->stream));
		cudaFree(h->d_scratch);
		h->d_scratch = nullptr;
		h->scratch_bytes = 0;
	}
	if (cudaMalloc(&h->d_scratch, bytes) != cudaSuccess) {
		cudaGetLastError();
		h->last_error = "cudaMalloc(scratch) failed";
		return RTLSDR_GPU_ERR_NOMEM;
	}
	h->scratch_bytes = bytes;
	return 0;
}

/* Layout of a descriptor blob: [read_off: n_reads x int64][segs: n_segs x int4][hop_of: n_reads x int] */
struct DescLayout {
	size_t off_reads, off_segs, off_hops, bytes;
	DescLayout(int n_reads, int n_segs)
	{
		off_reads = 0;
		off_segs = ((size_t)n_reads * 8 + 15) & ~(size_t)15;
		off_hops = off_segs + (size_t)n_segs * 16;
		bytes = off_hops + (size_t)n_reads * 4;
	}
};

/*
 * Sort the batch's reads by hop and cut each hop's run into segments of about
 * `total / target` reads.  Returns segment count.
 */
int build_desc(rtlsdr_gpu_scan *h, const std::vector<long long> &offs, const std::vector<int> &hops,
	       std::vector<long long> &s_offs, std::vector<int> &s_hops, std::vector<int4> &segs)
{
	const int n = (int)offs.size(), tc = h->cfg.tune_count;
	if (h->shape.path == PATH_RMS) {
		/* 1-bin hops: every read is reduced on its own (one atomic per read), so the reads keep their
		 * submission order = address order; sorting them by hop would turn the resident CTAs' working window
		 * from one contiguous stretch into 16 KiB pieces a whole sweep apart */
		s_offs = offs;
		s_hops = hops;
		segs.clear();
		return 0;
	}
	std::vector<int> count(tc + 1, 0);
	for (int i = 0; i < n; i++)
		count[hops[i] + 1]++;
	for (int i = 0; i < tc; i++)
		count[i + 1] += count[i];
	s_offs.resize(n);
	s_hops.resize(n);
	std::vector<int> cursor(count.begin(), count.end() - 1);
	for (int i = 0; i < n; i++) {
		int p = cursor[hops[i]]++;
		s_offs[p] = offs[i];
		s_hops[p] = hops[i];
	}
	segs.clear();
	if (h->shape.path == PATH_SMALL_U8 || h->shape.path == PATH_RMS || h->shape.path == PATH_LARGE)
		return 0; /* these kernels walk the hop-sorted reads themselves (equal runs per CTA / per-read work) */
	/* the decimating path runs in kDecimChunks chunks, each should still fill the GPU */
	const bool big_decim = h->shape.path == PATH_SMALL_DECIM && (size_t)n * (size_t)h->cfg.buf_len >= kDecimOverlapBytes;
	const int target = std::max(1, h->num_sms * h->ctas_per_sm) * (big_decim ? kDecimChunks : 1);
	int chunk = std::max(1, (n + target - 1) / target);
	/*
	 * A hop is at least one segment, so with many hops (or reads per hop that `chunk` does not divide) the
	 * default can leave a mostly empty last wave of CTAs: 623 hops x 16 reads on 296 slots = 3 rounds of 16
	 * reads where 33.7 per slot would do.  Among the shorter segment lengths pick the one with the smallest
	 * makespan: rounds of resident CTAs x (reads per segment + the cost of a segment's flush and pipeline fill).
	 */
	{
		const double per_seg = 0.35; /* flush + cold first load of a segment, in units of one read */
		double best = 1e300;
		int best_chunk = chunk;
		for (int k = 1; k <= 16; k++) {
			const int c = std::max(1, (chunk + k - 1) / k);
			long long nseg = 0;
			for (int hp = 0; hp < tc; hp++) {
				const int cnt = count[hp + 1] - count[hp];
				nseg += (cnt + c - 1) / c;
			}
			const long long rounds = (nseg + target - 1) / target;
			const double cost = (double)rounds * (c + per_seg);
			if (cost < best * 0.98) { /* prefer longer segments unless the gain is real */
				best = cost;
				best_chunk = c;
			}
			if (c == 1)
				break;
		}
		chunk = best_chunk;
	}
	for (int hp = 0; hp < tc; hp++) {
		int lo = count[hp], hi = count[hp + 1];
		int cnt = hi - lo;
		if (cnt <= 0)
			continue;
		int pieces = (cnt + chunk - 1) / chunk;
		for (int k = 0; k < pieces; k++) {
			int a = lo + (int)((long long)cnt * k / pieces), b = lo + (int)((long long)cnt * (k + 1) / pieces);
			if (b > a)
				segs.push_back(make_int4(hp, a, b - a, 0));
		}
	}
	return (int)segs.size();
}

/* ---- kernel dispatch --------------------------------------------------- */

int large_process(rtlsdr_gpu_scan *h, const uint8_t *base, const long long *d_offs, const int *d_hops, int n_reads);

/*
 * Launch a transform kernel; when the report epilogue is the previous kernel on the handle's own stream, as a
 * programmatic dependent launch: the epilogue calls griddepcontrol.launch_dependents at its top, the kernel reads
 * only its own inputs until griddepcontrol.wait in front of its first accumulator update, so the report costs no
 * time on the transform's critical path.  Every kernel launched through here has that wait (pdl_wait()).
 */
template <class K, class P>
int launch_after_epilogue(rtlsdr_gpu_scan *h, K kern, int grid, int block, int smem, const P &prm, bool allow_pdl = true)
{
	if (allow_pdl && h->last_was_epilogue && h->stream == h->own_stream) {
		cudaLaunchConfig_t cfg = {};
		cfg.gridDim = dim3(grid);
		cfg.blockDim = dim3(block);
		cfg.dynamicSmemBytes = smem;
		cfg.stream = h->stream;
		cudaLaunchAttribute attr[1];
		attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
		attr[0].val.programmaticStreamSerializationAllowed = 1;
		cfg.attrs = attr;
		cfg.numAttrs = 1;
		CU(cudaLaunchKernelEx(&cfg, kern, prm));
	} else {
		kern<<<grid, block, smem, h->stream>>>(prm);
	}
	h->last_was_epilogue = false;
	return 0;
}

template <int L, bool PEAK, bool IN16>
int launch_small_t(rtlsdr_gpu_scan *h, const SmallParams &prm)
{
	auto kern = scan_small_kernel<L, PEAK, IN16>;
	const int smem = SmallSmem<L>::bytes;
	static bool attr_set[64] = { false }; /* once per kernel instance and device, not per launch */
	if (h->cfg.device >= 64 || !attr_set[h->cfg.device]) {
		CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
		if (h->cfg.device < 64)
			attr_set[h->cfg.device] = true;
	}
	/* u8 reads: one resident wave of persistent CTAs, each with an equal share of the working sets;
	 * decimated images: one CTA per segment */
	const int grid = IN16 ? std::min(prm.n_segs, h->num_sms * 8)
			      : (int)std::min<long long>(2ll * prm.n_entries, (long long)h->num_sms * h->ctas_per_sm);
	if (int rc = launch_after_epilogue(h, kern, grid, kThreads, smem, prm, !IN16))
		return rc;
	return check_launch(h, "scan_small_kernel");
}

template <int L>
int launch_small_l(rtlsdr_gpu_scan *h, const SmallParams &prm, bool in16)
{
	if (h->cfg.peak_hold)
		return in16 ? launch_small_t<L, true, true>(h, prm) : launch_small_t<L, true, false>(h, prm);
	return in16 ? launch_small_t<L, false, true>(h, prm) : launch_small_t<L, false, false>(h, prm);
}

int launch_small(rtlsdr_gpu_scan *h, const SmallParams &prm, bool in16)
{
	switch (h->cfg.bin_e) {
	case 1: return launch_small_l<1>(h, prm, in16);
	case 2: return launch_small_l<2>(h, prm, in16);
	case 3: return launch_small_l<3>(h, prm, in16);
	case 4: return launch_small_l<4>(h, prm, in16);
	case 5: return launch_small_l<5>(h, prm, in16);
	case 6: return launch_small_l<6>(h, prm, in16);
	case 7: return launch_small_l<7>(h, prm, in16);
	case 8: return launch_small_l<8>(h, prm, in16);
	case 9: return launch_small_l<9>(h, prm, in16);
	case 10: return launch_small_l<10>(h, prm, in16);
	case 11: return launch_small_l<11>(h, prm, in16);
	case 12: return launch_small_l<12>(h, prm, in16);
	default: break;
	}
	return RTLSDR_GPU_ERR_CONFIG;
}

template <int L, bool PEAK, int NS>
int launch_fused_boxcar_t(rtlsdr_gpu_scan *h, const FusedBoxcarParams &prm)
{
	auto k = scan_boxcar_fused_kernel<L, PEAK, NS>;
	const int smem = FusedSmem<L>::bytes(prm.ds, NS);
	const int grid = std::min(prm.n_segs, h->num_sms * 8);
	CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
	if (int rc = launch_after_epilogue(h, k, grid, kThreads, smem, prm))
		return rc;
	return check_launch(h, "scan_boxcar_fused_kernel");
}

template <int L>
int launch_fused_boxcar_l(rtlsdr_gpu_scan *h, const FusedBoxcarParams &prm_in)
{
	FusedBoxcarParams prm = prm_in;
	/*
	 * Staging ring depth.  Two CTAs per SM (one streams while the other transforms) with 4 or
	 * 3 slots each is the measured best; only when not even 3 slots fit twice (ds > ~40) one
	 * CTA per SM with as many slots as fit takes over (measured at ds = 56: 274 -> 250 us;
	 * at ds = 28 one CTA with 8 slots was slower than two with 3: 197 vs 130 us).
	 */
	const int limit = 227 * 1024 - 1024;
	int slots;
	if (2 * (FusedSmem<L>::bytes(prm.ds, 4) + 1024) <= 227 * 1024) {
		slots = 4;
	} else if (2 * (FusedSmem<L>::bytes(prm.ds, 3) + 1024) <= 227 * 1024) {
		slots = 3;
	} else {
		const int fit = (limit - FusedSmem<L>::off_stage) / (512 * prm.ds);
		slots = fit >= 12 ? 12 : fit >= 8 ? 8 : fit >= 6 ? 6 : fit >= 4 ? 4 : fit >= 3 ? 3 : 2;
	}
	prm.slots = slots;
	const bool pk = h->cfg.peak_hold != 0;
#define FUSED_CASE(NSV)                                                                               \
	case NSV:                                                                                     \
		return pk ? launch_fused_boxcar_t<L, true, NSV>(h, prm) : launch_fused_boxcar_t<L, false, NSV>(h, prm)
	switch (slots) {
		FUSED_CASE(12);
		FUSED_CASE(8);
		FUSED_CASE(6);
		FUSED_CASE(4);
		FUSED_CASE(3);
	default:
		return pk ? launch_fused_boxcar_t<L, true, 2>(h, prm) : launch_fused_boxcar_t<L, false, 2>(h, prm);
	}
#undef FUSED_CASE
}

/*
 * Warp-specialised variant (producer / boxcar / transform roles, one CTA per SM).  The
 * single-role kernel's time is the SUM of its streaming and transform phases, this one's is
 * their maximum; measured faster for every ds (ds = 28: 53 -> 72 % of the HBM copy peak), so the
 * single-role kernel is only the fallback when the ring does not fit.
 * RTLSDR_GPU_BOXCAR_STREAM=0 / 1 / 2 / 3 forces the choice (A/B measurements, tests).
 */
constexpr int kStreamMinDs = 2; /* every boxcar factor (measured down to ds = 2: +20..30 % over the single-role kernel) */
constexpr int kStreamOneFftGroupDs = 24; /* from here on one transform group keeps up and leaves its registers unspilled */

template <int L, int FG>
int stream_boxcar_slots(int ds)
{
	const int fit = (227 * 1024 - StreamSmem<L, FG>::off_stage) / (512 * ds);
	return std::min(fit, kStreamMaxSlots);
}

template <int L, bool PEAK, int FG, int BG>
int launch_stream_boxcar_t(rtlsdr_gpu_scan *h, const FusedBoxcarParams &prm_in)
{
	FusedBoxcarParams prm = prm_in;
	prm.slots = stream_boxcar_slots<L, FG>(prm.ds);
	if (BG == 2)
		prm.slots &= ~1; /* even: a slot then always serves the same boxcar group, which sees every phase of its barriers */
	const int smem = StreamSmem<L, FG>::bytes(prm.ds, prm.slots);
	const int grid = std::min(prm.n_segs, h->num_sms);
	auto k = scan_boxcar_stream_kernel<L, PEAK, FG, BG>;
	CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
	if (int rc = launch_after_epilogue(h, k, grid, StreamShape<FG, BG>::threads, smem, prm))
		return rc;
	return check_launch(h, "scan_boxcar_stream_kernel");
}

template <int L>
int sym_boxcar_slots(int ds)
{
	const int fit = (227 * 1024 - SymSmem<L>::off_stage) / (512 * ds) / kSymGroups; /* per pipeline */
	return std::min(fit, kStreamMaxSlots);
}

/* symmetric worker groups (scan_boxcar_sym_kernel) */
template <int L, bool PEAK>
int launch_sym_boxcar_t(rtlsdr_gpu_scan *h, const FusedBoxcarParams &prm_in)
{
	FusedBoxcarParams prm = prm_in;
	prm.slots = sym_boxcar_slots<L>(prm.ds);
	const int smem = SymSmem<L>::bytes(prm.ds, prm.slots);
	const int grid = std::min(prm.n_segs, h->num_sms);
	auto k = scan_boxcar_sym_kernel<L, PEAK>;
	CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
	if (int rc = launch_after_epilogue(h, k, grid, kSymThreads, smem, prm))
		return rc;
	return check_launch(h, "scan_boxcar_sym_kernel");
}

/* 0 = single-role kernel; transform groups + boxcar groups: 1 = 1 + 2, 2 = 2 + 1, 3 = 2 + 2; 5 = symmetric workers */
template <int L>
int stream_boxcar_mode(const rtlsdr_gpu_scan *h)
{
	const int ds = h->cfg.downsample;
	/* measured on B200 (profiles/r01l_stream_modes.txt, r01n_stream_modes.txt): up to 512 bins and, at 1024 bins,
	 * below ds ~ 24 the symmetric worker kernel wins (N = 256: +25 %, N = 512: +8..16 %); the three-role kernel
	 * keeps the large-ds and the 2048 / 4096-bin cases (there the symmetric kernel's two rings get too shallow),
	 * with a second transform group below ds ~ 24 */
	int mode;
	if (ds < kStreamMinDs)
		mode = 0;
	else if (L <= 9 || (L == 10 && ds < kStreamOneFftGroupDs))
		mode = 5;
	else
		mode = ds < kStreamOneFftGroupDs ? 3 : 1;
	if (h->dbg_boxcar_mode >= 0)
		mode = h->dbg_boxcar_mode;
	if (mode == 5 && sym_boxcar_slots<L>(ds) < 3)
		mode = 1;
	if (mode == 1 && stream_boxcar_slots<L, 1>(ds) < 4)
		mode = 0;
	if ((mode == 2 || mode == 3) && stream_boxcar_slots<L, 2>(ds) < 4)
		mode = 0;
	return mode;
}

template <int L>
int launch_stream_boxcar_l(rtlsdr_gpu_scan *h, const FusedBoxcarParams &prm, int mode)
{
	const bool pk = h->cfg.peak_hold != 0;
	if (mode == 5)
		return pk ? launch_sym_boxcar_t<L, true>(h, prm) : launch_sym_boxcar_t<L, false>(h, prm);
	if (mode == 1)
		return pk ? launch_stream_boxcar_t<L, true, 1, 2>(h, prm) : launch_stream_boxcar_t<L, false, 1, 2>(h, prm);
	if (mode == 2)
		return pk ? launch_stream_boxcar_t<L, true, 2, 1>(h, prm) : launch_stream_boxcar_t<L, false, 2, 1>(h, prm);
	return pk ? launch_stream_boxcar_t<L, true, 2, 2>(h, prm) : launch_stream_boxcar_t<L, false, 2, 2>(h, prm);
}

int launch_fused_boxcar(rtlsdr_gpu_scan *h, const FusedBoxcarParams &prm)
{
#define STREAM_CASE(LV)                                                                               \
	case LV:                                                                                      \
		if (int mode = stream_boxcar_mode<LV>(h))                                             \
			return launch_stream_boxcar_l<LV>(h, prm, mode);                              \
		break
	switch (h->cfg.bin_e) {
		STREAM_CASE(8);
		STREAM_CASE(9);
		STREAM_CASE(10);
		STREAM_CASE(11);
		STREAM_CASE(12);
	default: break;
	}
#undef STREAM_CASE
	switch (h->cfg.bin_e) {
	case 8: return launch_fused_boxcar_l<8>(h, prm);
	case 9: return launch_fused_boxcar_l<9>(h, prm);
	case 10: return launch_fused_boxcar_l<10>(h, prm);
	case 11: return launch_fused_boxcar_l<11>(h, prm);
	case 12: return launch_fused_boxcar_l<12>(h, prm);
	default: return RTLSDR_GPU_ERR_CONFIG;
	}
}

/* narrow boxcar scans whose every read is exactly one FFT block: one fused kernel */
bool fused_boxcar_ok(const rtlsdr_gpu_scan *h)
{
	const int ds = h->cfg.downsample;
	return h->cfg.boxcar && ds >= 2 && ds <= 64 && h->cfg.bin_e >= 8 && h->cfg.bin_e <= 12 && h->shape.n_blocks == 1 &&
	       h->cfg.buf_len == 2 * h->shape.N * ds && !h->dbg_no_fused_boxcar;
}

/*
 * Decimate entries [e0, e0+n) (u8 reads at base + d_offs[e]) into c16 images in
 * scratch and compute their DC sums.  Scratch layout for n entries:
 *   [images n x image_stride c16][bufA n x pairs/2 c16][bufB n x pairs/4 c16][sums n x 2 int64]
 */
struct DecimScratch {
	c16 *img, *a, *b;
	long long *sums;
	int *ave;
	static bool halfband(const rtlsdr_gpu_scan *h)
	{
		return !(h->cfg.boxcar && h->cfg.downsample > 1) && h->cfg.downsample_passes > kChainMaxPasses;
	}
	/* bytes per entry (the 16 KiB of slack after the images is added by the caller) */
	static size_t per_entry(const rtlsdr_gpu_scan *h)
	{
		size_t pairs = (size_t)h->cfg.buf_len / 2;
		size_t b = (size_t)h->shape.image_stride * 4 + 16 + 8;
		if (halfband(h))
			b += (pairs / 2) * 4 + (pairs / 4 + 4) * 4;
		return b;
	}
	static size_t slack() { return kStageBytes + 1024; }
	DecimScratch(const rtlsdr_gpu_scan *h, int n, uint8_t *p)
	{
		size_t pairs = (size_t)h->cfg.buf_len / 2;
		img = (c16 *)p;
		p += (size_t)n * h->shape.image_stride * 4 + kStageBytes; /* a unit may read past the last image */
		a = b = nullptr;
		if (halfband(h)) {
			a = (c16 *)p;
			p += (size_t)n * (pairs / 2) * 4;
			b = (c16 *)p;
			p += (size_t)n * (pairs / 4 + 4) * 4;
		}
		p = (uint8_t *)(((uintptr_t)p + 15) & ~(uintptr_t)15);
		sums = (long long *)p;
		p += (size_t)n * 16;
		ave = (int *)p;
	}
};

int run_decimators(rtlsdr_gpu_scan *h, const uint8_t *base, const long long *d_offs, int n, const DecimScratch &sc)
{
	const int pairs = h->cfg.buf_len / 2;
	const int img_count = (int)h->shape.image_stride;
	int rc;
	if (h->cfg.boxcar && h->cfg.downsample > 1) {
		DecimParams p;
		p.base = base;
		p.read_off = d_offs;
		p.n_reads = n;
		p.pairs = pairs;
		p.ds = h->cfg.downsample;
		p.out = sc.img;
		p.out_stride = h->shape.image_stride;
		p.out_count = img_count;
		p.l_len = h->shape.l_len;
		p.sums = sc.sums;
		CU(cudaMemsetAsync(sc.sums, 0, (size_t)n * 16, h->stream));
		dim3 grid((img_count + 255) / 256, n);
		const int bytes = 2 * h->cfg.downsample;
		if (h->cfg.downsample <= kBoxcarStageMaxDs)
			boxcar_staged_kernel<<<grid, 256, 512 * h->cfg.downsample, h->stream>>>(p);
		else if (bytes % 16 == 0)
			boxcar_kernel<16><<<grid, 256, 0, h->stream>>>(p);
		else if (bytes % 8 == 0)
			boxcar_kernel<8><<<grid, 256, 0, h->stream>>>(p);
		else if (bytes % 4 == 0)
			boxcar_kernel<4><<<grid, 256, 0, h->stream>>>(p);
		else
			boxcar_kernel<2><<<grid, 256, 0, h->stream>>>(p);
		if ((rc = check_launch(h, "boxcar_kernel"))) /* DC sums are fused into the boxcar kernel */
			return rc;
	} else if (h->cfg.downsample_passes <= kChainMaxPasses) {
		/* fused fifth_order chain + FIR + DC sums, one kernel */
		const int passes = h->cfg.downsample_passes;
		const int M = pairs >> passes;
		HalfbandChainParams p;
		p.base = base;
		p.read_off = d_offs;
		p.pairs = pairs;
		p.passes = passes;
		p.use_fir = (h->cfg.comp_fir_size == 9 && passes <= 10) ? 1 : 0;
		const int *row = kCic9[passes];
		p.f1 = row[0]; p.f2 = row[1]; p.f3 = row[2]; p.f4 = row[3]; p.f5 = row[4];
		p.out = sc.img;
		p.out_stride = h->shape.image_stride;
		p.l_len = h->shape.l_len;
		p.sums = sc.sums;
		/* P <= 5: the register-streaming kernel computes final samples >= 16, the tile kernel only
		 * the eased-in head [0, 16) of every read (RTLSDR_GPU_NO_HB_STREAM=1: tile kernel for all) */
		const bool stream = passes <= kHbStreamMaxPasses && M >= 2 * kHbStreamHead && !h->dbg_no_hb_stream;
		const int smem = chain_tile(p, stream);
		CU(cudaFuncSetAttribute(halfband_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
		CU(cudaMemsetAsync(sc.sums, 0, (size_t)n * 16, h->stream));
		dim3 grid(stream ? 1 : (M + p.tile - 1) / p.tile, n);
		/* With the streaming kernel the tile kernel only computes the eased-in heads (final samples 0..15 of
		 * every read): small latency-bound CTAs that write other words than the streaming kernel and share
		 * only the atomically updated DC sums -- they run beside it on a stream of their own instead of in
		 * front of it (19 us of a 200 us step at -F 9, ds = 16). */
		cudaStream_t head_stream = h->stream;
		if (stream) {
			if (!h->hb_head_stream) {
				CU(cudaStreamCreateWithFlags(&h->hb_head_stream, cudaStreamNonBlocking));
				CU(cudaEventCreateWithFlags(&h->hb_fork, cudaEventDisableTiming));
				CU(cudaEventCreateWithFlags(&h->hb_join, cudaEventDisableTiming));
			}
			head_stream = h->hb_head_stream;
			CU(cudaEventRecord(h->hb_fork, h->stream)); /* behind the memset of the sums and whatever produced the input */
			CU(cudaStreamWaitEvent(head_stream, h->hb_fork, 0));
		}
		halfband_chain_kernel<<<grid, stream ? 64 : 256, smem, head_stream>>>(p);
		if ((rc = check_launch(h, "halfband_chain_kernel")))
			return rc;
		if (stream)
			CU(cudaEventRecord(h->hb_join, head_stream));
		if (stream) {
			HalfbandStreamParams q;
			q.base = base;
			q.read_off = d_offs;
			q.n_reads = n;
			q.pairs = pairs;
			q.use_fir = p.use_fir;
			q.f1 = p.f1; q.f2 = p.f2; q.f3 = p.f3; q.f4 = p.f4; q.f5 = p.f5;
			q.out = sc.img;
			q.out_stride = h->shape.image_stride;
			q.l_len = h->shape.l_len;
			q.sums = sc.sums;
			/* span: as long as possible (16 warm-up samples per span are recomputed) while the grid
			 * still fills at least half of the resident thread slots (640 per SM at 87 registers) */
			int span = M;
			while (span > 64 && (long long)n * ((M + span - 1) / span) < (long long)h->num_sms * 256)
				span /= 2;
			q.span = span;
			const long long threads = (long long)n * ((M + span - 1) / span);
			const int blocks = (int)((threads + 127) / 128);
			switch (passes) {
			case 1: halfband_stream_kernel<1><<<blocks, 128, 0, h->stream>>>(q); break;
			case 2: halfband_stream_kernel<2><<<blocks, 128, 0, h->stream>>>(q); break;
			case 3: halfband_stream_kernel<3><<<blocks, 128, 0, h->stream>>>(q); break;
			case 4: halfband_stream_kernel<4><<<blocks, 128, 0, h->stream>>>(q); break;
			default: halfband_stream_kernel<5><<<blocks, 128, 0, h->stream>>>(q); break;
			}
			if ((rc = check_launch(h, "halfband_stream_kernel")))
				return rc;
			CU(cudaStreamWaitEvent(h->stream, h->hb_join, 0)); /* heads done before the DC constants / the transform */
		}
	} else {
		const int passes = h->cfg.downsample_passes;
		const c16 *cur = nullptr;
		long long cur_stride = 0;
		int count = pairs;
		for (int j = 0; j < passes; j++) {
			HalfbandParams p;
			c16 *dst = (j & 1) ? sc.b : sc.a;
			long long dst_stride = (j & 1) ? (pairs / 4 + 4) : (pairs / 2);
			p.in = j == 0 ? (const void *)base : (const void *)cur;
			p.read_off = d_offs;
			p.in_stride = cur_stride;
			p.out = dst;
			p.out_stride = dst_stride;
			p.n_out = count / 2;
			dim3 grid((p.n_out + 255) / 256, n);
			if (j == 0)
				halfband_kernel<true><<<grid, 256, 0, h->stream>>>(p);
			else
				halfband_kernel<false><<<grid, 256, 0, h->stream>>>(p);
			if ((rc = check_launch(h, "halfband_kernel")))
				return rc;
			cur = dst;
			cur_stride = dst_stride;
			count /= 2;
		}
		FirParams f;
		f.in = cur;
		f.in_stride = cur_stride;
		f.out = sc.img;
		f.out_stride = h->shape.image_stride;
		f.count = count;
		f.use_fir = (h->cfg.comp_fir_size == 9 && passes <= 10) ? 1 : 0;
		const int *row = kCic9[passes <= 10 ? passes : 0];
		f.f1 = row[0]; f.f2 = row[1]; f.f3 = row[2]; f.f4 = row[3]; f.f5 = row[4];
		dim3 grid((count + 255) / 256, n);
		fir9_kernel<<<grid, 256, 0, h->stream>>>(f);
		if ((rc = check_launch(h, "fir9_kernel")))
			return rc;
		CU(cudaMemsetAsync(sc.sums, 0, (size_t)n * 16, h->stream));
		DcSumParams d;
		d.img = sc.img;
		d.stride = h->shape.image_stride;
		d.l_len = h->shape.l_len;
		d.sums = sc.sums;
		int nI = (h->shape.l_len + 1) / 2;
		dim3 grid_dc(std::max(1, std::min((nI + 1023) / 1024, 64)), n);
		dc_sums_c16_kernel<<<grid_dc, 256, 0, h->stream>>>(d);
		if ((rc = check_launch(h, "dc_sums_c16_kernel")))
			return rc;
	}
	DcFinalizeParams f;
	f.sums = sc.sums;
	f.ave = sc.ave;
	f.n = n;
	f.l_len = h->shape.l_len;
	dc_finalize_kernel<<<(2 * n + 255) / 256, 256, 0, h->stream>>>(f);
	return check_launch(h, "dc_finalize_kernel");
}

/*
 * Process one batch of reads already on the device.  `d_desc` holds the
 * descriptor blob (sorted read offsets, segments, hop per read).
 */
int launch_batch(rtlsdr_gpu_scan *h, const uint8_t *base, const uint8_t *d_desc, int n_reads, int n_segs,
		 const std::vector<int4> *segs_host)
{
	DescLayout lay(n_reads, n_segs);
	const long long *d_offs = (const long long *)(d_desc + lay.off_reads);
	const int4 *d_segs = (const int4 *)(d_desc + lay.off_segs);
	const int *d_hops = (const int *)(d_desc + lay.off_hops);
	int rc = 0;
	/* paths whose first kernel after a report is a transform kernel with a pdl_wait() keep the flag */
	const bool pdl_path = h->shape.path == PATH_SMALL_U8 || h->shape.path == PATH_RMS ||
			      (h->shape.path == PATH_SMALL_DECIM && fused_boxcar_ok(h));
	if (!pdl_path || h->d_level)
		h->last_was_epilogue = false;

	if (h->d_level) {
		LevelParams lp;
		lp.base = base;
		lp.read_off = d_offs;
		lp.hop_of = d_hops;
		lp.n_reads = n_reads;
		lp.buf_len = h->cfg.buf_len;
		lp.level = h->d_level;
		const int blocks = std::max(1, std::min((n_reads + 7) / 8, h->num_sms * 8));
		level_stats_kernel<<<blocks, 256, 0, h->stream>>>(lp);
		if ((rc = check_launch(h, "level_stats_kernel")))
			return rc;
	}

	if (h->shape.path == PATH_RMS) {
		RmsParams p;
		p.base = base;
		p.read_off = d_offs;
		p.hop_of = d_hops;
		p.n_reads = n_reads;
		p.buf_len = h->cfg.buf_len;
		p.peak = h->cfg.peak_hold;
		p.avg = h->d_avg;
		p.samples = h->d_smp64;
		TimedScope ts(h);
		if (h->cfg.buf_len == kRmsCtaBytes && !h->dbg_rms_warp) {
			/* one CTA per read, eight resident CTAs per SM */
			const int blocks = std::max(1, std::min(n_reads, h->num_sms * 8));
			if ((rc = launch_after_epilogue(h, rms_cta_kernel, blocks, 256, 0, p)))
				return rc;
			return check_launch(h, "rms_cta_kernel");
		}
		const int blocks = std::max(1, std::min((n_reads + 7) / 8, h->num_sms * 8));
		if ((rc = launch_after_epilogue(h, rms_kernel, blocks, 256, 0, p)))
			return rc;
		return check_launch(h, "rms_kernel");
	}

	if (h->shape.path == PATH_SMALL_U8) {
		SmallParams p;
		memset(&p, 0, sizeof(p));
		p.base = base;
		p.read_off = d_offs;
		p.hop_of = d_hops;
		p.n_entries = n_reads;
		p.stagger_ns = h->dbg_stagger_ns;
		p.avg = h->d_avg;
		p.samples = h->d_smp64;
		p.samples_per_read = h->shape.samples_per_read;
		p.tw = h->d_tw;
		p.twc = h->d_twc;
		p.win = h->d_win;
		p.tw0 = h->tw0;
		TimedScope ts(h);
		return launch_small(h, p, false);
	}

	if (h->shape.path == PATH_SMALL_DECIM && fused_boxcar_ok(h)) {
		FusedBoxcarParams p;
		memset(&p, 0, sizeof(p));
		p.base = base;
		p.read_off = d_offs;
		p.segs = d_segs;
		p.n_segs = n_segs;
		p.ds = h->cfg.downsample;
		p.avg = h->d_avg;
		p.samples = h->d_smp64;
		p.twc = h->d_twc;
		p.win = h->d_win;
		p.tw0 = h->tw0;
		TimedScope ts(h);
		return launch_fused_boxcar(h, p);
	}

	if (h->shape.path == PATH_SMALL_DECIM) {
		/* Entries are processed in chunks cut at segment boundaries.  Chunks alternate between
		 * two auxiliary streams and two scratch halves, so the decimators of one chunk (HBM
		 * bound) run while the transform of the previous one (issue bound) is still busy. */
		const size_t per = DecimScratch::per_entry(h);
		const int max_entries = (int)std::max<size_t>(1, (kScratchBudget / 2) / per);
		if (!segs_host)
			return RTLSDR_GPU_ERR_CONFIG;
		const int n_chunks = ((size_t)n_reads * (size_t)h->cfg.buf_len >= kDecimOverlapBytes) ? kDecimChunks : 1;
		const int want = std::max(1, std::min(max_entries, (n_reads + n_chunks - 1) / n_chunks));
		/* chunk boundaries first: the scratch must fit the largest one */
		std::vector<std::pair<size_t, size_t>> chunks;
		int cnt_max = 0;
		for (size_t si = 0; si < segs_host->size();) {
			size_t sj = si;
			int cnt = 0;
			while (sj < segs_host->size() && (cnt == 0 || cnt + (*segs_host)[sj].z <= want)) {
				cnt += (*segs_host)[sj].z;
				sj++;
			}
			cnt_max = std::max(cnt_max, cnt);
			chunks.push_back({ si, sj });
			si = sj;
		}
		const size_t half = ((per * (size_t)cnt_max + DecimScratch::slack()) + 255) & ~(size_t)255;
		if ((rc = ensure_scratch(h, 2 * half)))
			return rc;
		if (!h->aux[0]) {
			for (int i = 0; i < 2; i++) {
				CU(cudaStreamCreateWithFlags(&h->aux[i], cudaStreamNonBlocking));
				CU(cudaEventCreateWithFlags(&h->join_ev[i], cudaEventDisableTiming));
			}
			CU(cudaEventCreateWithFlags(&h->fork_ev, cudaEventDisableTiming));
		}
		cudaStream_t main_stream = h->stream;
		TimedScope ts(h);
		const bool overlap = chunks.size() > 1;
		if (overlap) {
			CU(cudaEventRecord(h->fork_ev, main_stream));
			CU(cudaStreamWaitEvent(h->aux[0], h->fork_ev, 0));
			CU(cudaStreamWaitEvent(h->aux[1], h->fork_ev, 0));
		}
		for (size_t c = 0; c < chunks.size() && !rc; c++) {
			const size_t si = chunks[c].first, sj = chunks[c].second;
			const int e0 = (*segs_host)[si].y;
			int cnt = 0;
			for (size_t k = si; k < sj; k++)
				cnt += (*segs_host)[k].z;
			if (overlap)
				h->stream = h->aux[c & 1];
			DecimScratch sc(h, cnt, h->d_scratch + (overlap ? (c & 1) * half : 0));
			rc = run_decimators(h, base, d_offs + e0, cnt, sc);
			if (!rc) {
				SmallParams p;
				memset(&p, 0, sizeof(p));
				p.base = (const uint8_t *)sc.img;
				p.read_off = nullptr; /* images are contiguous: entry e at (e - e0) * image bytes */
				p.regular_stride = h->shape.image_stride * 4;
				p.entry_base = e0;
				p.segs = d_segs + si;
				p.n_segs = (int)(sj - si);
				p.avg = h->d_avg;
				p.samples = h->d_smp64;
				p.samples_per_read = h->shape.samples_per_read;
				p.tw = h->d_tw;
				p.twc = h->d_twc;
				p.win = h->d_win;
				p.dc_ave = sc.ave;
				p.l_len = h->shape.l_len;
				p.n_blocks = h->shape.n_blocks;
				p.blocks_padded = h->shape.blocks_padded;
				p.tw0 = h->tw0;
				rc = launch_small(h, p, true);
			}
		}
		h->stream = main_stream;
		if (overlap) {
			for (int i = 0; i < 2; i++) {
				if (cudaEventRecord(h->join_ev[i], h->aux[i]) != cudaSuccess ||
				    cudaStreamWaitEvent(main_stream, h->join_ev[i], 0) != cudaSuccess) {
					h->last_error = "stream join failed";
					return RTLSDR_GPU_ERR_CUDA;
				}
			}
		}
		return rc;
	}

	/* PATH_LARGE */
	{
		TimedScope ts(h);
		return large_process(h, base, d_offs, d_hops, n_reads);
	}
}

int process_batch(rtlsdr_gpu_scan *h, const uint8_t *base, const std::vector<long long> &offs,
		  const std::vector<int> &hops)
{
	const int n = (int)offs.size();
	if (n == 0)
		return 0;
	std::vector<long long> s_offs;
	std::vector<int> s_hops;
	std::vector<int4> segs;
	int n_segs = build_desc(h, offs, hops, s_offs, s_hops, segs);
	DescLayout lay(n, n_segs);
	DescSlot *slot;
	int rc = desc_acquire(h, lay.bytes, &slot);
	if (rc)
		return rc;
	uint8_t *hp = (uint8_t *)slot->h;
	memcpy(hp + lay.off_reads, s_offs.data(), (size_t)n * 8);
	memcpy(hp + lay.off_segs, segs.data(), (size_t)n_segs * 16);
	memcpy(hp + lay.off_hops, s_hops.data(), (size_t)n * 4);
	h->last_was_epilogue = false;
	CU(cudaMemcpyAsync(slot->d, slot->h, lay.bytes, cudaMemcpyHostToDevice, h->stream));
	rc = launch_batch(h, base, (const uint8_t *)slot->d, n, n_segs, &segs);
	CU(cudaEventRecord(slot->done, h->stream));
	slot->used = true;
	if (rc)
		return rc;
	for (int i = 0; i < n; i++) {
		h->samples[hops[i]] += h->shape.samples_per_read;
		if (h->d_level)
			h->level_bytes[hops[i]] += (uint64_t)h->cfg.buf_len;
	}
	return 0;
}

int flush_ring(rtlsdr_gpu_scan *h)
{
	const int half = h->cur_half;
	const int n = (int)h->ring_hops.size();
	if (n == 0)
		return 0;
	const size_t B = (size_t)h->cfg.buf_len;
	h->last_was_epilogue = false;
	CU(cudaMemcpyAsync(h->d_ring[half], h->h_ring[half], (size_t)n * B, cudaMemcpyHostToDevice, h->stream));
	h->h2d += (uint64_t)n * B;
	std::vector<long long> offs(n);
	for (int i = 0; i < n; i++)
		offs[i] = (long long)i * (long long)B;
	int rc = process_batch(h, h->d_ring[half], offs, h->ring_hops);
	CU(cudaEventRecord(h->ring_done[half], h->stream));
	h->ring_busy[half] = true;
	h->ring_hops.clear();
	h->cur_half ^= 1;
	if (rc)
		return rc;
	if (h->ring_busy[h->cur_half]) {
		CU(cudaEventSynchronize(h->ring_done[h->cur_half]));
		h->ring_busy[h->cur_half] = false;
	}
	return 0;
}

int regular_offsets(const rtlsdr_gpu_scan *h, int hop_first, int hop_count, int passes, long long pass_stride,
		    long long hop_stride, std::vector<long long> &offs, std::vector<int> &hops)
{
	if (hop_first < 0 || hop_count <= 0 || hop_first + hop_count > h->cfg.tune_count)
		return RTLSDR_GPU_ERR_HOP;
	if (passes <= 0)
		return RTLSDR_GPU_ERR_CONFIG;
	offs.resize((size_t)passes * hop_count);
	hops.resize(offs.size());
	size_t i = 0;
	for (int p = 0; p < passes; p++)
		for (int k = 0; k < hop_count; k++, i++) {
			offs[i] = (long long)p * pass_stride + (long long)k * hop_stride;
			hops[i] = hop_first + k;
		}
	return 0;
}

void free_all(rtlsdr_gpu_scan *h)
{
	if (!h)
		return;
	cudaSetDevice(h->cfg.device);
	if (h->stream)
		cudaStreamSynchronize(h->stream);
	if (h->report_stream)
		cudaStreamSynchronize(h->report_stream);
	cudaFree(h->d_avg);
	cudaFree(h->d_avg_other);
	if (h->report_stream)
		cudaStreamDestroy(h->report_stream);
	if (h->ev_scan)
		cudaEventDestroy(h->ev_scan);
	for (int i = 0; i < 2; i++)
		if (h->ev_report[i])
			cudaEventDestroy(h->ev_report[i]);
	cudaFree(h->d_tw);
	cudaFree(h->d_level);
	cudaFree(h->d_done);
	cudaFree(h->d_twb);
	cudaFree(h->d_twc);
	cudaFree(h->d_win);
	cudaFree(h->d_db);
	cudaFree(h->d_iir);
	cudaFree(h->d_samples);
	cudaFree(h->d_scratch);
	cudaFree(h->d_bulk);
	cudaFree(h->d_csv_cols);
	cudaFree(h->d_csv_slots);
	cudaFree(h->d_csv_lens);
	cudaFree(h->d_csv_text);
	cudaFree(h->d_csv_len);
	if (h->h_csv_len)
		cudaFreeHost(h->h_csv_len);
	for (auto &c : h->reg_cache)
		cudaFree(c.d_desc);
	for (int i = 0; i < 2; i++) {
		if (h->aux[i])
			cudaStreamDestroy(h->aux[i]);
		if (h->join_ev[i])
			cudaEventDestroy(h->join_ev[i]);
	}
	if (h->fork_ev)
		cudaEventDestroy(h->fork_ev);
	if (h->hb_head_stream)
		cudaStreamDestroy(h->hb_head_stream);
	if (h->hb_fork)
		cudaEventDestroy(h->hb_fork);
	if (h->hb_join)
		cudaEventDestroy(h->hb_join);
	if (h->copy_stream)
		cudaStreamDestroy(h->copy_stream);
	if (h->bulk_free)
		cudaEventDestroy(h->bulk_free);
	for (auto e : h->chunk_ready)
		cudaEventDestroy(e);
	if (h->h_samples_pinned)
		cudaFreeHost(h->h_samples_pinned);
	for (int i = 0; i < 2; i++) {
		if (h->h_ring[i])
			cudaFreeHost(h->h_ring[i]);
		cudaFree(h->d_ring[i]);
		if (h->ring_done[i])
			cudaEventDestroy(h->ring_done[i]);
	}
	for (auto &s : h->desc) {
		if (s.h)
			cudaFreeHost(s.h);
		cudaFree(s.d);
		if (s.done)
			cudaEventDestroy(s.done);
	}
	for (auto &p : h->timed) {
		cudaEventDestroy(p.first);
		cudaEventDestroy(p.second);
	}
	for (auto e : h->ev_pool)
		cudaEventDestroy(e);
	if (h->ev_a)
		cudaEventDestroy(h->ev_a);
	if (h->ev_b)
		cudaEventDestroy(h->ev_b);
	if (h->own_stream)
		cudaStreamDestroy(h->own_stream);
	delete h;
}

/* dB rows (+ optional raw-bin / sample-count copies) of hops [hop0, hop0+nhops):
 * one kernel, outputs indexed from hop0 */
int run_epilogue(rtlsdr_gpu_scan *h, int hop0, int nhops, double *db, long long *avg_out, int *samples_out,
		 bool zero_after = false)
{
	EpilogueParams p;
	p.done = zero_after ? h->d_done : nullptr;
	p.avg_rw = h->d_avg;
	p.samples_rw = h->d_smp64;
	p.avg = h->d_avg;
	p.samples = h->d_smp64;
	p.db = db;
	p.avg_out = avg_out;
	p.samples_out = samples_out;
	p.bin_e = h->cfg.bin_e;
	p.i1 = h->shape.db_i1;
	p.i2 = h->shape.db_i2;
	p.rate = h->cfg.rate;
	p.hop0 = hop0;
	p.iir = h->d_iir;
	p.iir_alpha = h->cfg.iir_alpha;
	const int span = std::max(h->shape.db_count, avg_out ? h->shape.N : 0);
	dim3 grid((span + 255) / 256, nhops);
	epilogue_kernel<<<grid, 256, 0, h->stream>>>(p);
	h->last_was_epilogue = zero_after; /* nothing else follows it on the stream in the fused-zero case */
	return check_launch(h, "epilogue_kernel");
}

/* bytes of `rows` CSV rows at their widest (csv_text.cuh) */
size_t csv_bound(const rtlsdr_gpu_scan *h, int rows, size_t stamp_len)
{
	return (size_t)rows * (stamp_len + kCsvRowFixed + (size_t)kCsvValueMax * (size_t)h->shape.db_count);
}

/* rows [row_first, row_first + rows) of the column table, from dB rows and int32 counts in device memory, into
 * `text` (csv_bound() bytes) and `len` (-1 = a value outside the formatter's domain), on the handle's stream */
int run_csv(rtlsdr_gpu_scan *h, const char *stamp, size_t stamp_len, int row_first, int rows, const double *db,
	    long long db_stride, const int *samples, char *text, long long *len)
{
	const size_t slot = csv_bound(h, 1, stamp_len), need = slot * (size_t)rows;
	if (need > h->csv_slot_bytes) {
		cudaFree(h->d_csv_slots);
		h->d_csv_slots = nullptr;
		h->csv_slot_bytes = 0;
		CU(cudaMalloc(&h->d_csv_slots, need));
		h->csv_slot_bytes = need;
	}
	CsvRowParams p;
	p.db = db;
	p.db_stride = db_stride;
	p.samples = samples;
	p.cols = h->d_csv_cols;
	p.step = h->csv_step;
	p.row_first = row_first;
	p.db_count = h->shape.db_count;
	p.slots = h->d_csv_slots;
	p.slot_bytes = (long long)slot;
	p.lens = h->d_csv_lens;
	p.stamp_len = (int)stamp_len;
	memcpy(p.stamp, stamp, stamp_len);
	h->last_was_epilogue = false;
	csv_rows_kernel<<<rows, kCsvThreads, 0, h->stream>>>(p);
	if (int rc = check_launch(h, "csv_rows_kernel"))
		return rc;
	CsvPackParams q;
	q.slots = h->d_csv_slots;
	q.slot_bytes = (long long)slot;
	q.lens = h->d_csv_lens;
	q.text = text;
	q.len = len;
	csv_pack_kernel<<<rows, kCsvThreads, 0, h->stream>>>(q);
	return check_launch(h, "csv_pack_kernel");
}

} // namespace

/* large-FFT path needs the handle definition */
#include "scan_large_host.inl"

extern "C" {

const char *rtlsdr_gpu_scan_strerror(int err)
{
	switch (err) {
	case RTLSDR_GPU_OK: return "success";
	case RTLSDR_GPU_ERR_NULL: return "null handle or argument";
	case RTLSDR_GPU_ERR_CONFIG: return "invalid or unsupported configuration";
	case RTLSDR_GPU_ERR_HOP: return "hop index out of range";
	case RTLSDR_GPU_ERR_LENGTH: return "buffer length does not match buf_len";
	case RTLSDR_GPU_ERR_NO_DEVICE: return "no usable sm_100 CUDA device";
	case RTLSDR_GPU_ERR_CUDA: return "CUDA error";
	case RTLSDR_GPU_ERR_NOMEM: return "out of memory";
	case RTLSDR_GPU_ERR_ALIGN: return "device buffer or stride not 16-byte aligned";
	default: return "unknown error";
	}
}

const char *rtlsdr_gpu_scan_last_cuda_error(const rtlsdr_gpu_scan_t *h)
{
	return h ? h->last_error.c_str() : "";
}

void rtlsdr_gpu_scan_sine_table(int bin_e, int16_t *out)
{
	if (out && bin_e >= 0 && bin_e <= 24)
		host_sine_table(bin_e, out);
}

int rtlsdr_gpu_scan_window(const char *name, int n, int32_t *out)
{
	static const struct { const char *name; window_fn fn; } tab[] = {
		{ "rectangle", win_rectangle }, { "hamming", win_hamming }, { "blackman", win_blackman },
		{ "blackman-harris", win_blackman_harris }, { "hann-poisson", win_hann_poisson },
		{ "youssef", win_youssef }, { "kaiser", win_rectangle }, { "bartlett", win_bartlett },
	};
	window_fn fn = win_rectangle;
	int rc = -1;
	if (!out || n <= 0)
		return RTLSDR_GPU_ERR_NULL;
	for (size_t i = 0; name && i < sizeof(tab) / sizeof(tab[0]); i++)
		if (strcmp(name, tab[i].name) == 0) {
			fn = tab[i].fn;
			rc = 0;
		}
	for (int i = 0; i < n; i++)
		out[i] = (int32_t)(256 * fn(i, n));
	return rc;
}

void *rtlsdr_gpu_scan_host_alloc(size_t bytes)
{
	void *p = nullptr;
	if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
		cudaGetLastError();
		return nullptr;
	}
	return p;
}

void rtlsdr_gpu_scan_host_free(void *p)
{
	if (p)
		cudaFreeHost(p);
}

int rtlsdr_gpu_scan_init(const rtlsdr_gpu_scan_cfg_t *cfg_in, rtlsdr_gpu_scan_t **out)
{
	if (!cfg_in || !out)
		return RTLSDR_GPU_ERR_NULL;
	*out = nullptr;
	if (cfg_in->struct_size != sizeof(rtlsdr_gpu_scan_cfg_t) && cfg_in->struct_size != RTLSDR_GPU_SCAN_CFG_V1_SIZE)
		return RTLSDR_GPU_ERR_CONFIG;
	rtlsdr_gpu_scan_cfg_t full;
	memset(&full, 0, sizeof(full));
	memcpy(&full, cfg_in, cfg_in->struct_size); /* fields a shorter (older) struct lacks stay 0 */
	const rtlsdr_gpu_scan_cfg_t *cfg = &full;
	ScanShape shape;
	int rc = scan_shape(*cfg, &shape);
	if (rc)
		return rc;
	const int L = cfg->bin_e, N = shape.N;

	/* host tables: built, and the sine table checked, before any device work */
	std::vector<int2> tw, twc, twb;
	std::vector<uint16_t> win;
	PassTw tw0 = {};
	if (L > 0) {
		std::vector<int16_t> sine((size_t)N * 3 / 4);
		if (!cfg->sinewave)
			host_sine_table(L, sine.data());
		if ((rc = twiddles(cfg->sinewave ? cfg->sinewave : sine.data(), L, tw)))
			return rc;
		tw0 = first_stage_tw(tw, L);
		twc = compact_tw(tw, L, shape.path == PATH_LARGE ? 8 : L);
		if (shape.path == PATH_LARGE)
			twb = round_b_tw(tw, L);
		win = window16(cfg->window_coefs, N);
	}

	int ndev = 0;
	cudaDeviceProp prop;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || cfg->device < 0 || cfg->device >= ndev ||
	    cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess || prop.major != 10 ||
	    cudaSetDevice(cfg->device) != cudaSuccess) {
		cudaGetLastError();
		return RTLSDR_GPU_ERR_NO_DEVICE;
	}

	rtlsdr_gpu_scan *h = new (std::nothrow) rtlsdr_gpu_scan();
	if (!h)
		return RTLSDR_GPU_ERR_NOMEM;
	h->cfg = *cfg;
	if ((rc = read_debug_switches(h))) {
		delete h;
		return rc;
	}
	h->cfg.window_coefs = nullptr;
	h->cfg.sinewave = nullptr;
	h->shape = shape;
	h->tw0 = tw0;
	h->num_sms = prop.multiProcessorCount;
	h->samples.assign(cfg->tune_count, 0);

	rc = RTLSDR_GPU_ERR_CUDA;
	do {
		if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess)
			break;
		h->stream = h->own_stream;
		const size_t avg_bytes = ((size_t)cfg->tune_count * N + (size_t)cfg->tune_count) * sizeof(long long);
		if (cudaMalloc(&h->d_avg, avg_bytes) != cudaSuccess ||
		    cudaMalloc(&h->d_db, (size_t)cfg->tune_count * h->shape.db_count * sizeof(double)) != cudaSuccess ||
		    cudaMalloc(&h->d_samples, (size_t)cfg->tune_count * sizeof(int)) != cudaSuccess ||
		    cudaMallocHost(&h->h_samples_pinned, (size_t)cfg->tune_count * sizeof(int)) != cudaSuccess) {
			rc = RTLSDR_GPU_ERR_NOMEM;
			break;
		}
		h->d_smp64 = h->d_avg + (size_t)cfg->tune_count * N;
		if (cfg->flags & RTLSDR_GPU_FLAG_ASYNC_REPORT) {
			if (!alloc_fill(&h->d_avg_other, avg_bytes, 0, h->stream, &rc) ||
			    cudaStreamCreateWithFlags(&h->report_stream, cudaStreamNonBlocking) != cudaSuccess ||
			    cudaEventCreateWithFlags(&h->ev_scan, cudaEventDisableTiming) != cudaSuccess ||
			    cudaEventCreateWithFlags(&h->ev_report[0], cudaEventDisableTiming) != cudaSuccess ||
			    cudaEventCreateWithFlags(&h->ev_report[1], cudaEventDisableTiming) != cudaSuccess)
				break;
		}
		if (!alloc_fill(&h->d_done, (size_t)cfg->tune_count * sizeof(unsigned), 0, h->stream, &rc) ||
		    cudaMemsetAsync(h->d_avg, 0, avg_bytes, h->stream) != cudaSuccess)
			break;
		/* smoothing state of the printed bins, NaN (all bits set) = no report yet */
		const size_t iir_bytes = (size_t)cfg->tune_count * (size_t)(h->shape.db_count - 1) * sizeof(double);
		if (cfg->iir_alpha > 0.0 && !alloc_fill(&h->d_iir, iir_bytes, 0xFF, h->stream, &rc))
			break;
		if (cfg->flags & RTLSDR_GPU_FLAG_LEVEL_STATS) {
			if (!alloc_fill(&h->d_level, (size_t)cfg->tune_count * 2 * sizeof(unsigned long long), 0, h->stream, &rc))
				break;
			h->level_bytes.assign(cfg->tune_count, 0);
		}
		if (!upload(&h->d_tw, tw, &rc) || !upload(&h->d_win, win, &rc) || !upload(&h->d_twc, twc, &rc) ||
		    !upload(&h->d_twb, twb, &rc))
			break;

		/* staging ring */
		size_t ring = cfg->ring_bytes ? cfg->ring_bytes : kDefaultRing;
		const size_t B = (size_t)cfg->buf_len;
		h->ring_reads = (int)std::max<size_t>(1, ring / B);
		h->ring_bytes = (size_t)h->ring_reads * B;
		bool ok = true;
		for (int i = 0; i < 2 && ok; i++) {
			ok = cudaMallocHost(&h->h_ring[i], h->ring_bytes) == cudaSuccess &&
			     cudaMalloc(&h->d_ring[i], h->ring_bytes) == cudaSuccess &&
			     cudaEventCreateWithFlags(&h->ring_done[i], cudaEventDisableTiming) == cudaSuccess;
		}
		if (!ok) {
			rc = RTLSDR_GPU_ERR_NOMEM;
			break;
		}
		h->ring_hops.reserve(h->ring_reads);
		if (cfg->flags & RTLSDR_GPU_FLAG_SHORT_READS)
			h->hop_shadow.assign((size_t)cfg->tune_count * B, 0);
		if (cudaStreamSynchronize(h->stream) != cudaSuccess)
			break;
		rc = 0;
	} while (0);
	if (rc) {
		cudaGetLastError();
		free_all(h);
		return rc;
	}
	*out = h;
	return 0;
}

void rtlsdr_gpu_scan_close(rtlsdr_gpu_scan_t *h)
{
	free_all(h);
}

void *rtlsdr_gpu_scan_get_stream(rtlsdr_gpu_scan_t *h)
{
	return h ? (void *)h->stream : nullptr;
}

void *rtlsdr_gpu_scan_get_report_stream(rtlsdr_gpu_scan_t *h)
{
	if (!h)
		return nullptr;
	return (void *)((h->report_stream && !h->d_level) ? h->report_stream : h->stream);
}

int rtlsdr_gpu_scan_set_stream(rtlsdr_gpu_scan_t *h, void *cuda_stream)
{
	if (!h)
		return RTLSDR_GPU_ERR_NULL;
	CU(cudaSetDevice(h->cfg.device));
	CU(cudaStreamSynchronize(h->stream));
	h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
	h->last_was_epilogue = false;
	return 0;
}

int rtlsdr_gpu_scan_submit(rtlsdr_gpu_scan_t *h, int hop, const uint8_t *buf, uint32_t len)
{
	if (!h || !buf)
		return RTLSDR_GPU_ERR_NULL;
	if (hop < 0 || hop >= h->cfg.tune_count)
		return RTLSDR_GPU_ERR_HOP;
	const size_t B = (size_t)h->cfg.buf_len;
	if (len > (uint32_t)h->cfg.buf_len || (len < (uint32_t)h->cfg.buf_len && h->hop_shadow.empty()))
		return RTLSDR_GPU_ERR_LENGTH;
	uint8_t *slot = h->h_ring[h->cur_half] + h->ring_hops.size() * B;
	if (!h->hop_shadow.empty()) {
		/* RTLSDR_GPU_FLAG_SHORT_READS: tunes[hop].buf8 of the reference -- a short read overwrites the first
		 * n_read bytes, the rest still holds the hop's previous read, and the WHOLE buffer is processed
		 * (rtl_power.c:657-659) */
		uint8_t *shadow = h->hop_shadow.data() + (size_t)hop * B;
		memcpy(shadow, buf, len);
		memcpy(slot, shadow, B);
	} else {
		memcpy(slot, buf, B);
	}
	h->ring_hops.push_back(hop);
	if ((int)h->ring_hops.size() >= h->ring_reads) {
		CU(cudaSetDevice(h->cfg.device));
		return flush_ring(h);
	}
	return 0;
}

int rtlsdr_gpu_scan_flush(rtlsdr_gpu_scan_t *h)
{
	if (!h)
		return RTLSDR_GPU_ERR_NULL;
	CU(cudaSetDevice(h->cfg.device));
	return flush_ring(h);
}

int rtlsdr_gpu_scan_sync(rtlsdr_gpu_scan_t *h)
{
	if (!h)
		return RTLSDR_GPU_ERR_NULL;
	CU(cudaSetDevice(h->cfg.device));
	int rc = flush_ring(h);
	if (rc)
		return rc;
	CU(cudaStreamSynchronize(h->stream));
	return 0;
}

constexpr size_t kRegCacheEntries = 16;
constexpr int kBatchChunks = 4;

/* regular (strided) batch already on the device; descriptors are cached per (base, shape) */
static int submit_regular(rtlsdr_gpu_scan_t *h, int hop_first, int hop_count, int passes, const void *dev_buf,
			  int64_t pass_stride, int64_t hop_stride)
{
	RegularKey key;
	key.base = dev_buf;
	key.hop_first = hop_first;
	key.hop_count = hop_count;
	key.passes = passes;
	key.pass_stride = pass_stride;
	key.hop_stride = hop_stride;
	key.valid = true;
	int rc;
	rtlsdr_gpu_scan::RegCache *hit = nullptr;
	for (auto &c : h->reg_cache)
		if (c.key == key)
			hit = &c;
	if (!hit) {
		std::vector<long long> offs, s_offs;
		std::vector<int> hops, s_hops;
		if ((rc = regular_offsets(h, hop_first, hop_count, passes, pass_stride, hop_stride, offs, hops)))
			return rc;
		if (h->reg_cache.size() < kRegCacheEntries) {
			h->reg_cache.emplace_back();
			hit = &h->reg_cache.back();
		} else {
			hit = &h->reg_cache[0];
			for (auto &c : h->reg_cache)
				if (c.stamp < hit->stamp)
					hit = &c;
		}
		hit->key.valid = false;
		const int n = (int)offs.size();
		const int n_segs = build_desc(h, offs, hops, s_offs, s_hops, hit->segs);
		DescLayout lay(n, n_segs);
		if (hit->cap < lay.bytes) {
			CU(cudaStreamSynchronize(h->stream)); /* an in-flight kernel may still read the old table */
			cudaFree(hit->d_desc);
			hit->d_desc = nullptr;
			hit->cap = 0;
			CU(cudaMalloc(&hit->d_desc, lay.bytes));
			hit->cap = lay.bytes;
		}
		DescSlot *slot;
		if ((rc = desc_acquire(h, lay.bytes, &slot)))
			return rc;
		uint8_t *hp = (uint8_t *)slot->h;
		memcpy(hp + lay.off_reads, s_offs.data(), (size_t)n * 8);
		memcpy(hp + lay.off_segs, hit->segs.data(), (size_t)n_segs * 16);
		memcpy(hp + lay.off_hops, s_hops.data(), (size_t)n * 4);
		h->last_was_epilogue = false;
		CU(cudaMemcpyAsync(hit->d_desc, slot->h, lay.bytes, cudaMemcpyHostToDevice, h->stream));
		CU(cudaEventRecord(slot->done, h->stream));
		slot->used = true;
		key.n_reads = n;
		key.n_segs = n_segs;
		hit->key = key;
	}
	hit->stamp = ++h->reg_stamp;
	rc = launch_batch(h, (const uint8_t *)dev_buf, (const uint8_t *)hit->d_desc, hit->key.n_reads, hit->key.n_segs,
			  &hit->segs);
	if (rc)
		return rc;
	for (int k = 0; k < hop_count; k++) {
		h->samples[hop_first + k] += h->shape.samples_per_read * passes;
		if (h->d_level)
			h->level_bytes[hop_first + k] += (uint64_t)h->cfg.buf_len * (uint64_t)passes;
	}
	return 0;
}

int rtlsdr_gpu_scan_submit_device(rtlsdr_gpu_scan_t *h, int hop_first, int hop_count, int passes,
				  const void *dev_buf, int64_t pass_stride, int64_t hop_stride)
{
	if (!h || !dev_buf)
		return RTLSDR_GPU_ERR_NULL;
	if (((uintptr_t)dev_buf & 15) || (pass_stride & 15) || (hop_stride & 15))
		return RTLSDR_GPU_ERR_ALIGN;
	if (hop_first < 0 || hop_count <= 0 || hop_first + hop_count > h->cfg.tune_count)
		return RTLSDR_GPU_ERR_HOP;
	if (passes <= 0)
		return RTLSDR_GPU_ERR_CONFIG;
	CU(cudaSetDevice(h->cfg.device));
	int rc = flush_ring(h); /* keep submission order */
	if (rc)
		return rc;
	return submit_regular(h, hop_first, hop_count, passes, dev_buf, pass_stride, hop_stride);
}

/* device landing area of submit_batch / submit_reads (grown on demand) + the copy stream and its events */
static int bulk_prepare(rtlsdr_gpu_scan_t *h, size_t extent)
{
	if (h->bulk_bytes < extent) {
		CU(cudaStreamSynchronize(h->stream));
		if (h->copy_stream)
			CU(cudaStreamSynchronize(h->copy_stream));
		cudaFree(h->d_bulk);
		h->d_bulk = nullptr;
		h->bulk_bytes = 0;
		if (cudaMalloc(&h->d_bulk, extent) != cudaSuccess) {
			cudaGetLastError();
			return RTLSDR_GPU_ERR_NOMEM;
		}
		h->bulk_bytes = extent;
		for (auto &c : h->reg_cache)
			c.key.valid = false;
	}
	if (!h->copy_stream) {
		CU(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
		CU(cudaEventCreateWithFlags(&h->bulk_free, cudaEventDisableTiming));
		h->chunk_ready.resize(kBatchChunks, nullptr);
		for (auto &e : h->chunk_ready)
			CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
	}
	int rc = flush_ring(h);
	if (rc)
		return rc;
	if (h->bulk_used)
		CU(cudaStreamWaitEvent(h->copy_stream, h->bulk_free, 0)); /* previous batch's kernels are done with d_bulk */
	return 0;
}

int rtlsdr_gpu_scan_submit_batch(rtlsdr_gpu_scan_t *h, int hop_first, int hop_count, int passes,
				 const uint8_t *buf, int64_t pass_stride, int64_t hop_stride)
{
	if (!h || !buf)
		return RTLSDR_GPU_ERR_NULL;
	if ((pass_stride & 15) || (hop_stride & 15) || ((uintptr_t)buf & 15))
		return RTLSDR_GPU_ERR_ALIGN;
	if (hop_first < 0 || hop_count <= 0 || hop_first + hop_count > h->cfg.tune_count)
		return RTLSDR_GPU_ERR_HOP;
	if (passes <= 0 || pass_stride < 0 || hop_stride < 0)
		return RTLSDR_GPU_ERR_CONFIG;
	CU(cudaSetDevice(h->cfg.device));
	const size_t B = (size_t)h->cfg.buf_len;
	const size_t pass_extent = (size_t)(hop_count - 1) * (size_t)hop_stride + B;
	const size_t extent = (size_t)(passes - 1) * (size_t)pass_stride + pass_extent;
	int rc = bulk_prepare(h, extent);
	if (rc)
		return rc;
	/* Chunks of whole passes: chunk c+1 crosses PCIe while chunk c is transformed.  Passes must
	 * not interleave in memory for that (pass_stride covers one pass), else one chunk. */
	int chunks = (passes >= 2 * kBatchChunks && (size_t)pass_stride >= pass_extent) ? kBatchChunks : 1;
	for (int c = 0; c < chunks; c++) {
		const int p0 = (int)((long long)passes * c / chunks), p1 = (int)((long long)passes * (c + 1) / chunks);
		const size_t off = (size_t)p0 * (size_t)pass_stride;
		const size_t bytes = (size_t)(p1 - p0 - 1) * (size_t)pass_stride + pass_extent;
		CU(cudaMemcpyAsync(h->d_bulk + off, buf + off, bytes, cudaMemcpyHostToDevice, h->copy_stream));
		CU(cudaEventRecord(h->chunk_ready[c], h->copy_stream));
		h->h2d += bytes;
	}
	for (int c = 0; c < chunks; c++) {
		const int p0 = (int)((long long)passes * c / chunks), p1 = (int)((long long)passes * (c + 1) / chunks);
		h->last_was_epilogue = false;
		CU(cudaStreamWaitEvent(h->stream, h->chunk_ready[c], 0));
		rc = submit_regular(h, hop_first, hop_count, p1 - p0, h->d_bulk + (size_t)p0 * (size_t)pass_stride,
				    pass_stride, hop_stride);
		if (rc)
			return rc;
	}
	CU(cudaEventRecord(h->bulk_free, h->stream));
	h->bulk_used = true;
	return 0;
}

int rtlsdr_gpu_scan_submit_reads(rtlsdr_gpu_scan_t *h, int n_reads, const int32_t *hops, const uint8_t *buf, int64_t stride)
{
	if (!h || !buf || !hops)
		return RTLSDR_GPU_ERR_NULL;
	if ((stride & 15) || ((uintptr_t)buf & 15))
		return RTLSDR_GPU_ERR_ALIGN;
	if (n_reads <= 0 || stride < (int64_t)h->cfg.buf_len)
		return RTLSDR_GPU_ERR_CONFIG;
	for (int i = 0; i < n_reads; i++)
		if (hops[i] < 0 || hops[i] >= h->cfg.tune_count)
			return RTLSDR_GPU_ERR_HOP;
	CU(cudaSetDevice(h->cfg.device));
	const size_t B = (size_t)h->cfg.buf_len;
	int rc = bulk_prepare(h, (size_t)(n_reads - 1) * (size_t)stride + B);
	if (rc)
		return rc;
	/* chunks of consecutive reads: chunk c+1 crosses PCIe while chunk c is transformed */
	const int chunks = n_reads >= 64 * kBatchChunks ? kBatchChunks : 1;
	for (int c = 0; c < chunks; c++) {
		const int r0 = (int)((long long)n_reads * c / chunks), r1 = (int)((long long)n_reads * (c + 1) / chunks);
		const size_t off = (size_t)r0 * (size_t)stride, bytes = (size_t)(r1 - r0 - 1) * (size_t)stride + B;
		CU(cudaMemcpyAsync(h->d_bulk + off, buf + off, bytes, cudaMemcpyHostToDevice, h->copy_stream));
		CU(cudaEventRecord(h->chunk_ready[c], h->copy_stream));
		h->h2d += bytes;
	}
	std::vector<long long> offs;
	std::vector<int> hp;
	for (int c = 0; c < chunks; c++) {
		const int r0 = (int)((long long)n_reads * c / chunks), r1 = (int)((long long)n_reads * (c + 1) / chunks);
		offs.resize((size_t)(r1 - r0));
		hp.assign(hops + r0, hops + r1);
		for (int i = r0; i < r1; i++)
			offs[(size_t)(i - r0)] = (long long)i * (long long)stride;
		h->last_was_epilogue = false;
		CU(cudaStreamWaitEvent(h->stream, h->chunk_ready[c], 0));
		if ((rc = process_batch(h, h->d_bulk, offs, hp)))
			return rc;
	}
	CU(cudaEventRecord(h->bulk_free, h->stream));
	h->bulk_used = true;
	return 0;
}

/* CUDA loads kernels lazily, and the first launch of a not-yet-loaded kernel can block until the kernels already
 * running on the device have finished -- among them, possibly, the very flag_wait_kernel that this launch is
 * meant to release.  Both kernels are therefore loaded (cudaFuncGetAttributes) before either is launched. */
static int flag_kernels_loaded()
{
	static bool loaded[64] = { false }; /* per device: modules load per context */
	int dev = 0;
	if (cudaGetDevice(&dev) != cudaSuccess)
		return RTLSDR_GPU_ERR_CUDA;
	if (dev >= 0 && dev < 64 && loaded[dev])
		return 0;
	cudaFuncAttributes attr;
	if (cudaFuncGetAttributes(&attr, flag_signal_kernel) != cudaSuccess ||
	    cudaFuncGetAttributes(&attr, flag_signal_many_kernel) != cudaSuccess ||
	    cudaFuncGetAttributes(&attr, flag_wait_kernel) != cudaSuccess) {
		cudaGetLastError();
		return RTLSDR_GPU_ERR_CUDA;
	}
	if (dev >= 0 && dev < 64)
		loaded[dev] = true;
	return 0;
}

int rtlsdr_gpu_scan_flag_signal(void *cuda_stream, void *dev_flag, uint32_t value)
{
	if (!dev_flag)
		return RTLSDR_GPU_ERR_NULL;
	if ((uintptr_t)dev_flag & 3)
		return RTLSDR_GPU_ERR_ALIGN;
	if (int rc = flag_kernels_loaded())
		return rc;
	flag_signal_kernel<<<1, 1, 0, (cudaStream_t)cuda_stream>>>((unsigned *)dev_flag, value);
	return cudaGetLastError() == cudaSuccess ? 0 : RTLSDR_GPU_ERR_CUDA;
}

int rtlsdr_gpu_scan_flag_signal_many(void *cuda_stream, void *const *dev_flags, int count, uint32_t value)
{
	if (!dev_flags)
		return RTLSDR_GPU_ERR_NULL;
	if (count <= 0 || count > kFlagSignalMax)
		return RTLSDR_GPU_ERR_CONFIG;
	FlagList list;
	for (int i = 0; i < count; i++) {
		if (!dev_flags[i])
			return RTLSDR_GPU_ERR_NULL;
		if ((uintptr_t)dev_flags[i] & 3)
			return RTLSDR_GPU_ERR_ALIGN;
		list.flag[i] = (unsigned *)dev_flags[i];
	}
	if (int rc = flag_kernels_loaded())
		return rc;
	flag_signal_many_kernel<<<1, 32, 0, (cudaStream_t)cuda_stream>>>(list, count, value);
	return cudaGetLastError() == cudaSuccess ? 0 : RTLSDR_GPU_ERR_CUDA;
}

int rtlsdr_gpu_scan_flag_wait(void *cuda_stream, const void *dev_flags, int count, uint32_t value, uint32_t timeout_ms,
			      void *dev_timed_out)
{
	if (!dev_flags)
		return RTLSDR_GPU_ERR_NULL;
	if (((uintptr_t)dev_flags & 3) || ((uintptr_t)dev_timed_out & 3))
		return RTLSDR_GPU_ERR_ALIGN;
	if (count <= 0 || count > 1024)
		return RTLSDR_GPU_ERR_CONFIG;
	if (int rc = flag_kernels_loaded())
		return rc;
	const unsigned long long ns = (unsigned long long)(timeout_ms ? timeout_ms : 10000u) * 1000000ull;
	flag_wait_kernel<<<1, (count + 31) & ~31, 0, (cudaStream_t)cuda_stream>>>((const unsigned *)dev_flags, count, value, ns,
										    (unsigned *)dev_timed_out);
	return cudaGetLastError() == cudaSuccess ? 0 : RTLSDR_GPU_ERR_CUDA;
}

int rtlsdr_gpu_scan_db_count(const rtlsdr_gpu_scan_t *h)
{
	return h ? h->shape.db_count : RTLSDR_GPU_ERR_NULL;
}

static int collect_range(rtlsdr_gpu_scan_t *h, int hop0, int nhops, int64_t *avg, int *samples, double *db)
{
	CU(cudaSetDevice(h->cfg.device));
	int rc = flush_ring(h);
	if (rc)
		return rc;
	const size_t N = (size_t)h->shape.N;
	if (db) {
		if ((rc = run_epilogue(h, hop0, nhops, h->d_db, nullptr, nullptr)))
			return rc;
		CU(cudaMemcpyAsync(db, h->d_db, (size_t)nhops * h->shape.db_count * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
		h->d2h += (uint64_t)nhops * h->shape.db_count * sizeof(double);
	}
	if (avg) {
		CU(cudaMemcpyAsync(avg, h->d_avg + (size_t)hop0 * N, (size_t)nhops * N * sizeof(long long),
				   cudaMemcpyDeviceToHost, h->stream));
		h->d2h += (uint64_t)nhops * N * sizeof(long long);
	}
	std::vector<long long> dev_smp;
	if (h->samples_on_device && samples) { /* after merge_device(): the counts live in d_smp64 only */
		dev_smp.resize(nhops);
		CU(cudaMemcpyAsync(dev_smp.data(), h->d_smp64 + hop0, (size_t)nhops * sizeof(long long), cudaMemcpyDeviceToHost,
				   h->stream));
	}
	/* read-and-zero, like csv_dbm (rtl_power.c:761-764) */
	h->last_was_epilogue = false;
	if (nhops == h->cfg.tune_count) {
		CU(cudaMemsetAsync(h->d_avg, 0, ((size_t)nhops * N + (size_t)nhops) * sizeof(long long), h->stream));
	} else {
		CU(cudaMemsetAsync(h->d_avg + (size_t)hop0 * N, 0, (size_t)nhops * N * sizeof(long long), h->stream));
		CU(cudaMemsetAsync(h->d_smp64 + hop0, 0, (size_t)nhops * sizeof(long long), h->stream));
	}
	if (h->d_level)
		CU(cudaMemsetAsync(h->d_level + 2 * (size_t)hop0, 0, (size_t)nhops * 2 * sizeof(unsigned long long), h->stream));
	CU(cudaStreamSynchronize(h->stream));
	for (int i = 0; i < nhops; i++) {
		if (samples)
			samples[i] = dev_smp.empty() ? h->samples[hop0 + i] : (int)dev_smp[i];
		h->samples[hop0 + i] = 0;
		if (h->d_level)
			h->level_bytes[hop0 + i] = 0;
	}
	if (nhops == h->cfg.tune_count)
		h->samples_on_device = false; /* everything is zero again: the host mirror is exact from here on */
	return 0;
}

int rtlsdr_gpu_scan_collect(rtlsdr_gpu_scan_t *h, int hop, int64_t *avg, int *samples, double *db)
{
	if (!h)
		return RTLSDR_GPU_ERR_NULL;
	if (hop < 0 || hop >= h->cfg.tune_count)
		return RTLSDR_GPU_ERR_HOP;
	return collect_range(h, hop, 1, avg, samples, db);
}

int rtlsdr_gpu_scan_collect_all(rtlsdr_gpu_scan_t *h, int64_t *avg, int *samples, double *db)
{
	if (!h)
		return RTLSDR_GPU_ERR_NULL;
	return collect_range(h, 0, h->cfg.tune_count, avg, samples, db);
}

int rtlsdr_gpu_scan_collect_device(rtlsdr_gpu_scan_t *h, void *dev_avg, void *dev_samples, void *dev_db)
{
	if (!h)
		return RTLSDR_GPU_ERR_NULL;
	CU(cudaSetDevice(h->cfg.device));
	int rc = flush_ring(h);
	if (rc)
		return rc;
	const size_t N = (size_t)h->shape.N, tc = (size_t)h->cfg.tune_count;
	/* one kernel writes dB rows, raw bins and sample counts straight into the
	 * caller's buffers (e.g. the NCCL send buffer), one memset clears the state */
	/* up to 8192 bins the last epilogue block of a hop also zeroes it (no memset launch) */
	const bool fused_zero = N <= 8192;
	if (h->report_stream && !h->d_level) {
		/* asynchronous report: the epilogue of THIS accumulator set runs on report_stream behind everything
		 * submitted so far, the handle's stream moves on to the other set at once */
		cudaStream_t main_stream = h->stream;
		CU(cudaEventRecord(h->ev_scan, main_stream));
		CU(cudaStreamWaitEvent(h->report_stream, h->ev_scan, 0));
		h->stream = h->report_stream;
		rc = run_epilogue(h, 0, (int)tc, (double *)dev_db, (long long *)dev_avg, (int *)dev_samples, fused_zero);
		if (!rc && !fused_zero) {
			if (cudaMemsetAsync(h->d_avg, 0, (tc * N + tc) * sizeof(long long), h->report_stream) != cudaSuccess)
				rc = RTLSDR_GPU_ERR_CUDA;
		}
		h->stream = main_stream;
		h->last_was_epilogue = false;
		if (rc)
			return rc;
		CU(cudaEventRecord(h->ev_report[h->cur_acc], h->report_stream));
		h->report_pending[h->cur_acc] = true;
		std::swap(h->d_avg, h->d_avg_other);
		h->d_smp64 = h->d_avg + tc * N;
		h->cur_acc ^= 1;
		if (h->report_pending[h->cur_acc]) /* the set the next submits use: its last report (two collects ago) is done */
			CU(cudaStreamWaitEvent(main_stream, h->ev_report[h->cur_acc], 0));
		std::fill(h->samples.begin(), h->samples.end(), 0);
		h->samples_on_device = false;
		return 0;
	}
	if ((rc = run_epilogue(h, 0, (int)tc, (double *)dev_db, (long long *)dev_avg, (int *)dev_samples, fused_zero)))
		return rc;
	if (!fused_zero) {
		h->last_was_epilogue = false;
		CU(cudaMemsetAsync(h->d_avg, 0, (tc * N + tc) * sizeof(long long), h->stream));
	}
	if (h->d_level) {
		h->last_was_epilogue = false;
		CU(cudaMemsetAsync(h->d_level, 0, tc * 2 * sizeof(unsigned long long), h->stream));
		std::fill(h->level_bytes.begin(), h->level_bytes.end(), 0);
	}
	std::fill(h->samples.begin(), h->samples.end(), 0);
	h->samples_on_device = false;
	return 0;
}

int rtlsdr_gpu_scan_set_csv_columns(rtlsdr_gpu_scan_t *h, int rows, const int32_t *low, const int32_t *high, double step)
{
	if (!h || !low || !high)
		return RTLSDR_GPU_ERR_NULL;
	if (rows < 1 || !(step >= 0.0 && step < kCsvStepLimit))
		return RTLSDR_GPU_ERR_CONFIG;
	CU(cudaSetDevice(h->cfg.device));
	std::vector<int2> cols((size_t)rows);
	for (int i = 0; i < rows; i++)
		cols[i] = make_int2(low[i], high[i]);
	if (rows > h->csv_rows) {
		cudaFree(h->d_csv_cols); /* implicit device synchronisation: no kernel still reads the old table */
		cudaFree(h->d_csv_lens);
		h->d_csv_cols = nullptr;
		h->d_csv_lens = nullptr;
		h->csv_rows = 0;
		CU(cudaMalloc(&h->d_csv_cols, (size_t)rows * sizeof(int2)));
		CU(cudaMalloc(&h->d_csv_lens, (size_t)rows * sizeof(int)));
	} else {
		CU(cudaStreamSynchronize(h->stream));
	}
	h->last_was_epilogue = false;
	CU(cudaMemcpyAsync(h->d_csv_cols, cols.data(), (size_t)rows * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
	CU(cudaStreamSynchronize(h->stream));
	h->h2d += (uint64_t)rows * sizeof(int2);
	h->csv_rows = rows;
	h->csv_step = step;
	return 0;
}

int64_t rtlsdr_gpu_scan_csv_capacity(const rtlsdr_gpu_scan_t *h, int rows, size_t stamp_len)
{
	if (!h)
		return RTLSDR_GPU_ERR_NULL;
	if (rows < 0 || stamp_len >= (size_t)kCsvStampMax)
		return RTLSDR_GPU_ERR_CONFIG;
	return (int64_t)csv_bound(h, rows, stamp_len);
}

int rtlsdr_gpu_scan_collect_csv(rtlsdr_gpu_scan_t *h, const char *stamp, char *text, size_t cap, size_t *len)
{
	if (!h || !stamp || !text || !len)
		return RTLSDR_GPU_ERR_NULL;
	const size_t stamp_len = strlen(stamp);
	const int tc = h->cfg.tune_count;
	if (stamp_len >= (size_t)kCsvStampMax || h->csv_rows < tc)
		return RTLSDR_GPU_ERR_CONFIG;
	const size_t bound = csv_bound(h, tc, stamp_len);
	if (cap < bound)
		return RTLSDR_GPU_ERR_LENGTH;
	CU(cudaSetDevice(h->cfg.device));
	int rc = flush_ring(h);
	if (rc)
		return rc;
	if (!h->d_csv_len) {
		CU(cudaMalloc(&h->d_csv_len, sizeof(long long)));
		CU(cudaMallocHost(&h->h_csv_len, sizeof(long long)));
	}
	if (bound > h->csv_text_bytes) {
		cudaFree(h->d_csv_text);
		h->d_csv_text = nullptr;
		h->csv_text_bytes = 0;
		CU(cudaMalloc(&h->d_csv_text, bound));
		h->csv_text_bytes = bound;
	}
	/* the epilogue's dB rows and counts stay on the device: only the text crosses PCIe */
	if ((rc = run_epilogue(h, 0, tc, h->d_db, nullptr, h->d_samples)))
		return rc;
	if ((rc = run_csv(h, stamp, stamp_len, 0, tc, h->d_db, h->shape.db_count, h->d_samples, h->d_csv_text, h->d_csv_len)))
		return rc;
	CU(cudaMemcpyAsync(h->h_csv_len, h->d_csv_len, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
	CU(cudaStreamSynchronize(h->stream));
	const long long n = *h->h_csv_len;
	if (n < 0 || (size_t)n > bound)
		return RTLSDR_GPU_ERR_CONFIG; /* cannot happen for the epilogue's values; the accumulators are kept */
	CU(cudaMemcpyAsync(text, h->d_csv_text, (size_t)n, cudaMemcpyDeviceToHost, h->stream));
	h->d2h += (uint64_t)n + sizeof(long long);
	/* read-and-zero, like csv_dbm (rtl_power.c:761-764) */
	CU(cudaMemsetAsync(h->d_avg, 0, ((size_t)tc * h->shape.N + (size_t)tc) * sizeof(long long), h->stream));
	if (h->d_level)
		CU(cudaMemsetAsync(h->d_level, 0, (size_t)tc * 2 * sizeof(unsigned long long), h->stream));
	CU(cudaStreamSynchronize(h->stream));
	std::fill(h->samples.begin(), h->samples.end(), 0);
	if (h->d_level)
		std::fill(h->level_bytes.begin(), h->level_bytes.end(), 0);
	h->samples_on_device = false;
	*len = (size_t)n;
	return 0;
}

int rtlsdr_gpu_scan_format_csv_device(rtlsdr_gpu_scan_t *h, const char *stamp, int row_first, int rows,
				      const void *dev_db, int64_t db_stride, const void *dev_samples, void *dev_text,
				      size_t cap, void *dev_len)
{
	if (!h || !stamp || !dev_db || !dev_samples || !dev_text || !dev_len)
		return RTLSDR_GPU_ERR_NULL;
	if (((uintptr_t)dev_db & 7) || ((uintptr_t)dev_samples & 3) || ((uintptr_t)dev_len & 7))
		return RTLSDR_GPU_ERR_ALIGN;
	const size_t stamp_len = strlen(stamp);
	if (stamp_len >= (size_t)kCsvStampMax || !h->d_csv_cols || db_stride < h->shape.db_count)
		return RTLSDR_GPU_ERR_CONFIG;
	if (rows < 1 || row_first < 0 || row_first > h->csv_rows - rows)
		return RTLSDR_GPU_ERR_HOP;
	if (cap < csv_bound(h, rows, stamp_len))
		return RTLSDR_GPU_ERR_LENGTH;
	CU(cudaSetDevice(h->cfg.device));
	return run_csv(h, stamp, stamp_len, row_first, rows, (const double *)dev_db, (long long)db_stride,
		       (const int *)dev_samples, (char *)dev_text, (long long *)dev_len);
}

int rtlsdr_gpu_scan_merge_device(rtlsdr_gpu_scan_t *h, const void *dev_avg, const void *dev_samples, int sets,
				 int64_t set_stride)
{
	if (!h || !dev_avg || !dev_samples)
		return RTLSDR_GPU_ERR_NULL;
	if (sets <= 0 || (sets > 1 && set_stride <= 0))
		return RTLSDR_GPU_ERR_CONFIG;
	if (((uintptr_t)dev_avg & 7) || ((uintptr_t)dev_samples & 3) || (set_stride & 7))
		return RTLSDR_GPU_ERR_ALIGN;
	CU(cudaSetDevice(h->cfg.device));
	int rc = flush_ring(h);
	if (rc)
		return rc;
	MergeParams p;
	p.avg = h->d_avg;
	p.samples = h->d_smp64;
	p.ext_avg = (const uint8_t *)dev_avg;
	p.ext_smp = (const uint8_t *)dev_samples;
	p.stride = set_stride;
	p.bins = (long long)h->cfg.tune_count * h->shape.N;
	p.hops = h->cfg.tune_count;
	p.sets = sets;
	p.peak = h->cfg.peak_hold ? 1 : 0;
	const int grid = (int)std::min<long long>((p.bins + 255) / 256, (long long)h->num_sms * 8);
	h->last_was_epilogue = false;
	merge_sets_kernel<<<std::max(grid, 1), 256, 0, h->stream>>>(p);
	h->samples_on_device = true; /* the host mirror of tunes[i].samples no longer knows the totals */
	return check_launch(h, "merge_sets_kernel");
}

int rtlsdr_gpu_scan_level_stats(rtlsdr_gpu_scan_t *h, int hop, uint64_t *overload, uint64_t *high_level, uint64_t *bytes)
{
	if (!h)
		return RTLSDR_GPU_ERR_NULL;
	if (hop < 0 || hop >= h->cfg.tune_count)
		return RTLSDR_GPU_ERR_HOP;
	if (!h->d_level)
		return RTLSDR_GPU_ERR_CONFIG;
	CU(cudaSetDevice(h->cfg.device));
	int rc = flush_ring(h);
	if (rc)
		return rc;
	unsigned long long v[2] = { 0, 0 };
	h->last_was_epilogue = false;
	CU(cudaMemcpyAsync(v, h->d_level + 2 * (size_t)hop, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
	CU(cudaStreamSynchronize(h->stream));
	if (overload)
		*overload = v[0];
	if (high_level)
		*high_level = v[1];
	if (bytes)
		*bytes = h->level_bytes[hop];
	return 0;
}

int rtlsdr_gpu_scan_stats(const rtlsdr_gpu_scan_t *h, uint64_t *kernel_launches, uint64_t *h2d_bytes, uint64_t *d2h_bytes)
{
	if (!h)
		return RTLSDR_GPU_ERR_NULL;
	if (kernel_launches)
		*kernel_launches = h->launches;
	if (h2d_bytes)
		*h2d_bytes = h->h2d;
	if (d2h_bytes)
		*d2h_bytes = h->d2h;
	return 0;
}

int rtlsdr_gpu_scan_set_timing(rtlsdr_gpu_scan_t *h, int every)
{
	if (!h)
		return RTLSDR_GPU_ERR_NULL;
	h->timing = every > 0;
	h->timing_every = every > 0 ? every : 1;
	h->timing_count = 0;
	return 0;
}

int rtlsdr_gpu_scan_kernel_time(rtlsdr_gpu_scan_t *h, double *ms, uint64_t *launches)
{
	if (!h)
		return RTLSDR_GPU_ERR_NULL;
	CU(cudaSetDevice(h->cfg.device));
	double total = 0;
	uint64_t n = 0;
	if (h->timing) {
		CU(cudaStreamSynchronize(h->stream));
		for (auto &p : h->timed) {
			float t = 0;
			if (cudaEventElapsedTime(&t, p.first, p.second) == cudaSuccess) {
				total += t;
				n++;
			}
			h->ev_pool.push_back(p.first);
			h->ev_pool.push_back(p.second);
		}
		h->timed.clear();
	}
	h->timing = true; /* first call arms the timers */
	if (ms)
		*ms = total;
	if (launches)
		*launches = n;
	return 0;
}

} /* extern "C" */
