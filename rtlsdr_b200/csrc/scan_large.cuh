/*
 * scan_large.cuh -- N >= 8192 bins (bin_e 13..21): one FFT block per read, too
 * big for one CTA's shared memory (4N bytes = 32 KiB .. 8 MiB).
 *
 * fix_fft (reference src/rtl_power.c:271-327) is a radix-2 DIT on bit-reversed
 * data: stage s pairs positions that differ in bit s.  The stages are run in
 * up to three rounds, each a kernel over 4096-sample tiles that reuses the
 * register-blocked engine of scan_kernels.cuh; between rounds the packed int16
 * data lives in a global scratch (L2 resident: 512 KiB per read at N = 2^17):
 *
 *   round A  stages 0..7     reads the u8 buffer (or a decimated c16 image),
 *                            removes DC, applies the window, and performs the
 *                            bit-reversal as a tile transpose: a tile is 16
 *                            consecutive input samples x 256 strided rows, so
 *                            both the gather and the scatter move >= 32-byte runs
 *   round B  stages 8..15    in place on the scratch, tile = consecutive
 *                            positions x 2^LB strided rows
 *   round C  stages 16..L-1  (N > 65536) register-only, 2^(L-16) strided points
 *                            per thread, then |X|^2 accumulation in natural bin
 *                            order (coalesced 64-bit atomics)
 * The last round accumulates |X|^2 / peak hold (rtl_power.c:708-716).
 * Rounding, halving, twiddles and int16 wrap are those of butterfly().
 */
#pragma once
#include "scan_kernels.cuh"

namespace rscan {

struct LargeParams {
	const uint8_t *base;        /* u8 reads or decimated c16 images */
	const long long *read_off;  /* byte offset per entry, NULL = regular */
	long long regular_stride;
	int entry_base;             /* first entry of this chunk */
	const int *hop_of;          /* hop per entry (absolute entry index) */
	c16 *scratch;               /* [chunk][N] */
	const long long *dc_sums;   /* [chunk][2] */
	const int2 *dc_consts;      /* u8 reads: [chunk] (127 + average of I, of Q), written by dc_sums_u8_kernel */
	const int2 *twc_a;          /* round A: host-built compact table, stage s (4..7), group m at (1<<s)-16+m */
	long long *avg;
	long long *samples;         /* [tune_count] */
	int samples_per_read;
	const int2 *tw;             /* [N/2] */
	const int2 *twb;            /* round-B re-ordered copy, see TwLargeB */
	const uint16_t *win;        /* [N] */
	int L;
	int n_entries;              /* entries in this chunk */
	int c_reads;                /* reads per CTA of round C (round_c_reads) */
	int tiles_log2;             /* pipelined rounds: log2 of the 4096-sample tiles per read (L - 12) */
	PassTw tw0;
};

SCAN_DEV long long large_entry_offset(const LargeParams &prm, int e)
{
	return prm.read_off ? prm.read_off[e] : (long long)(e - prm.entry_base) * prm.regular_stride;
}

/* per-read byte sums of I and Q for the u8 input (remove_dc, rtl_power.c:586-588) */
struct DcSumU8Params {
	const uint8_t *base;
	const long long *read_off;
	int entry_base;
	int buf_len;
	long long *sums; /* [chunk][2], zeroed by the host */
	unsigned *tickets; /* [chunk], zeroed by the host */
	int2 *consts;    /* [chunk]: the constants round A subtracts from the raw bytes (127 + int16 average) */
};

__global__ void __launch_bounds__(256)
dc_sums_u8_kernel(const SCAN_GRID_CONSTANT DcSumU8Params prm)
{
	const int rel = blockIdx.y;
	pdl_launch_dependents(); /* round A's CTAs may take free slots and load their twiddle table meanwhile */
	const uint8_t *src = prm.base + prm.read_off[prm.entry_base + rel];
	unsigned sI = 0, sQ = 0; /* <= 2^21 bytes of 255 per component: fits */
	const int stride = gridDim.x * blockDim.x * 16;
	for (int i = (blockIdx.x * blockDim.x + threadIdx.x) * 16; i < prm.buf_len; i += 8 * stride) {
		uint4 q[8]; /* 128 bytes in flight per thread: one resident wave of CTAs streams at HBM speed */
#pragma unroll
		for (int j = 0; j < 8; ++j)
			q[j] = (i + j * stride < prm.buf_len) ? __ldg((const uint4 *)(src + i + j * stride)) : uint4{ 0, 0, 0, 0 };
#pragma unroll
		for (int j = 0; j < 8; ++j) {
			sI = __dp4a(q[j].x, 0x00010001u, sI);
			sQ = __dp4a(q[j].x, 0x01000100u, sQ);
			sI = __dp4a(q[j].y, 0x00010001u, sI);
			sQ = __dp4a(q[j].y, 0x01000100u, sQ);
			sI = __dp4a(q[j].z, 0x00010001u, sI);
			sQ = __dp4a(q[j].z, 0x01000100u, sQ);
			sI = __dp4a(q[j].w, 0x00010001u, sI);
			sQ = __dp4a(q[j].w, 0x01000100u, sQ);
		}
	}
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) {
		sI += __shfl_xor_sync(0xffffffffu, sI, o);
		sQ += __shfl_xor_sync(0xffffffffu, sQ, o);
	}
	__shared__ unsigned part[2][8];
	if ((threadIdx.x & 31) == 0) {
		part[0][threadIdx.x >> 5] = sI;
		part[1][threadIdx.x >> 5] = sQ;
	}
	__syncthreads();
	if (threadIdx.x != 0)
		return;
	long long tI = 0, tQ = 0;
	for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
		tI += part[0][w];
		tQ += part[1][w];
	}
	/* The sums become remove_dc's averages here (rtl_power.c:581-596: divisors = the interleaved length and
	 * length - 1, truncating), so that round A's CTAs -- one per tile -- load two words instead of each waiting
	 * for a 64-bit division in front of their first barrier.  One CTA per read (many reads): no atomics at all;
	 * several CTAs per read: the last one to arrive (ticket) converts the total. */
	if (gridDim.x > 1) {
		atomicAdd((unsigned long long *)(prm.sums + 2 * rel), (unsigned long long)tI);
		atomicAdd((unsigned long long *)(prm.sums + 2 * rel + 1), (unsigned long long)tQ);
		__threadfence();
		if (atomicAdd(prm.tickets + rel, 1u) != gridDim.x - 1)
			return;
		tI = (long long)atomicAdd((unsigned long long *)(prm.sums + 2 * rel), 0ull);
		tQ = (long long)atomicAdd((unsigned long long *)(prm.sums + 2 * rel + 1), 0ull);
	}
	const long long half = prm.buf_len / 2;
	prm.consts[rel] = int2{ 127 + dc_average(tI - 127ll * half, prm.buf_len),
				127 + dc_average(tQ - 127ll * half, prm.buf_len - 1) };
}

/* ---- round A ----------------------------------------------------------- */

struct TwLargeA {
	static constexpr bool kTrivial = true;
	const int2 *twc;     /* compact: stage s (4..7), group m at twc[(1<<s)-16+m] */
	const PassTw *tw0;
	template <int K>
	SCAN_DEV int2 get(int s, int pa) const
	{
		const int m = pa & ((1 << s) - 1);
		if constexpr (K == 0)
			return tw0->w[(1 << s) - 1 + m];
		else
			return twc[(1 << s) - 16 + m];
	}
};

constexpr int kLargeSmemA = kXchWords * 4 + 240 * 8 + 16;

template <bool IN16>
__global__ void __launch_bounds__(kThreads, 2)
large_round_a_kernel(const SCAN_GRID_CONSTANT LargeParams prm)
{
	SCAN_DYN_SMEM(smem);
	c16 *stage = (c16 *)smem;
	int2 *twc = (int2 *)(smem + kXchWords * 4);
	int *dck = (int *)(smem + kXchWords * 4 + 240 * 8);
	const int t = threadIdx.x, L = prm.L;
	const int tile = blockIdx.x, rel = blockIdx.y, e = prm.entry_base + rel;
	const long long N = 1ll << L;
	const uint8_t *src = prm.base + large_entry_offset(prm, e);

	if (t < 240)
		twc[t] = __ldg(prm.twc_a + t);
	/* The rounds of one chunk are launched programmatically dependent on each other: a kernel reads what its
	 * predecessor wrote only behind pdl_wait().  Round A has many waves, so only its LAST wave lets round B's
	 * CTAs in early (they would otherwise sit on shared memory that round A's own CTAs need). */
	if ((long long)(gridDim.y - 1 - blockIdx.y) * gridDim.x + (gridDim.x - 1 - blockIdx.x) < 4 * 148)
		pdl_launch_dependents();
	pdl_wait();
	if (t == 0 && tile == 0)
		atomicAdd((unsigned long long *)(prm.samples + prm.hop_of[e]), (unsigned long long)prm.samples_per_read);
	if constexpr (!IN16) {
		if (t == 0)
			*(int2 *)dck = prm.dc_consts[rel];
	} else if (t < 2) {
		dck[t] = dc_average(prm.dc_sums[2 * rel + t], (int)(2 * N) - t);
	}

	__syncthreads();
	const int kI = dck[0], kQ = dck[1];

	/* gather: thread t owns row i = t = 16 consecutive input samples and their 16 window
	 * coefficients (two 16-byte loads each); convert, remove DC, window, and park the c16
	 * results column-major so that the engine finds column c, row i at stage[c*256 + i] */
	{
		const long long n0 = ((long long)t << (L - 8)) + 16 * tile;
		const uint4 wa = __ldg((const uint4 *)(prm.win + n0));
		const uint4 wb = __ldg((const uint4 *)(prm.win + n0 + 8));
		const unsigned ww[8] = { wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w };
		if constexpr (!IN16) {
			const uint4 a = __ldg((const uint4 *)(src + 2 * n0));
			const uint4 b = __ldg((const uint4 *)(src + 2 * n0 + 16));
			const unsigned w[8] = { a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w };
#pragma unroll
			for (int c = 0; c < 16; ++c) {
				const unsigned raw = (w[c >> 1] >> (16 * (c & 1))) & 0xFFFFu;
				const int wv = (int)((ww[c >> 1] >> (16 * (c & 1))) & 0xFFFFu);
				stage[xch_idx(c * 256 + t)] = c16_pack(((int)(raw & 0xFFu) - kI) * wv, ((int)(raw >> 8) - kQ) * wv);
			}
		} else {
#pragma unroll
			for (int k = 0; k < 4; ++k) {
				const uint4 a = __ldg((const uint4 *)(src + 4 * n0 + 16 * k));
				const unsigned raw[4] = { a.x, a.y, a.z, a.w };
#pragma unroll
				for (int j = 0; j < 4; ++j) {
					const int c = 4 * k + j;
					const int wv = (int)((ww[c >> 1] >> (16 * (c & 1))) & 0xFFFFu);
					stage[xch_idx(c * 256 + t)] = c16_pack((c16_re(raw[j]) - kI) * wv, (c16_im(raw[j]) - kQ) * wv);
				}
			}
		}
	}
	__syncthreads();

	/* position 16t + r is column c = t >> 4, row bitrev8(q) */
	X2 x[kPts];
	const int c = t >> 4;
#pragma unroll
	for (int r = 0; r < kPts; ++r) {
		const int i = (brev4(r) << 4) | brev_bits((unsigned)(t & 15), 4);
		x[r] = x_unpack(stage[xch_idx(c * 256 + i)]);
	}

	TwLargeA tw;
	tw.twc = twc;
	tw.tw0 = &prm.tw0;
	engine_fft<8>(x, stage, t, tw);

	/* scatter: column n_low lands on positions (bitrev(n_low) << 8) | q */
	c16 *dst = prm.scratch + (long long)rel * N;
#pragma unroll
	for (int r = 0; r < kPts; ++r) {
		const int p = last_pos<8>(t, r);
		const int cc = p >> 8, q = p & 255;
		const long long P = ((long long)brev_bits((unsigned)(16 * tile + cc), L - 8) << 8) | q;
		dst[P] = x_pack(x[r]);
	}
}

/* ---- round B ----------------------------------------------------------- */

/*
 * Round-B twiddles.  Stage 8+se pairs positions whose low 8+se bits m = (ilow << 8) | plow
 * select tw[m << (L-9-se)].  For se >= 4 the lanes of a warp differ in ilow, i.e. their
 * entries are 2^(L-1-se) apart in tw[]: one 32-byte sector per lane.  The host therefore
 * also provides the same values re-ordered as twb[se][plow][ilow] (ilow fastest), so that a
 * warp reads one or two contiguous 128-byte runs.
 */
SCAN_DEV constexpr long long twb_offset(int se) { return 256ll * ((1 << se) - 16); } /* se >= 4 */

template <int LB>
struct TwLargeB {
	static constexpr bool kTrivial = false;
	const int2 *tw;
	const int2 *twb;
	int plow0, L;
	template <int K>
	SCAN_DEV int2 get(int se, int pa) const
	{
		const int col = pa >> LB, i = pa & ((1 << LB) - 1);
		const int ilow = i & ((1 << se) - 1);
		if (K >= 1)
			return __ldg(twb + twb_offset(se) + ((long long)(plow0 + col) << se) + ilow);
		const long long m = ((long long)ilow << 8) | (plow0 + col);
		return __ldg(tw + (m << (L - 9 - se)));
	}
};

SCAN_DEV void accumulate_bin(long long *dst, c16 x, bool peak)
{
	const int re = c16_re(x), im = c16_im(x);
	const unsigned pw = (unsigned)(re * re) + (unsigned)(im * im);
	if (peak)
		atomicMax(dst, (long long)pw);
	else
		atomicAdd((unsigned long long *)dst, (unsigned long long)pw);
}

/* Tile transposes of round B: columns are 2^LB words apart, so on top of the engine's
 * p>>4 padding the column index is spread over the banks with 2 * (p >> 8). */
SCAN_DEV int tile_idx(int p) { return p + (p >> 4) + 2 * (p >> 8); }
constexpr int kLargeSmemB = (kWS + kWS / 16 + 2 * (kWS / 256) + 16) * 4;

template <int LB, bool LAST, bool PEAK>
__global__ void __launch_bounds__(kThreads, 2) /* (3 CTAs per SM at 80 registers: measured 103 vs 105 G samples/s) */
large_round_b_kernel(const SCAN_GRID_CONSTANT LargeParams prm)
{
	constexpr bool SK = false;
	[[maybe_unused]] unsigned long long *const s2 = nullptr;
#include "large_round_b_body.inl"
}

/* RTLSDR_GPU_FLAG_SPECTRAL_KURTOSIS, N <= 2^16: the last round B with pw^2 added to s2 [tune_count << L][2] beside
 * each |X|^2 (sk.cuh) */
template <int LB>
__global__ void __launch_bounds__(kThreads, 2)
large_round_b_sk_kernel(const SCAN_GRID_CONSTANT LargeParams prm, unsigned long long *s2)
{
	constexpr bool SK = true, LAST = true;
	[[maybe_unused]] constexpr bool PEAK = false;
#include "large_round_b_body.inl"
}

/*
 * Round B (stages 8..15, not the last round), software pipelined, items in TILE-MAJOR order
 * (all reads of one tile, then the next tile): a resident grid of CTAs walks equal runs of the (tile, read)
 * items like scan_small_kernel walks reads.  A tile is 256 strided rows x 16 consecutive positions and stays in
 * the scratch's own row-major order in shared memory, so the next one arrives by 8-byte cp.async while this one
 * is transformed, and the result leaves with 16-byte loads / stores.  Word (row i, column c) lives at
 *     272 * (i >> 4) + 16 * (i & 15) + (c ^ 2 * (((i >> 1) ^ (i >> 5)) & 7))
 * (16 pad words per 16 rows + an XOR on column bits 1..3): the engine reads register r of thread t at row
 * 16 * (t & 15) + r, column t >> 4 and writes it back at row 16 * r + (t & 15) -- both patterns touch 32
 * different banks per warp, and column pairs stay adjacent and 8-byte aligned.
 * The twiddles of a tile depend on its 16 columns only, not on the read: in tile-major order a CTA's whole run
 * uses one or two sets, kept in shared memory (the 16 x 240 values of stages 12..15 are contiguous in the
 * host's re-ordered table twb[se][plow][ilow], those of stages 8..11 are 16 x 15 gathered values).  The
 * one-tile-per-CTA kernel fetches 30 twiddles per thread and tile through L1/L2 (61 KB requested per 16 KB
 * tile; ncu: 0.93 long-scoreboard stall cycles per issued instruction).
 */
constexpr int kTileRowWords = 4352; /* 16 row groups x 272 words */
constexpr int kTwsWords = (16 * 240 + 16 * 15 + 16) * 2; /* int2 tables of one tile */
constexpr int kLargeSmemBP = kTileRowWords * 4 * 2 + kXchWords * 4 + kTwsWords * 4;

SCAN_DEV int tile_row_swz(int i) { return 2 * (((i >> 1) ^ (i >> 5)) & 7); }
SCAN_DEV int tile_row_base(int i) { return 272 * (i >> 4) + 16 * (i & 15); }

struct TwLargeBS {
	static constexpr bool kTrivial = false;
	const int2 *t1; /* [se = 4..7][col][ilow]: stage se at 16 * ((1 << se) - 16) */
	const int2 *t0; /* [col][15]: stage se < 4, group g at (1 << se) - 1 + g */
	template <int K>
	SCAN_DEV int2 get(int se, int pa) const
	{
		const int col = pa >> 8, ilow = pa & ((1 << se) - 1);
		if (K >= 1)
			return t1[16 * ((1 << se) - 16) + (col << se) + ilow];
		return t0[col * 15 + (1 << se) - 1 + ilow];
	}
};

__global__ void __launch_bounds__(kThreads, 2)
large_round_b_pipe_kernel(const SCAN_GRID_CONSTANT LargeParams prm)
{
	constexpr int LB = 8;
	SCAN_DYN_SMEM(smem);
	c16 *in = (c16 *)smem;                 /* two tiles */
	c16 *xch = in + 2 * kTileRowWords;
	int2 *tws1 = (int2 *)(xch + kXchWords);
	int2 *tws0 = tws1 + 16 * 240;
	const int t = threadIdx.x, L = prm.L;
	const long long N = 1ll << L;
	const int n_rel = prm.n_entries;
	const long long W = (long long)n_rel << prm.tiles_log2;
	const long long w0 = W * blockIdx.x / gridDim.x, w1 = W * (blockIdx.x + 1) / gridDim.x;
	if (w0 >= w1)
		return;
	/* item w = tile * n_rel + rel */
	int tile = (int)(w0 / n_rel), rel = (int)(w0 - (long long)tile * n_rel);

	auto tile_ptr = [&](int tl, int rl) {
		return prm.scratch + (long long)rl * N + ((long long)(tl >> 4) << (8 + LB)) + (tl & 15) * 16;
	};
	auto prefetch = [&](int tl, int rl, int buf) {
		const c16 *data = tile_ptr(tl, rl);
		c16 *dst = in + buf * kTileRowWords;
#pragma unroll
		for (int k = 0; k < 8; ++k) {
			const int q = t + kThreads * k, i = q >> 3, j = q & 7;
			cp_async8(dst + tile_row_base(i) + ((2 * j) ^ tile_row_swz(i)), data + ((long long)i << 8) + 2 * j);
		}
		cp_async_commit();
	};
	auto load_tables = [&](int tl) {
		const int plow0 = (tl & 15) * 16;
#pragma unroll
		for (int se = 4; se < 8; ++se) {
			const int2 *src = prm.twb + twb_offset(se) + ((long long)plow0 << se);
			int2 *dst = tws1 + 16 * ((1 << se) - 16);
			for (int k = t; k < (8 << se); k += kThreads) /* 16 << se entries, two per 16-byte copy */
				cp_async16(dst + 2 * k, src + 2 * k);
		}
		if (t < 240) {
			const int col = t / 15, e = t % 15;
			int se = 0;
			while (e >= (2 << se) - 1)
				se++;
			const long long m = ((long long)(e - ((1 << se) - 1)) << 8) | (plow0 + col);
			tws0[t] = prm.tw[m << (L - 9 - se)];
		}
		cp_async_commit();
	};
	/* this tile's twiddle tables do not depend on round A: they are on their way before the wait */
	pdl_launch_dependents();
	load_tables(tile);
	int tab_tile = tile;
	pdl_wait();
	prefetch(tile, rel, 0);
	TwLargeBS tw;
	tw.t1 = tws1;
	tw.t0 = tws0;
	for (long long w = w0; w < w1; ++w) {
		const int buf = (int)(w - w0) & 1;
		c16 *cur = in + buf * kTileRowWords;
		c16 *data = const_cast<c16 *>(tile_ptr(tile, rel));
		cp_async_wait_all();
		__syncthreads(); /* tile w has landed for everybody; the other buffer's stores of item w-1 have been read */
		int ntile = tile, nrel = rel + 1;
		if (nrel == n_rel)
			nrel = 0, ntile++;
		if (w + 1 < w1)
			prefetch(ntile, nrel, buf ^ 1);
		if (tile != tab_tile) { /* CTA-uniform, once or twice per run: nobody reads the old tables any more */
			tab_tile = tile;
			load_tables(tile);
			cp_async_wait_all();
			__syncthreads();
		}
		X2 x[kPts];
		{
			const int col = t >> 4;
#pragma unroll
			for (int r = 0; r < kPts; ++r) {
				const int i = ((t & 15) << 4) | r;
				x[r] = x_unpack(cur[tile_row_base(i) + (col ^ tile_row_swz(i))]);
			}
		}
		run_pass<0, LB>(x, t, tw);
		exchange<0, 1, false>(x, xch, t, t);
		run_pass<1, LB>(x, t, tw);
		{
			const int col = t >> 4;
#pragma unroll
			for (int r = 0; r < kPts; ++r) {
				const int i = (r << 4) | (t & 15);
				cur[tile_row_base(i) + (col ^ tile_row_swz(i))] = x_pack(x[r]);
			}
		}
		__syncthreads();
#pragma unroll
		for (int k = 0; k < 4; ++k) {
			const int q = t + kThreads * k, i = q >> 2, j = q & 3;
			const int s = tile_row_swz(i);
			uint4 v = *(const uint4 *)(cur + tile_row_base(i) + ((4 * j) ^ (s & 12)));
			if (s & 2)
				v = uint4{ v.z, v.w, v.x, v.y };
			*(uint4 *)(data + ((long long)i << 8) + 4 * j) = v;
		}
		tile = ntile, rel = nrel;
	}
}

/* ---- round C ----------------------------------------------------------- */

constexpr int kRoundCReads = 16; /* reads one CTA of round C walks through at most */

/* reads per CTA of round C: up to kRoundCReads (register accumulation before the atomics), fewer when the
 * launch would otherwise not fill the GPU (at least ~4 CTAs of `cta_x` per SM) */
inline int round_c_reads(int n_reads, int cta_x)
{
	const long long want = ((long long)n_reads * cta_x + 591) / 592;
	return (int)(want < 1 ? 1 : (want > kRoundCReads ? kRoundCReads : want));
}

/*
 * VEC consecutive positions per thread (16-byte loads for VEC = 4) and the NEXT read's words requested before
 * the current read's butterflies: the round is a pure stream over the scratch (4 bytes per sample, one butterfly
 * per 2^LC points and stage), so what matters is bytes in flight -- the scalar version (two 4-byte loads in
 * flight per thread) ran at 2.3 TB/s.
 */
template <int LC, bool PEAK, int VEC>
__global__ void __launch_bounds__(kThreads)
large_round_c_kernel(const SCAN_GRID_CONSTANT LargeParams prm)
{
	constexpr bool SK = false;
	[[maybe_unused]] unsigned long long *const s2 = nullptr;
#include "large_round_c_body.inl"
}

/* RTLSDR_GPU_FLAG_SPECTRAL_KURTOSIS, N >= 2^17: round C with 128-bit sum |X|^4 register partials beside the power
 * sums, flushed into s2 [tune_count << L][2] at the same hop changes */
template <int LC, int VEC>
__global__ void __launch_bounds__(kThreads)
large_round_c_sk_kernel(const SCAN_GRID_CONSTANT LargeParams prm, unsigned long long *s2)
{
	constexpr bool SK = true, PEAK = false;
#include "large_round_c_body.inl"
}

/* positions per thread of round C for 2^LC strided points: 16-byte loads while the accumulators fit */
constexpr int round_c_vec(int lc) { return lc <= 2 ? 4 : (lc == 3 ? 2 : 1); }

} // namespace rscan
