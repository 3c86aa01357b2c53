/*
 * scan_guard.cuh -- RTLSDR_GPU_FLAG_GUARD_BITS: fix_fft (rtl_power.c:271-327) carried with F = 8 fractional guard
 * bits in int32, for every bin count (2^1 .. 2^21) and every front end.
 *
 * The front end is the reference's (u8 - 127, decimators, remove_dc, wrapping int16 window multiply); its int16
 * output x becomes v = x << 8.  The transform keeps fix_fft's bit reversal, halved Q15 twiddles and per-stage
 * halving; only the data is wider:
 *   R(p) = (p + 2^14) >> 15 on the exact (64-bit) product,
 *   t = (R(wr br) - R(wi bi), R(wr bi) + R(wi br)),  q = a >> 1,  a' = q + t,  b' = q - t    (int32)
 * Every value stays below 2^15 * sqrt(2) * 2^8 plus one unit per stage < 2^24, so int32 never wraps.
 * The per-block power is pw = (re^2 + im^2 + 2^7) >> 8 < 2^40 (exact in 64 bits); the bins add it (or keep the
 * maximum under peak hold) in the handle's int64 bins, and SK adds pw^2 < 2^80 to the 128-bit S2.
 *
 * Two plain kernels instead of the tuned int16 engine (a complex sample is two words here):
 *   guard_fft_a_kernel  a CTA takes runs of 4096-position working sets: gathers the front-end output in
 *                       bit-reversed order into shared memory (32 KiB of int2) and runs stages 0 .. min(L, 12)-1,
 *                       one radix-2 stage per barrier.  N <= 4096: 4096/N whole blocks per working set, |X|^2 is
 *                       accumulated right there.  N > 4096: the working set is 4096 consecutive positions of the
 *                       read's one block and goes to a global scratch (8 bytes per sample).
 *   guard_fft_b_kernel  N > 4096: stages 12 .. L-1.  A CTA owns a column set, positions c*C + j + (k << 12),
 *                       j < C = 2^(24-L), k < 2^(L-12), for a run of reads, and accumulates their |X|^2 in
 *                       registers: its bins do not change from read to read.
 * Register partials are flushed with global atomics when the hop changes and at the end of a CTA's run.
 */
#pragma once
#include "scan_kernels.cuh"
#include "sk.cuh"

namespace rscan {

constexpr int kGuardF = 8;

enum GuardMode { GUARD_SUM = 0, GUARD_PEAK = 1, GUARD_SK = 2 };

struct GuardParams {
	const uint8_t *base;        /* u8 reads, or decimated c16 images (IN16) */
	const long long *read_off;  /* u8: byte offset per absolute entry */
	long long regular_stride;   /* IN16: image bytes; image of entry e (relative) at base + e * regular_stride */
	int entry_base;             /* absolute index of this launch's entry 0 */
	int n_entries;
	const int *hop_of;          /* hop per absolute entry */
	const int2 *dc_u8;          /* u8: [n_entries] 127 + remove_dc's averages (dc_sums_u8_kernel) */
	const int *dc_ave;          /* IN16: [n_entries][2] remove_dc's averages (dc_finalize_kernel) */
	int l_len;                  /* IN16: int16 values remove_dc covers */
	int n_blocks;               /* FFT blocks per read */
	int blocks_padded;          /* IN16: blocks per image */
	int L;
	const int2 *tw;             /* [N/2] halved twiddles */
	const uint16_t *win;        /* [N] low 16 bits of the window */
	int2 *scratch;              /* N > 4096: [n_entries][N] after stages 0..11 */
	long long *avg;             /* [hops << L] */
	long long *samples;         /* [hops] */
	int samples_per_read;
	unsigned long long *s2;     /* GUARD_SK: [hops << L][2] (lo, hi) */
	int b_groups;               /* guard_fft_b_kernel: CTAs (grid.y) sharing the reads */
};

constexpr int kGuardSlots = kWS / kThreads; /* 16 positions per thread */

/* R(w * b) = (w * b + 2^14) >> 15, exact */
SCAN_DEV int guard_mpy(int w, int b)
{
	return (int)(((long long)w * b + 16384) >> 15);
}

/* one radix-2 butterfly of fix_fft on int32 data: a' = a/2 + w*b, b' = a/2 - w*b */
SCAN_DEV void guard_butterfly(int2 &a, int2 &b, int2 w)
{
	const int tr = guard_mpy(w.x, b.x) - guard_mpy(w.y, b.y);
	const int ti = guard_mpy(w.x, b.y) + guard_mpy(w.y, b.x);
	const int qr = a.x >> 1, qi = a.y >> 1;
	b = make_int2(qr - tr, qi - ti);
	a = make_int2(qr + tr, qi + ti);
}

SCAN_DEV unsigned long long guard_power(int2 v)
{
	const long long p = (long long)v.x * v.x + (long long)v.y * v.y;
	return ((unsigned long long)p + (1ull << (kGuardF - 1))) >> kGuardF;
}

/* pw^2 (< 2^80) as (lo, hi) */
SCAN_DEV void guard_square(unsigned long long pw, unsigned long long &lo, unsigned long long &hi)
{
#ifdef SCAN_EMU
	const unsigned __int128 p = (unsigned __int128)pw * pw;
	lo = (unsigned long long)p;
	hi = (unsigned long long)(p >> 64);
#else
	lo = pw * pw;
	hi = __umul64hi(pw, pw);
#endif
}

template <int MODE>
struct GuardAcc {
	unsigned long long a[kGuardSlots];
	unsigned long long lo[MODE == GUARD_SK ? kGuardSlots : 1];
	unsigned long long hi[MODE == GUARD_SK ? kGuardSlots : 1];

	SCAN_DEV void zero()
	{
#pragma unroll
		for (int i = 0; i < kGuardSlots; ++i) {
			a[i] = 0;
			if constexpr (MODE == GUARD_SK) {
				lo[i] = 0;
				hi[i] = 0;
			}
		}
	}
	SCAN_DEV void add(int i, unsigned long long pw)
	{
		if constexpr (MODE == GUARD_PEAK) {
			a[i] = pw > a[i] ? pw : a[i];
		} else {
			a[i] += pw;
			if constexpr (MODE == GUARD_SK) {
				unsigned long long l, h;
				guard_square(pw, l, h);
				lo[i] += l;
				hi[i] += h + (lo[i] < l ? 1ull : 0ull);
			}
		}
	}
	/* slot j into slot i (same bin) */
	SCAN_DEV void fold(int i, int j)
	{
		if constexpr (MODE == GUARD_PEAK) {
			a[i] = a[j] > a[i] ? a[j] : a[i];
		} else {
			a[i] += a[j];
			if constexpr (MODE == GUARD_SK) {
				lo[i] += lo[j];
				hi[i] += hi[j] + (lo[i] < lo[j] ? 1ull : 0ull);
			}
		}
	}
	/* slots i >= M into slot i mod M (they hold the same bin) */
	template <int M>
	SCAN_DEV void fold_to()
	{
#pragma unroll
		for (int i = M; i < kGuardSlots; ++i)
			fold(i % M, i);
	}
	SCAN_DEV void flush(int i, long long *bins, unsigned long long *s2, long long bin)
	{
		if constexpr (MODE == GUARD_PEAK) {
			if (a[i])
				atomicMax(bins + bin, (long long)a[i]);
		} else {
			if (a[i])
				atomicAdd((unsigned long long *)(bins + bin), a[i]);
			if constexpr (MODE == GUARD_SK) {
				if (lo[i] | hi[i])
					sk_atomic_add(s2 + 2 * bin, lo[i], hi[i]);
			}
		}
	}
};

/* the radix-2 stages [s0, s1) of positions laid out in shared memory; pos(b) gives the shared index of the
 * upper input of butterfly b (< 2048) at stage s, its partner is `half` entries further on, and twg(b) its
 * twiddle group in the whole transform */
template <class Idx>
SCAN_DEV void guard_stages(int2 *sh, const int2 *tw, int L, int s0, int s1, int t, const Idx &idx)
{
	for (int s = s0; s < s1; ++s) {
#pragma unroll 4
		for (int r = 0; r < kWS / 2 / kThreads; ++r) {
			const int b = t + r * kThreads;
			int i, p;
			long long g;
			idx(s, b, i, p, g);
			const int2 w = __ldg(tw + (g << (L - 1 - s)));
			int2 a = sh[i], c = sh[p];
			guard_butterfly(a, c, w);
			sh[i] = a;
			sh[p] = c;
		}
		__syncthreads();
	}
}

/* front end of sample k (index inside its read) of relative entry e, times 2^F */
template <bool IN16>
SCAN_DEV int2 guard_front(const GuardParams &prm, const uint8_t *src, int e, long long k)
{
	const int wv = (int)prm.win[k & ((1ll << prm.L) - 1)];
	int re, im;
	if constexpr (!IN16) {
		const unsigned raw = *(const uint16_t *)(src + 2 * k);
		const int2 c = prm.dc_u8[e];
		re = ((int)(raw & 0xFFu) - c.x) * wv;
		im = ((int)(raw >> 8) - c.y) * wv;
	} else {
		const c16 raw = ((const c16 *)src)[k];
		re = c16_re(raw);
		im = c16_im(raw);
		if (2 * k < prm.l_len)
			re -= prm.dc_ave[2 * e];
		if (2 * k + 1 < prm.l_len)
			im -= prm.dc_ave[2 * e + 1];
		re *= wv;
		im *= wv;
	}
	/* the reference's int16 store of the windowed value, then the guard bits */
	return make_int2((int)(int16_t)(uint16_t)(re & 0xFFFF) * (1 << kGuardF),
			 (int)(int16_t)(uint16_t)(im & 0xFFFF) * (1 << kGuardF));
}

template <bool IN16, int MODE>
__global__ void __launch_bounds__(kThreads)
guard_fft_a_kernel(const SCAN_GRID_CONSTANT GuardParams prm)
{
	__shared__ int2 sh[kWS];
	const int t = threadIdx.x, L = prm.L;
	const long long N = 1ll << L;
	const bool small = L <= 12;
	/* working sets per read: N <= 4096: ceil(n_blocks N / 4096) sets of 4096/N blocks; N > 4096: N / 4096 */
	const long long span = small ? (long long)prm.n_blocks * N : N;
	const int wpr = (int)((span + kWS - 1) / kWS);
	const long long items = (long long)prm.n_entries * wpr;
	const long long lo = items * blockIdx.x / gridDim.x, hi = items * (blockIdx.x + 1) / gridDim.x;
	const int sl = small ? L : 12;

	GuardAcc<MODE> acc;
	acc.zero();
	for (long long it = lo; it < hi; ++it) {
		const int e = (int)(it / wpr), w = (int)(it - (long long)e * wpr);
		const int hop = prm.hop_of[prm.entry_base + e];
		const uint8_t *src = IN16 ? prm.base + (long long)e * prm.regular_stride
					  : prm.base + prm.read_off[prm.entry_base + e];
		if (w == 0 && t == 0) /* tunes[hop].samples += ds per FFT block (rtl_power.c:717) */
			atomicAdd((unsigned long long *)(prm.samples + hop), (unsigned long long)prm.samples_per_read);

		/* gather: position P of the working set holds sample brev(P) of its block (rtl_power.c:282-297) */
#pragma unroll 4
		for (int i = 0; i < kGuardSlots; ++i) {
			const int P = t + i * kThreads;
			const long long G = (long long)w * kWS + P;
			int2 v = make_int2(0, 0);
			if (G < span) {
				const long long blk = G >> L;
				const long long k = (blk << L) | brev_bits((unsigned)(G & (N - 1)), L);
				v = guard_front<IN16>(prm, src, e, k);
			}
			sh[P] = v;
		}
		__syncthreads();
		guard_stages(sh, prm.tw, L, 0, sl, t, [](int s, int b, int &i, int &p, long long &g) {
			const int half = 1 << s;
			g = b & (half - 1);
			i = ((b >> s) << (s + 1)) | (int)g;
			p = i + half;
		});

		if (!small) {
			int2 *dst = prm.scratch + (long long)e * N + (long long)w * kWS;
#pragma unroll 4
			for (int i = 0; i < kGuardSlots; ++i)
				dst[t + i * kThreads] = sh[t + i * kThreads];
		} else {
#pragma unroll
			for (int i = 0; i < kGuardSlots; ++i) {
				const long long G = (long long)w * kWS + t + i * kThreads;
				if (G < span)
					acc.add(i, guard_power(sh[t + i * kThreads]));
			}
		}
		__syncthreads(); /* sh is refilled by the next working set */

		if (small) {
			const bool last = it + 1 >= hi;
			const int next_hop = last ? -1 : prm.hop_of[prm.entry_base + (int)((it + 1) / wpr)];
			if (next_hop != hop) {
				/* slot i holds bin (t + 256 i) mod N: fold the slots that share a bin, then one atomic per bin */
				const int m = N > kThreads ? (int)(N / kThreads) : 1;
				switch (m) { /* constant slot indices keep the partials in registers */
				case 1: acc.template fold_to<1>(); break;
				case 2: acc.template fold_to<2>(); break;
				case 4: acc.template fold_to<4>(); break;
				case 8: acc.template fold_to<8>(); break;
				default: break;
				}
				long long *bins = prm.avg + ((long long)hop << L);
				unsigned long long *s2 = MODE == GUARD_SK ? prm.s2 + ((long long)hop << (L + 1)) : nullptr;
#pragma unroll
				for (int i = 0; i < kGuardSlots; ++i)
					if (i < m)
						acc.flush(i, bins, s2, (t + i * kThreads) & (N - 1));
				acc.zero();
			}
		}
	}
}

template <int MODE>
__global__ void __launch_bounds__(kThreads)
guard_fft_b_kernel(const SCAN_GRID_CONSTANT GuardParams prm)
{
	__shared__ int2 sh[kWS];
	const int t = threadIdx.x, L = prm.L;
	const long long N = 1ll << L;
	const int lk = L - 12, C = kWS >> lk; /* 2^lk strided rows of C consecutive positions */
	const int c = blockIdx.x;
	const int e_lo = (int)((long long)prm.n_entries * blockIdx.y / gridDim.y);
	const int e_hi = (int)((long long)prm.n_entries * (blockIdx.y + 1) / gridDim.y);

	GuardAcc<MODE> acc;
	acc.zero();
	for (int e = e_lo; e < e_hi; ++e) {
		const int hop = prm.hop_of[prm.entry_base + e];
		const int2 *src = prm.scratch + (long long)e * N + (long long)c * C;
#pragma unroll 4
		for (int i = 0; i < kGuardSlots; ++i) {
			const int x = t + i * kThreads, k = x / C, j = x - k * C;
			sh[x] = src[((long long)k << 12) + j];
		}
		__syncthreads();
		guard_stages(sh, prm.tw, L, 12, L, t, [C, c](int s, int b, int &i, int &p, long long &g) {
			const int sb = s - 12, half = 1 << sb;
			const int kk = b / C, j = b - kk * C;
			const int gk = kk & (half - 1);
			const int ki = ((kk >> sb) << (sb + 1)) | gk;
			i = ki * C + j;
			p = i + half * C;
			g = ((long long)gk << 12) | (c * C + j);
		});
#pragma unroll
		for (int i = 0; i < kGuardSlots; ++i)
			acc.add(i, guard_power(sh[t + i * kThreads]));
		__syncthreads();

		if (e + 1 >= e_hi || prm.hop_of[prm.entry_base + e + 1] != hop) {
			long long *bins = prm.avg + ((long long)hop << L);
			unsigned long long *s2 = MODE == GUARD_SK ? prm.s2 + ((long long)hop << (L + 1)) : nullptr;
#pragma unroll
			for (int i = 0; i < kGuardSlots; ++i) {
				const int x = t + i * kThreads, k = x / C, j = x - k * C;
				acc.flush(i, bins, s2, ((long long)k << 12) + (long long)c * C + j);
			}
			acc.zero();
		}
	}
}

} // namespace rscan
