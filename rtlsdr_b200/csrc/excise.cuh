/*
 * excise.cuh -- spectral-kurtosis RFI excision (RTLSDR_GPU_FLAG_SK_EXCISION, Nita & Gary 2010): the interval is cut
 * into sub-integrations, a bin's sub-integration joins its long-term average only when its SK lies within
 * [1 - k_low sigma(M), 1 + k_high sigma(M)].
 *
 * State per hop and bin, natural FFT order, beside S1 (the bins) and S2 (sk.cuh):
 *   snap_s1 int64, snap_s2 (lo, hi) u64  S1 and S2 at the last fold
 *   c1      int64                        the clean power sum
 *   b1      int32                        the clean FFT-block count
 * and per hop snap_smp (int64), the sample counter at the last fold: 36 B per bin.  Every read-and-zero of the
 * handle also zeroes this state for the hops it zeroes.
 */
#pragma once
#include "scan_kernels.cuh"
#include "sk.cuh"

namespace rscan {

struct ExciseFoldParams {
	const long long *avg;               /* [hops << bin_e] S1 */
	const long long *samples;           /* [hops] */
	const unsigned long long *s2;       /* [hops << bin_e][2] */
	long long *snap_s1;                 /* [hops << bin_e] */
	unsigned long long *snap_s2;        /* [hops << bin_e][2] */
	long long *c1;                      /* [hops << bin_e] */
	int *b1;                            /* [hops << bin_e] */
	long long *snap_smp;                /* [hops] */
	unsigned *ticket;                   /* [hops], 0 between launches */
	double k_low, k_high;
	int bin_e;
	int downsample;
};

/* One sub-integration of every hop closes: grid (bins / 256, hops).  Per bin
 *   M = (samples - snap_smp) / ds, dS1 = S1 - snap_s1, dS2 = S2 - snap_s2 (128-bit, borrow out of the low word),
 *   sk = sk_from_moments(dS1, dS2, M), flagged iff sk is not NaN and sk < 1 - k_low sigma or sk > 1 + k_high sigma,
 *   clean: c1 += dS1, b1 += M; then the snapshots move to S1, S2.
 * The hop's snap_smp is read by every CTA of the hop, so the last CTA to finish (ticket) moves it.  About 96 B of
 * memory traffic per bin.  Plain stream order behind the transforms (no programmatic dependent launch either way). */
__global__ void __launch_bounds__(256)
excise_fold_kernel(const SCAN_GRID_CONSTANT ExciseFoldParams prm)
{
	const int hop = blockIdx.y;
	const int n = 1 << prm.bin_e;
	const int j = blockIdx.x * blockDim.x + threadIdx.x;
	const long long smp = prm.samples[hop];
	const long long M = (smp - prm.snap_smp[hop]) / prm.downsample;
	if (j < n) {
		const double sigma = sk_sigma(M);
		const double lo = sk_add(1.0, -sk_mul(prm.k_low, sigma)), hi = sk_add(1.0, sk_mul(prm.k_high, sigma));
		const long long b = ((long long)hop << prm.bin_e) + j;
		const long long S1 = prm.avg[b];
		const unsigned long long s2lo = prm.s2[2 * b], s2hi = prm.s2[2 * b + 1];
		const unsigned long long plo = prm.snap_s2[2 * b], phi = prm.snap_s2[2 * b + 1];
		const long long d1 = S1 - prm.snap_s1[b];
		const unsigned long long dlo = s2lo - plo, dhi = s2hi - phi - (s2lo < plo ? 1ull : 0ull);
		const double sk = sk_from_moments(d1, dlo, dhi, M);
		const bool flagged = sk == sk && (sk < lo || sk > hi);
		if (!flagged) {
			prm.c1[b] += d1;
			prm.b1[b] += (int)M;
		}
		prm.snap_s1[b] = S1;
		prm.snap_s2[2 * b] = s2lo;
		prm.snap_s2[2 * b + 1] = s2hi;
	}
	__shared__ unsigned ticket;
	__threadfence();
	__syncthreads();
	if (threadIdx.x == 0)
		ticket = atomicAdd(prm.ticket + hop, 1u);
	__syncthreads();
	if (ticket == gridDim.x - 1 && threadIdx.x == 0) {
		prm.snap_smp[hop] = smp;
		prm.ticket[hop] = 0;
	}
}

struct ExciseReportParams {
	const long long *c1;                /* [hops << bin_e] */
	const int *b1;                      /* [hops << bin_e] */
	const long long *snap_smp;          /* [hops] */
	int *samples_out;                   /* optional [hops]: snap_smp */
	double *db;                         /* optional [hops][db_count] excised dB rows */
	double *flagged;                    /* optional [hops][db_count] flag fractions */
	int bin_e;
	int i1, i2;
	int rate;
	int downsample;
};

/* The excised report (a peek: nothing is zeroed), in the dB row's layout: bin 0 takes bin 1's (c1, b1) (csv_dbm's
 * DC nuke), half swap, crop [i1, i2], duplicate of bin i2.  The dB row is the epilogue's (epilogue_body.inl) with the
 * hop's sample count replaced by the bin's clean samples s = (double)(b1 * ds): 10 log10(v / rate / s), the duplicate
 * 10 log10(v / (rate * s)), never smoothed; b1 = 0 gives a quiet NaN with the sign bit clear.  The flag fraction is
 * (F - b1) / F, F = snap_smp / ds the folded FFT blocks, NaN when F = 0.  Grid (db_count / 256, hops).  (C1 and B1
 * themselves are plain copies of the state, made with cudaMemcpyAsync.) */
template <bool GUARD>
__global__ void __launch_bounds__(256)
excised_report_kernel(const SCAN_GRID_CONSTANT ExciseReportParams prm)
{
	const int hop = blockIdx.y;
	const int n = 1 << prm.bin_e;
	const int count = prm.i2 - prm.i1 + 2;
	const int k = blockIdx.x * blockDim.x + threadIdx.x;
	const long long base = (long long)hop << prm.bin_e;
	if (prm.samples_out && k == 0)
		prm.samples_out[hop] = (int)prm.snap_smp[hop];
	if (k >= count || !(prm.db || prm.flagged))
		return;
	const int i = (k < count - 1) ? prm.i1 + k : prm.i2;
	int j = (i + n / 2) & (n - 1); /* undo the half swap */
	if (j == 0)
		j = 1;                     /* avg[0] = avg[1] */
	const long long v = prm.c1[base + j];
	const int B = prm.b1[base + j];
	const long long o = (long long)hop * count + k;
	if (prm.db) {
		double d = NAN;
		if (B != 0) {
			const double rate = (double)prm.rate, s = (double)((long long)B * prm.downsample);
			if (k < count - 1)
				d = __ddiv_rn(__ddiv_rn(epilogue_value<GUARD>(v), rate), s);
			else
				d = __ddiv_rn(epilogue_value<GUARD>(v), __dmul_rn(rate, s));
			d = 10 * log10(d);
		}
		prm.db[o] = d;
	}
	if (prm.flagged) {
		const long long F = prm.snap_smp[hop] / prm.downsample;
		prm.flagged[o] = F == 0 ? (double)NAN : sk_div((double)(F - B), (double)F);
	}
}

} // namespace rscan
