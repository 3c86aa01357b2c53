/*
 * sk.cuh -- spectral kurtosis per bin (Nita & Gary 2010) from the two power moments
 *   S1 = sum |X|^2   (the handle's int64 bins, rtl_power.c:708-716)
 *   S2 = sum |X|^4   (unsigned 128-bit: pw = re^2 + im^2 <= 2^31, pw^2 <= 2^62, so a full-scale input
 *                     overflows 64 bits after four FFT blocks)
 * over the M FFT blocks of an interval:
 *   SK = (M+1)/(M-1) * (M * S2 / S1^2 - 1),  quiet NaN when M < 2 or S1 = 0.
 *
 * The evaluation order is fixed and every step is a correctly rounded IEEE double operation, so the device
 * (`__dmul_rn` / `__ddiv_rn` / `__dadd_rn`: no contraction) and a host build of this header compute the same bits:
 *   s1 = rn(S1); s2 = rn(S2); a = M*s2; b = s1*s1; c = a/b; d = c - 1; e = (M+1)/(M-1); sk = e*d
 * Host builds must not contract either (nothing here has a multiply feeding an add, so no FMA can form).
 *
 * S2 lives in device memory as two u64 words (lo, hi) per bin.  Global accumulation is exact and independent of
 * the order: atomicAdd on lo returns the old word, and a wrap (old + v < old) adds 1 to hi.
 */
#pragma once
#include "scan_compat.cuh"

#if defined(__CUDACC__) && !defined(SCAN_EMU)
#define SK_HD __host__ __device__ __forceinline__
#else
#define SK_HD inline
#endif

#include <math.h>

namespace rscan {

/* round-to-nearest-even u64 -> double */
SK_HD double sk_u64_to_double(unsigned long long v)
{
#ifdef __CUDA_ARCH__
	return __ull2double_rn(v);
#else
	return (double)v;
#endif
}

SK_HD int sk_clz64(unsigned long long v) /* v != 0 */
{
#ifdef __CUDA_ARCH__
	return __clzll((long long)v);
#else
	return __builtin_clzll(v);
#endif
}

/* correctly rounded (hi:lo) -> double, equal to gcc's (double)(unsigned __int128): keep the top 64 bits, OR every
 * bit shifted out into bit 0 (a sticky bit below the 53 kept ones, so ties and "above a tie" round as they must),
 * round that, and scale by the exact power of two */
SK_HD double sk_u128_to_double(unsigned long long lo, unsigned long long hi)
{
	if (hi == 0)
		return sk_u64_to_double(lo);
	const int sh = 64 - sk_clz64(hi); /* 1..64 bits above the low word */
	const unsigned long long top = sh == 64 ? hi : (hi << (64 - sh)) | (lo >> sh);
	const unsigned long long lost = sh == 64 ? lo : lo & ((1ull << sh) - 1);
	return ldexp(sk_u64_to_double(top | (lost != 0 ? 1ull : 0ull)), sh);
}

SK_HD double sk_mul(double a, double b)
{
#ifdef __CUDA_ARCH__
	return __dmul_rn(a, b);
#else
	return a * b;
#endif
}

SK_HD double sk_div(double a, double b)
{
#ifdef __CUDA_ARCH__
	return __ddiv_rn(a, b);
#else
	return a / b;
#endif
}

SK_HD double sk_add(double a, double b)
{
#ifdef __CUDA_ARCH__
	return __dadd_rn(a, b);
#else
	return a + b;
#endif
}

/* the SK estimator of one bin: S1 (>= 0), S2 = (s2_hi:s2_lo), M FFT blocks */
SK_HD double sk_from_moments(long long S1, unsigned long long s2_lo, unsigned long long s2_hi, long long M)
{
	if (M < 2 || S1 == 0)
		return NAN;
	const double s1 = sk_u64_to_double((unsigned long long)S1), s2 = sk_u128_to_double(s2_lo, s2_hi);
	const double a = sk_mul((double)M, s2), b = sk_mul(s1, s1);
	const double c = sk_div(a, b), d = sk_add(c, -1.0);
	const double e = sk_div((double)(M + 1), (double)(M - 1));
	return sk_mul(e, d);
}

SK_HD double sk_sqrt(double a)
{
#ifdef __CUDA_ARCH__
	return __dsqrt_rn(a);
#else
	return sqrt(a);
#endif
}

/* the standard deviation of the estimator over M blocks of single-block power (Nita & Gary 2010, N = d = 1):
 *   sigma = sqrt(4 M^2 / ((M-1)(M+2)(M+3))), quiet NaN when M < 2,
 * as m = rn(M); a = (4*m)*m; b = ((m-1)*(m+2))*(m+3); sigma = sqrt(a/b), every step correctly rounded */
SK_HD double sk_sigma(long long M)
{
	if (M < 2)
		return NAN;
	const double m = (double)M;
	const double a = sk_mul(sk_mul(4.0, m), m);
	const double b = sk_mul(sk_mul(sk_add(m, -1.0), sk_add(m, 2.0)), sk_add(m, 3.0));
	return sk_sqrt(sk_div(a, b));
}

/* ---- device accumulation ------------------------------------------------ */

/* pw^2 into a register partial (lo, carry count): exact over up to 2^32 additions */
SCAN_DEV void sk_accumulate(unsigned long long &lo, unsigned &hi, unsigned pw)
{
	const unsigned long long p2 = (unsigned long long)pw * pw;
	lo += p2;
	hi += lo < p2 ? 1u : 0u;
}

/* (hi:lo) into the 128-bit word pair at p (global or shared memory) */
SCAN_DEV void sk_atomic_add(unsigned long long *p, unsigned long long lo, unsigned long long hi)
{
	const unsigned long long old = atomicAdd(p, lo);
	hi += old + lo < old ? 1ull : 0ull;
	if (hi)
		atomicAdd(p + 1, hi);
}

/* The SK row of every hop of a report, in the dB row's layout (rtl_power.c:732-760): bin 0 takes bin 1's moments
 * (csv_dbm's DC nuke), then the half swap, the crop [i1, i2] and the duplicate of bin i2.  M = samples / ds
 * (rtl_power.c:717 adds ds per FFT block).  Reads S1 and the sample counters, so it runs on the handle's stream in
 * front of the report epilogue that zeroes them. */
struct SkReportParams {
	const long long *avg;               /* [hops << bin_e] S1, natural order */
	const long long *samples;           /* [hops] */
	const unsigned long long *s2;       /* [hops << bin_e][2] (lo, hi) */
	double *sk;                         /* [hops][db_count], indexed from hop0 */
	int bin_e;
	int i1, i2;
	int downsample;
	int hop0;
};

__global__ void __launch_bounds__(256)
sk_report_kernel(const SCAN_GRID_CONSTANT SkReportParams prm)
{
	const int hop = prm.hop0 + blockIdx.y;
	const int n = 1 << prm.bin_e;
	const int count = prm.i2 - prm.i1 + 2;
	const int k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= count)
		return;
	const int i = (k < count - 1) ? prm.i1 + k : prm.i2;
	int j = (i + n / 2) & (n - 1); /* undo the half swap */
	if (j == 0)
		j = 1;                     /* avg[0] = avg[1] */
	const long long b = ((long long)hop << prm.bin_e) + j;
	prm.sk[(long long)blockIdx.y * count + k] =
		sk_from_moments(prm.avg[b], prm.s2[2 * b], prm.s2[2 * b + 1], prm.samples[hop] / prm.downsample);
}

/* Reads of the same hops on several SK handles (rtlsdr_gpu_scan_merge_sk_device): `sets` external sets -- S1 int64
 * [bins], int32 counts [hops] and S2 (lo, hi) u64 [bins][2] at ext_* + s * stride -- are added into this handle's
 * accumulators.  S2 is added as an unsigned 128-bit value (a wrap of the low word carries into the high word), so the
 * merged sums do not depend on how the reads were grouped.  No peak hold on an SK handle. */
struct MergeSkParams {
	long long *avg;                     /* [bins] */
	long long *samples;                 /* [hops] */
	unsigned long long *s2;             /* [bins][2] */
	const uint8_t *ext_avg;
	const uint8_t *ext_smp;
	const uint8_t *ext_s2;
	long long stride;
	long long bins;
	int hops;
	int sets;
};

__global__ void __launch_bounds__(256)
merge_sk_sets_kernel(const SCAN_GRID_CONSTANT MergeSkParams prm)
{
	const long long step = (long long)gridDim.x * blockDim.x;
	const long long first = (long long)blockIdx.x * blockDim.x + threadIdx.x;
	for (long long i = first; i < prm.bins; i += step) {
		long long v = prm.avg[i];
		unsigned long long lo = prm.s2[2 * i], hi = prm.s2[2 * i + 1];
		for (int s = 0; s < prm.sets; ++s) {
			v += ((const long long *)(prm.ext_avg + s * prm.stride))[i];
			const unsigned long long *e = (const unsigned long long *)(prm.ext_s2 + s * prm.stride) + 2 * i;
			const unsigned long long el = e[0];
			lo += el;
			hi += e[1] + (lo < el ? 1ull : 0ull);
		}
		prm.avg[i] = v;
		prm.s2[2 * i] = lo;
		prm.s2[2 * i + 1] = hi;
	}
	for (long long i = first; i < prm.hops; i += step) {
		long long v = prm.samples[i];
		for (int s = 0; s < prm.sets; ++s)
			v += ((const int *)(prm.ext_smp + s * prm.stride))[i];
		prm.samples[i] = v;
	}
}

} // namespace rscan
