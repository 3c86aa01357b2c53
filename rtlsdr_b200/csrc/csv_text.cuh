/*
 * csv_text.cuh -- rtl_power's CSV rows formatted on the GPU, byte-identical to
 * the host's printf (rtl_power.c:739-760, 995-998; host/rtl_power_plan.c
 * rp_csv_row):  "<stamp>low, high, step, samples, dB, ..., dB\n".
 *
 * %.2f is exact 64-bit integer arithmetic on the double's bits, no floating
 * point and no tables.  |v| = M * 2^E:
 *   E >= 0:  Q = (M << E) * 100
 *   E <  0:  k = -E, N = 100 * M, Q = N >> k, rounded half to even against
 *            2^(k-1) with the remainder N mod 2^k (glibc's rounding in the
 *            default mode); k > 62 means |v| * 100 < 2^-3, Q = 0
 * then Q / 100 "." Q % 100 in two digits, '-' whenever the sign bit is set
 * (glibc prints -0.00), and inf / nan with the sign bit.  Domain: finite
 * |v| < 2^53 (so N < 2^60), plus inf and NaN.
 *
 * A report's finite dB values are 10*log10 of an int64 bin over an int32 rate
 * and an int32 count, within (-187, 190); the -s iir values are convex
 * combinations of those.  A row therefore only accepts dB text of at most 7
 * characters ("-999.99"), which bounds a row by stamp_len + kCsvRowFixed +
 * kCsvValueMax * db_count bytes; anything wider can only come from a caller's
 * own buffer and is reported as an error instead of printed.
 *
 * %.4f (the spectral-kurtosis rows) needs M * 10^4, which does not fit 64 bits: with k = -E the integer part is
 * M >> k, and the fraction F = M mod 2^k gives the four decimals D = F * 10^4 >> k, computed exactly in 128 bits
 * (__umul64hi on the device, unsigned __int128 in the emulator build) and rounded half to even against the
 * remainder like %.2f (Q = integer * 10^4 + D has D's parity); a carry to D = 10^4 moves into the integer part.
 * k > 67 means |v| * 10^4 < 2^-1, D = 0.  Sign bit kept (-0.0000), inf with the sign, and every NaN prints "nan"
 * (the SK rows' format, not glibc's "-nan").  Domain: finite |v| < 2^53, plus inf and NaN.  An SK value is at
 * most M + 1 < 2^31 + 1 (Cauchy-Schwarz: M * S2 >= S1^2), so an SK row accepts value text of at most 15
 * characters ("2147483649.0000") and is bounded like a dB row with kCsvSkValueMax per value.
 *
 * Three kernels: csv_rows_kernel (dB) or csv_sk_rows_kernel (SK) formats row r into slot r of a scratch area
 * (one CTA per row, a block-wide scan places the variable-width values), then
 * csv_pack_kernel moves every slot to its place in the contiguous text (each
 * CTA sums the lengths of the rows before it) and the last CTA stores the
 * total length, or -1 if any row held a value outside the domain.
 */
#pragma once
#include "scan_compat.cuh"

#ifdef SCAN_EMU
#include <cstring>
#endif

namespace rscan {

constexpr int kCsvStampMax = 128; /* stamp bytes carried in the kernel parameters (length < this) */
constexpr int kCsvRowFixed = 56;  /* "low, high, step, samples, " at their widest (54) and the newline, rounded up */
constexpr int kCsvValueMax = 9;   /* "-999.99, " */
constexpr int kCsvSkValueMax = 17; /* "2147483649.0000, ": SK <= M + 1 (Cauchy-Schwarz) and M < 2^31 */
constexpr int kCsvThreads = 256;
constexpr double kCsvStepLimit = 2147483648.0; /* step column: 0 <= step < 2^31 */

SCAN_DEV unsigned long long csv_bits(double v)
{
#ifdef SCAN_EMU
	unsigned long long b;
	memcpy(&b, &v, sizeof(b));
	return b;
#else
	return (unsigned long long)__double_as_longlong(v);
#endif
}

/* decimal digits of u (< 10^19) written backwards from `end`; returns the new start */
SCAN_DEV char *csv_digits_rev(unsigned long long u, char *end)
{
	do {
		*--end = (char)('0' + (int)(u % 10));
		u /= 10;
	} while (u);
	return end;
}

/* printf("%i", v) into out (at most 11 bytes); returns the length */
SCAN_DEV int csv_fmt_i(int v, char *out)
{
	char tmp[12];
	char *e = tmp + sizeof(tmp);
	const unsigned long long u = v < 0 ? (unsigned long long)(-(long long)v) : (unsigned long long)v;
	char *s = csv_digits_rev(u, e);
	if (v < 0)
		*--s = '-';
	const int n = (int)(e - s);
	for (int i = 0; i < n; i++)
		out[i] = s[i];
	return n;
}

/* printf("%.2f", v) into out (at most 20 bytes); returns the length, or -1 for a finite |v| >= 2^53 */
SCAN_DEV int csv_fmt_f2(double v, char *out)
{
	const unsigned long long b = csv_bits(v);
	const int neg = (int)(b >> 63), e = (int)((b >> 52) & 0x7FF);
	const unsigned long long frac = b & ((1ull << 52) - 1);
	int n = 0;
	if (neg)
		out[n++] = '-';
	if (e == 0x7FF) {
		out[n++] = frac ? 'n' : 'i';
		out[n++] = frac ? 'a' : 'n';
		out[n++] = frac ? 'n' : 'f';
		return n;
	}
	const unsigned long long M = e ? (frac | (1ull << 52)) : frac;
	const int E = (e ? e : 1) - 1075;
	unsigned long long Q;
	if (E >= 0) {
		if (E > 0) /* |v| >= 2^53 */
			return -1;
		Q = M * 100;
	} else if (-E > 62) {
		Q = 0;
	} else {
		const int k = -E;
		const unsigned long long N = M * 100;
		const unsigned long long r = N & ((1ull << k) - 1), half = 1ull << (k - 1);
		Q = N >> k;
		if (r > half || (r == half && (Q & 1)))
			Q++;
	}
	char tmp[20];
	char *end = tmp + sizeof(tmp);
	*--end = (char)('0' + (int)(Q % 10));
	*--end = (char)('0' + (int)(Q / 10 % 10));
	*--end = '.';
	char *s = csv_digits_rev(Q / 100, end);
	for (char *p = s; p < tmp + sizeof(tmp); p++)
		out[n++] = *p;
	return n;
}

/* the high word of the 128-bit product a * b */
SCAN_DEV unsigned long long csv_mul_hi(unsigned long long a, unsigned long long b)
{
#ifdef SCAN_EMU
	return (unsigned long long)(((unsigned __int128)a * b) >> 64);
#else
	return __umul64hi(a, b);
#endif
}

/* printf("%.4f", v) into out (at most 22 bytes), except that a NaN of either sign prints "nan"; returns the length,
 * or -1 for a finite |v| >= 2^53 */
SCAN_DEV int csv_fmt_f4(double v, char *out)
{
	const unsigned long long b = csv_bits(v);
	const int neg = (int)(b >> 63), e = (int)((b >> 52) & 0x7FF);
	const unsigned long long frac = b & ((1ull << 52) - 1);
	int n = 0;
	if (e == 0x7FF && frac) {
		out[0] = 'n';
		out[1] = 'a';
		out[2] = 'n';
		return 3;
	}
	if (neg)
		out[n++] = '-';
	if (e == 0x7FF) {
		out[n++] = 'i';
		out[n++] = 'n';
		out[n++] = 'f';
		return n;
	}
	const unsigned long long M = e ? (frac | (1ull << 52)) : frac;
	const int E = (e ? e : 1) - 1075;
	unsigned long long I = 0, D = 0; /* integer part, four decimals */
	if (E > 0) {                     /* |v| >= 2^53 */
		return -1;
	} else if (E == 0) {
		I = M;
	} else if (-E <= 67) {           /* else |v| * 10^4 < 2^66 / 2^68: rounds to 0 */
		const int k = -E;
		I = k < 64 ? M >> k : 0;
		const unsigned long long F = k < 64 ? M & ((1ull << k) - 1) : M;
		/* (nh:nl) = F * 10^4 < 2^67; D = that >> k, rounded half to even against the remainder (rh:rl) */
		const unsigned long long nl = F * 10000ull, nh = csv_mul_hi(F, 10000ull);
		unsigned long long rl, rh, hl, hh;
		if (k < 64) {
			D = (nl >> k) | (nh << (64 - k));
			rl = nl & ((1ull << k) - 1);
			rh = 0;
			hl = 1ull << (k - 1);
			hh = 0;
		} else {
			D = nh >> (k - 64);
			rl = nl;
			rh = nh & ((1ull << (k - 64)) - 1);
			hl = k == 64 ? 1ull << 63 : 0ull;
			hh = k == 64 ? 0ull : 1ull << (k - 65);
		}
		const bool above = rh > hh || (rh == hh && rl > hl), tie = rh == hh && rl == hl;
		if (above || (tie && (D & 1)))
			D++;
		if (D == 10000) {
			I++;
			D = 0;
		}
	}
	char tmp[24];
	char *end = tmp + sizeof(tmp);
	for (int i = 0; i < 4; i++) {
		*--end = (char)('0' + (int)(D % 10));
		D /= 10;
	}
	*--end = '.';
	char *s = csv_digits_rev(I, end);
	for (char *p = s; p < tmp + sizeof(tmp); p++)
		out[n++] = *p;
	return n;
}

struct CsvRowParams {
	const double *db;      /* row r's values at db + r * db_stride */
	long long db_stride;   /* doubles */
	const int *samples;    /* [rows] */
	const int2 *cols;      /* [table rows] (low, high); row r uses cols[row_first + r] */
	double step;
	int row_first;
	int db_count;
	char *slots;           /* row r at slots + r * slot_bytes */
	long long slot_bytes;
	int *lens;             /* [rows]: bytes of row r, -1 if a value is outside the domain */
	int stamp_len;
	char stamp[kCsvStampMax];
};

/* one CTA per row; kCsvThreads threads */
__global__ void __launch_bounds__(kCsvThreads)
csv_rows_kernel(const SCAN_GRID_CONSTANT CsvRowParams prm)
{
#define CSV_FMT_VALUE(v, out) csv_fmt_f2(v, out)
#define CSV_VALUE_WIDTH (kCsvValueMax - 2)
#include "csv_rows_body.inl"
#undef CSV_FMT_VALUE
#undef CSV_VALUE_WIDTH
}

/* the SK rows: the same prefix, prm.db holds SK values printed as %.4f ("nan" for any NaN) */
__global__ void __launch_bounds__(kCsvThreads)
csv_sk_rows_kernel(const SCAN_GRID_CONSTANT CsvRowParams prm)
{
#define CSV_FMT_VALUE(v, out) csv_fmt_f4(v, out)
#define CSV_VALUE_WIDTH (kCsvSkValueMax - 2)
#include "csv_rows_body.inl"
#undef CSV_FMT_VALUE
#undef CSV_VALUE_WIDTH
}

struct CsvPackParams {
	const char *slots;
	long long slot_bytes;
	const int *lens;
	char *text;
	long long *len;        /* total bytes, or -1 */
};

/* one CTA per row: offset = the lengths of the rows before it */
__global__ void __launch_bounds__(kCsvThreads)
csv_pack_kernel(const SCAN_GRID_CONSTANT CsvPackParams prm)
{
	__shared__ long long part[kCsvThreads];
	__shared__ int bad[kCsvThreads];
	const int row = blockIdx.x, t = threadIdx.x;
	long long s = 0;
	int b = 0;
	for (int i = t; i <= row; i += kCsvThreads) {
		const int n = prm.lens[i];
		b |= n < 0;
		if (i < row)
			s += n;
	}
	part[t] = s;
	bad[t] = b;
	__syncthreads();
	for (int d = kCsvThreads / 2; d > 0; d >>= 1) {
		if (t < d) {
			part[t] += part[t + d];
			bad[t] |= bad[t + d];
		}
		__syncthreads();
	}
	const long long off = part[0];
	const int n = prm.lens[row];
	if (bad[0]) {
		if (row == (int)gridDim.x - 1 && t == 0)
			*prm.len = -1;
		return;
	}
	const char *src = prm.slots + (long long)row * prm.slot_bytes;
	for (int i = t; i < n; i += kCsvThreads)
		prm.text[off + i] = src[i];
	if (row == (int)gridDim.x - 1 && t == 0)
		*prm.len = off + n;
}

} // namespace rscan
