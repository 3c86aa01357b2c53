/*
 * TEST INFRASTRUCTURE ONLY -- the guard-bit transform of RTLSDR_GPU_FLAG_GUARD_BITS (include/rtlsdr_gpu_scan.h) in
 * plain C: fix_fft (oracle/scan_oracle.c, rtl_power.c:271-327) with its data carried in int32 with F = 8 fractional
 * bits, the per-read scan around it (the oracle's front end unchanged) with S2 in unsigned __int128, and the dB
 * epilogue with the exact 2^-8 scale.  Includes the oracle's source for its static helpers (wrap16, bit_reverse,
 * boxcar_decimate); the oracle itself is not changed.  Built by tests/test_guard.py with the oracle's flags:
 *   gcc -O3 -fwrapv -fPIC -shared -Ioracle
 */
#include "scan_oracle.c"

#include <assert.h>

#define GUARD_F 8
#define GUARD_BOUND (1 << 24)

/* R(p) = (p + 2^14) >> 15 on the exact product (arithmetic shift) */
static int32_t guard_mpy(int32_t w, int32_t b)
{
	return (int32_t)(((int64_t)w * b + 16384) >> 15);
}

static void guard_check(int32_t v)
{
	/* |v| < 2^15 * sqrt(2) * 2^F plus one unit per stage < 2^24: int32 never wraps */
	assert(v > -GUARD_BOUND && v < GUARD_BOUND);
	(void)v;
}

/* fix_fft on v[2n] (re, im) int32, same permutation, twiddles, halving and rounding as oracle_fix_fft */
int oracle_fix_fft_guard(int32_t *v, int m, const int16_t *sine, int log2_nwave)
{
	int n = 1 << m, nwave = 1 << log2_nwave;
	int s, g, i;
	if (n > nwave)
		return -1;
	for (i = 1; i < n; i++) {
		int r = (int)bit_reverse((unsigned)i, m);
		if (r > i) {
			int32_t tr = v[2 * i], ti = v[2 * i + 1];
			v[2 * i] = v[2 * r];
			v[2 * i + 1] = v[2 * r + 1];
			v[2 * r] = tr;
			v[2 * r + 1] = ti;
		}
	}
	for (s = 0; s < m; s++) {
		int half = 1 << s, span = half << 1;
		int k = log2_nwave - 1 - s;
		for (g = 0; g < half; g++) {
			int j = g << k;
			int32_t wr = (int16_t)(sine[j + nwave / 4] >> 1);
			int32_t wi = (int16_t)(wrap16(-(int32_t)sine[j]) >> 1);
			for (i = g; i < n; i += span) {
				int p = i + half;
				int32_t br = v[2 * p], bi = v[2 * p + 1];
				int32_t tr = guard_mpy(wr, br) - guard_mpy(wi, bi);
				int32_t ti = guard_mpy(wr, bi) + guard_mpy(wi, br);
				int32_t qr = v[2 * i] >> 1, qi = v[2 * i + 1] >> 1;
				v[2 * p] = qr - tr;
				v[2 * p + 1] = qi - ti;
				v[2 * i] = qr + tr;
				v[2 * i + 1] = qi + ti;
				guard_check(v[2 * p]);
				guard_check(v[2 * p + 1]);
				guard_check(v[2 * i]);
				guard_check(v[2 * i + 1]);
			}
		}
	}
	return 0;
}

/* the front end of oracle_scan_read: work[buf_len] int16 before the window, returns len */
static int guard_front(const oracle_cfg_t *cfg, const uint8_t *buf8, int16_t *work)
{
	int ds = cfg->downsample, ds_p = cfg->downsample_passes, buf_len = cfg->buf_len, len, j;
	for (j = 0; j < buf_len; j++)
		work[j] = (int16_t)((int)buf8[j] - 127);
	if (cfg->boxcar && ds > 1) {
		boxcar_decimate(work, buf_len, ds);
	} else if (ds_p) {
		for (j = 0; j < ds_p; j++) {
			oracle_fifth_order(work, buf_len >> j);
			oracle_fifth_order(work + 1, (buf_len >> j) - 1);
		}
		if (cfg->comp_fir_size == 9 && ds_p <= 10) {
			oracle_generic_fir(work, buf_len >> ds_p, oracle_cic9(ds_p));
			oracle_generic_fir(work + 1, (buf_len >> ds_p) - 1, oracle_cic9(ds_p));
		}
	}
	len = buf_len / ds;
	oracle_remove_dc(work, len);
	oracle_remove_dc(work + 1, len - 1);
	return len;
}

/*
 * oracle_scan_read with the guard transform: avg[j] += pw (or the maximum under peak_hold), pw = (re^2 + im^2 + 2^7)
 * >> 8, samples += ds per block; s2 (may be NULL) [2 * bin] (lo, hi) += pw^2 in unsigned __int128.  `work` holds
 * buf_len int16, `v` 2N int32.  bin_e >= 1.
 */
void oracle_scan_read_guard(const oracle_cfg_t *cfg, const uint8_t *buf8, int16_t *work, int32_t *v, int64_t *avg,
			    int *samples, uint64_t *s2)
{
	int n = 1 << cfg->bin_e, len, offset, j;
	len = guard_front(cfg, buf8, work);
	for (offset = 0; offset < len; offset += 2 * n) {
		int16_t *blk = work + offset;
		for (j = 0; j < n; j++) {
			v[2 * j] = (int32_t)wrap16((int32_t)blk[2 * j] * cfg->window[j]) * (1 << GUARD_F);
			v[2 * j + 1] = (int32_t)wrap16((int32_t)blk[2 * j + 1] * cfg->window[j]) * (1 << GUARD_F);
		}
		oracle_fix_fft_guard(v, cfg->bin_e, cfg->sine, cfg->bin_e);
		for (j = 0; j < n; j++) {
			int64_t re = v[2 * j], im = v[2 * j + 1];
			uint64_t pw = ((uint64_t)(re * re + im * im) + (1u << (GUARD_F - 1))) >> GUARD_F;
			assert(pw < (1ull << 40));
			if (!cfg->peak_hold)
				avg[j] += (int64_t)pw;
			else if ((int64_t)pw > avg[j])
				avg[j] = (int64_t)pw;
			if (s2) {
				unsigned __int128 acc = ((unsigned __int128)s2[2 * j + 1] << 64) | s2[2 * j];
				acc += (unsigned __int128)pw * pw;
				s2[2 * j] = (uint64_t)acc;
				s2[2 * j + 1] = (uint64_t)(acc >> 64);
			}
		}
		*samples += cfg->downsample;
	}
}

/* the int16 front-end output of one read (for the float64 DFT reference): windowed blocks, returns the block count */
int oracle_guard_front_blocks(const oracle_cfg_t *cfg, const uint8_t *buf8, int16_t *work, int16_t *out)
{
	int n = 1 << cfg->bin_e, len = guard_front(cfg, buf8, work), offset, j, b = 0;
	for (offset = 0; offset < len; offset += 2 * n, b++)
		for (j = 0; j < 2 * n; j++)
			out[(size_t)b * 2 * n + j] = wrap16((int32_t)work[offset + j] * cfg->window[j >> 1]);
	return b;
}

/* oracle_epilogue for guard bins: v = (double)avg * 2^-8 (exact), then the reference's chain */
int oracle_epilogue_guard(int64_t *avg, int bin_e, double crop, int rate, int samples, double *db)
{
	int len = 1 << bin_e, i, i1, i2, k = 0;
	double v;
	avg[0] = avg[1];
	for (i = 0; i < len / 2; i++) {
		int64_t t = avg[i];
		avg[i] = avg[i + len / 2];
		avg[i + len / 2] = t;
	}
	i1 = 0 + (int)((double)len * crop * 0.5);
	i2 = (len - 1) - (int)((double)len * crop * 0.5);
	for (i = i1; i <= i2; i++) {
		v = (double)avg[i];
		v *= 0x1p-8;
		v /= (double)rate;
		v /= (double)samples;
		db[k++] = 10 * log10(v);
	}
	v = (double)avg[i2] * 0x1p-8 / ((double)rate * (double)samples);
	db[k++] = 10 * log10(v);
	return k;
}
