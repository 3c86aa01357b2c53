/*
 * TEST INFRASTRUCTURE ONLY -- the spectral-kurtosis moment of the C oracle: oracle_scan_read (oracle/scan_oracle.c)
 * plus the unsigned 128-bit sum of p^2, p = re^2 + im^2 being what avg[bin] adds per FFT block.  Includes the
 * oracle's source for its static helpers (wrap16, boxcar_decimate); the oracle itself is not changed.  Built by
 * tests/test_sk.py with the oracle's flags:
 *   gcc -O3 -DNDEBUG -fwrapv -fPIC -shared -Ioracle
 */
#include "scan_oracle.c"

/* s2[2 * bin] (lo), s2[2 * bin + 1] (hi); sums only (no peak hold), bin_e >= 1 */
void oracle_scan_read_sk(const oracle_cfg_t *cfg, const uint8_t *buf8, int16_t *work,
			 int64_t *avg, int *samples, uint64_t *s2)
{
	int n = 1 << cfg->bin_e, ds = cfg->downsample, ds_p = cfg->downsample_passes;
	int buf_len = cfg->buf_len, len, offset, j;

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
	for (offset = 0; offset < len; offset += 2 * n) {
		int16_t *blk = work + offset;
		for (j = 0; j < n; j++) {
			blk[2 * j] = wrap16((int32_t)blk[2 * j] * cfg->window[j]);
			blk[2 * j + 1] = wrap16((int32_t)blk[2 * j + 1] * cfg->window[j]);
		}
		oracle_fix_fft(blk, cfg->bin_e, cfg->sine, cfg->bin_e);
		for (j = 0; j < n; j++) {
			int64_t re = blk[2 * j], im = blk[2 * j + 1];
			uint64_t p = (uint64_t)(re * re + im * im);
			unsigned __int128 acc = ((unsigned __int128)s2[2 * j + 1] << 64) | s2[2 * j];
			acc += (unsigned __int128)(p * p);
			avg[j] += (int64_t)p;
			s2[2 * j] = (uint64_t)acc;
			s2[2 * j + 1] = (uint64_t)(acc >> 64);
		}
		*samples += ds;
	}
}
