/* scan_host.cuh -- host arithmetic of a scan, no CUDA calls: config checks, read geometry and the constant
 * tables the kernels read.  rtlsdr_gpu_scan_init() and the CPU emulator (tests/emu) both build them here. */
#pragma once
#include "../../include/rtlsdr_gpu_scan.h"
#include "scan_kernels.cuh"

#include <algorithm>
#include <vector>

namespace rscan {

enum Path { PATH_RMS, PATH_SMALL_U8, PATH_SMALL_DECIM, PATH_LARGE };

struct ScanShape {
	Path path = PATH_SMALL_U8;
	int N = 1;
	int l_len = 0, n_blocks = 0, blocks_padded = 0, samples_per_read = 0;
	long long image_stride = 0; /* c16 per decimated image */
	int db_i1 = 0, db_i2 = 0, db_count = 2;
};

/* 0, or RTLSDR_GPU_ERR_CONFIG for a configuration the library does not run */
inline int scan_shape(const rtlsdr_gpu_scan_cfg_t &cfg, ScanShape *out)
{
	if (!(cfg.iir_alpha >= 0.0 && cfg.iir_alpha <= 1.0))
		return RTLSDR_GPU_ERR_CONFIG;
	if (cfg.tune_count <= 0 || cfg.tune_count > 3000 /* MAX_TUNES, rtl_power.c:113 */ ||
	    cfg.bin_e < 0 || cfg.bin_e > 21 /* rtl_power.c:483 */ || cfg.downsample < 1 ||
	    cfg.downsample_passes < 0 || cfg.downsample_passes > 20 || cfg.buf_len < 16 ||
	    (cfg.buf_len & 15) || cfg.rate <= 0 || !(cfg.crop >= 0.0 && cfg.crop <= 1.0))
		return RTLSDR_GPU_ERR_CONFIG;
	const int N = 1 << cfg.bin_e;
	const bool box = cfg.boxcar && cfg.downsample > 1;
	const bool hb = !box && cfg.downsample_passes > 0;
	if (hb && cfg.downsample != (1 << cfg.downsample_passes))
		return RTLSDR_GPU_ERR_CONFIG;
	if (hb && ((cfg.buf_len >> cfg.downsample_passes) < 24 || (cfg.buf_len & ((4 << cfg.downsample_passes) - 1))))
		return RTLSDR_GPU_ERR_CONFIG;
	if (!box && !hb && cfg.downsample != 1 && cfg.bin_e > 0) {
		/* ds > 1 without a decimator: the reference would still divide lengths by ds
		 * (rtl_power.c:692-695); the planner never produces this, reject it */
		return RTLSDR_GPU_ERR_CONFIG;
	}

	ScanShape s;
	s.N = N;
	/* geometry of one read (rtl_power.c:692-695, 717) */
	if (cfg.bin_e == 0) {
		s.path = PATH_RMS;
		s.samples_per_read = 1;
	} else {
		s.l_len = cfg.buf_len / cfg.downsample;
		s.n_blocks = (s.l_len + 2 * N - 1) / (2 * N);
		s.samples_per_read = s.n_blocks * cfg.downsample;
		if (cfg.bin_e <= 12) {
			if (!box && !hb) {
				if (cfg.buf_len != kStageBytes)
					return RTLSDR_GPU_ERR_CONFIG; /* planner gives 16384 whenever 2N <= 16384 (rtl_power.c:501-504) */
				s.path = PATH_SMALL_U8;
			} else {
				s.path = PATH_SMALL_DECIM;
				/* images of consecutive reads are contiguous; keep each 16-byte aligned */
				s.blocks_padded = s.n_blocks;
				while (((long long)s.blocks_padded * N) % 4)
					s.blocks_padded++;
				s.image_stride = (long long)s.blocks_padded * N;
			}
		} else {
			s.path = PATH_LARGE;
			if (s.n_blocks != 1 || (box || hb ? s.l_len != 2 * N : cfg.buf_len != 2 * N))
				return RTLSDR_GPU_ERR_CONFIG; /* 2N*ds >= 16384 always holds here, so one block per read */
			s.image_stride = N;
		}
	}
	/* what csv_dbm prints (rtl_power.c:741-748) */
	s.db_i1 = 0 + (int)((double)N * cfg.crop * 0.5);
	s.db_i2 = (N - 1) - (int)((double)N * cfg.crop * 0.5);
	if (s.db_i2 < s.db_i1)
		return RTLSDR_GPU_ERR_CONFIG;
	s.db_count = s.db_i2 - s.db_i1 + 2;
	*out = s;
	return 0;
}

/* twiddles of a 2^L transform: wr = Sinewave[j+N/4] >> 1, wi = (-Sinewave[j]) >> 1 (rtl_power.c:305-308).  The kernels
 * special-case the angle-0 and quarter-turn groups of the first four stages: (wr, 0) and (0, wi).  True for every table
 * sine_table() builds (Sinewave[0] = Sinewave[N/2] = 0); RTLSDR_GPU_ERR_CONFIG for a table where it is not. */
inline int twiddles(const int16_t *sine, int L, std::vector<int2> &tw)
{
	const int N = 1 << L, half = std::max(N / 2, 1);
	tw.resize(half);
	for (int j = 0; j < half; j++)
		tw[j] = make_int2((int16_t)(sine[j + N / 4] >> 1), (int16_t)((int16_t)(-sine[j]) >> 1));
	return tw[0].y != 0 || (N >= 4 && tw[N / 4].x != 0) ? RTLSDR_GPU_ERR_CONFIG : 0;
}

/* the first four stages' twiddles: stage b, group g at w[(1<<b)-1+g] */
inline PassTw first_stage_tw(const std::vector<int2> &tw, int L)
{
	PassTw tw0 = {};
	for (int b = 0; b < 4 && b < L; b++)
		for (int g = 0; g < (1 << b); g++)
			tw0.w[(1 << b) - 1 + g] = tw[(size_t)g << (L - 1 - b)];
	return tw0;
}

/* compact table of stages 4..s_end-1: stage s, group m at (1<<s)-16+m = tw[m << (L-1-s)].  The small path
 * takes s_end = L (empty for N <= 16), the large path's round A s_end = 8. */
inline std::vector<int2> compact_tw(const std::vector<int2> &tw, int L, int s_end)
{
	std::vector<int2> twc(s_end > 4 ? (size_t)(1 << s_end) - 16 : 0);
	for (int st = 4; st < s_end; st++)
		for (int m = 0; m < (1 << st); m++)
			twc[(size_t)(1 << st) - 16 + m] = tw[(size_t)m << (L - 1 - st)];
	return twc;
}

/* large path, round B: twb[se][plow][ilow] = tw[((ilow << 8) | plow) << (L-9-se)], se = 4 .. min(8, L-8)-1 */
inline std::vector<int2> round_b_tw(const std::vector<int2> &tw, int L)
{
	const int lb = std::min(8, L - 8);
	std::vector<int2> twb((size_t)256 * 240, make_int2(0, 0));
	for (int se = 4; se < lb; se++)
		for (int plow = 0; plow < 256; plow++)
			for (int ilow = 0; ilow < (1 << se); ilow++)
				twb[(size_t)256 * ((1 << se) - 16) + ((size_t)plow << se) + ilow] =
					tw[((size_t)((ilow << 8) | plow)) << (L - 9 - se)];
	return twb;
}

/* the window as the kernels read it: the low 16 bits of window_coefs[N] (rectangle without one) */
inline std::vector<uint16_t> window16(const int32_t *coefs, int N)
{
	std::vector<uint16_t> win(N);
	for (int i = 0; i < N; i++)
		win[i] = (uint16_t)((coefs ? coefs[i] : 256) & 0xFFFF);
	return win;
}

/* Sets p.tile and p.cap0 of a -F chain of p.passes levels and returns the kernel's dynamic shared memory.
 * stream: the register-streaming kernel computes final samples >= 16 and the tile kernel only the
 * eased-in head [0, 16) of every read. */
inline int chain_tile(HalfbandChainParams &p, bool stream)
{
	if (stream) {
		/* head tiles span (16 + 9) * 2^P + 5 * (2^P - 1) + 9 <= 964 level-0 samples: small buffers, many CTAs per SM */
		p.tile = kHbStreamHead;
		p.cap0 = 1024;
	} else {
		p.cap0 = 8192; /* level-0 samples a tile may span (32 KiB) */
		/* level-0 span of a tile: (tile + 9) * 2^P + 5 * (2^P - 1) + 9 samples at most */
		p.tile = std::min(p.pairs >> p.passes, std::min(256, std::max(8, (p.cap0 >> p.passes) - 16)));
	}
	return (p.cap0 + p.cap0 / 2 + 16) * 4;
}

} // namespace rscan
