/*
 * TEST INFRASTRUCTURE ONLY -- runs the real kernel source
 * (rtlsdr_b200/csrc/scan_kernels.cuh, scan_large.cuh) on the CPU through
 * cuda_emu.h so that index math / data flow can be parity-checked against the
 * oracle on a box without a GPU.  Built by tests/test_emu_kernels.py with
 *   g++ -std=c++20 -O2 -DSCAN_EMU -Itests/emu -Irtlsdr_b200/csrc -shared -fPIC
 */
#include "scan_host.cuh"
#include "scan_kernels.cuh"
#include "scan_large.cuh"

#include <cstdio>
#include <vector>

using namespace rscan;

namespace {

template <int L, bool PEAK, bool IN16>
void run_small_t(const SmallParams &prm)
{
	/* u8 reads: prm.n_segs carries the grid size (CTAs share the reads in equal runs) */
	cuda_emu::launch(dim3(prm.n_segs), dim3(kThreads), SmallSmem<L>::bytes,
			 [&]() { scan_small_kernel<L, PEAK, IN16>(prm); });
}

template <int L>
void run_small_l(const SmallParams &prm, int peak, int in16)
{
	if (peak)
		in16 ? run_small_t<L, true, true>(prm) : run_small_t<L, true, false>(prm);
	else
		in16 ? run_small_t<L, false, true>(prm) : run_small_t<L, false, false>(prm);
}

void run_small(int L, const SmallParams &prm, int peak, int in16)
{
	switch (L) {
	case 1: run_small_l<1>(prm, peak, in16); break;
	case 2: run_small_l<2>(prm, peak, in16); break;
	case 3: run_small_l<3>(prm, peak, in16); break;
	case 4: run_small_l<4>(prm, peak, in16); break;
	case 5: run_small_l<5>(prm, peak, in16); break;
	case 6: run_small_l<6>(prm, peak, in16); break;
	case 7: run_small_l<7>(prm, peak, in16); break;
	case 8: run_small_l<8>(prm, peak, in16); break;
	case 9: run_small_l<9>(prm, peak, in16); break;
	case 10: run_small_l<10>(prm, peak, in16); break;
	case 11: run_small_l<11>(prm, peak, in16); break;
	case 12: run_small_l<12>(prm, peak, in16); break;
	default: break;
	}
}

/* the tables rtlsdr_gpu_scan_init() builds (scan_host.cuh), from the oracle's Sinewave[] and window_coefs[] */
struct Tables {
	std::vector<int2> tw, twc;
	std::vector<uint16_t> win;
	PassTw tw0;
	Tables(const int16_t *sine, const int32_t *coefs, int L, int s_end)
	{
		twiddles(sine, L, tw); /* the oracle's sine_table() always passes the check */
		tw0 = first_stage_tw(tw, L);
		twc = compact_tw(tw, L, s_end);
		win = window16(coefs, 1 << L);
	}
};

} // namespace

extern "C" {

/* u8 path: reads [n_reads][16384] sorted by hop, hop_of [n_reads]; `grid` CTAs share the working sets in equal runs */
void emu_small_u8(int L, int peak, const uint8_t *reads, int n_reads, const int *hop_of, int grid,
		  const int16_t *sine, const int32_t *win, long long *avg, long long *samples)
{
	const Tables t(sine, win, L, L);
	std::vector<long long> offs(n_reads);
	for (int i = 0; i < n_reads; i++)
		offs[i] = (long long)i * kStageBytes;
	SmallParams p;
	memset(&p, 0, sizeof(p));
	p.base = reads;
	p.read_off = offs.data();
	p.hop_of = hop_of;
	p.n_entries = n_reads;
	p.n_segs = grid; /* run_small_t launches n_segs CTAs */
	p.avg = avg;
	p.samples = samples;
	p.samples_per_read = kStageBytes / (2 << L); /* FFT blocks per read (ds = 1) */
	p.tw = t.tw.data();
	p.twc = t.twc.data();
	p.win = t.win.data();
	p.tw0 = t.tw0;
	run_small(L, p, peak, 0);
}

/*
 * decimating path: u8 reads [n_reads][buf_len] -> images -> spectra.
 * mode 0 = boxcar(ds), mode 1 = fifth_order x ds_p (+ 9-tap FIR if fir5 != NULL)
 */
static int g_hb_span = 64;
void emu_set_hb_span(int span) { g_hb_span = span; }

void emu_small_decim(int L, int peak, const uint8_t *reads, int n_reads, int buf_len, int ds, int ds_p,
		     int mode, const int *fir5, const int *segs, int n_segs, const int16_t *sine,
		     const int32_t *win, long long *avg, uint32_t *image_out, long long *sums_out)
{
	const rtlsdr_gpu_scan_cfg_t cfg = { .tune_count = 1, .bin_e = L, .buf_len = buf_len, .downsample = ds,
					    .downsample_passes = ds_p, .boxcar = mode == 0, .rate = 1 };
	ScanShape shape;
	if (scan_shape(cfg, &shape))
		return; /* avg stays 0 */
	const Tables t(sine, win, L, L);
	const int pairs = buf_len / 2, l_len = shape.l_len;
	const long long stride = shape.image_stride;
	std::vector<long long> offs(n_reads);
	for (int i = 0; i < n_reads; i++)
		offs[i] = (long long)i * buf_len;
	std::vector<c16> img((size_t)n_reads * stride + kWS, 0xDEADBEEFu); /* padding must not matter */
	std::vector<long long> sums((size_t)n_reads * 2, 0);

	if (mode == 0) {
		DecimParams d;
		d.base = reads;
		d.read_off = offs.data();
		d.n_reads = n_reads;
		d.pairs = pairs;
		d.ds = ds;
		d.out = img.data();
		d.out_stride = stride;
		d.out_count = (int)stride;
		d.l_len = l_len;
		d.sums = sums.data();
		dim3 grid((unsigned)((stride + 255) / 256), n_reads);
		const int bytes = 2 * ds;
		if (ds <= kBoxcarStageMaxDs)
			cuda_emu::launch(grid, dim3(256), 512 * ds, [&]() { boxcar_staged_kernel(d); });
		else if (bytes % 16 == 0)
			cuda_emu::launch(grid, dim3(256), 0, [&]() { boxcar_kernel<16>(d); });
		else if (bytes % 8 == 0)
			cuda_emu::launch(grid, dim3(256), 0, [&]() { boxcar_kernel<8>(d); });
		else if (bytes % 4 == 0)
			cuda_emu::launch(grid, dim3(256), 0, [&]() { boxcar_kernel<4>(d); });
		else
			cuda_emu::launch(grid, dim3(256), 0, [&]() { boxcar_kernel<2>(d); });
	} else if (ds_p <= 7) {
		const int M = pairs >> ds_p;
		HalfbandChainParams hp;
		hp.base = reads;
		hp.read_off = offs.data();
		hp.pairs = pairs;
		hp.passes = ds_p;
		hp.use_fir = fir5 ? 1 : 0;
		hp.f1 = fir5 ? fir5[0] : 0; hp.f2 = fir5 ? fir5[1] : 0; hp.f3 = fir5 ? fir5[2] : 0;
		hp.f4 = fir5 ? fir5[3] : 0; hp.f5 = fir5 ? fir5[4] : 0;
		hp.out = img.data();
		hp.out_stride = stride;
		hp.l_len = l_len;
		hp.sums = sums.data();
		const bool stream = mode == 2 && ds_p <= kHbStreamMaxPasses; /* mode 2: streaming kernel + 16-sample head tiles */
		const int smem = chain_tile(hp, stream);
		cuda_emu::launch(dim3(stream ? 1 : (M + hp.tile - 1) / hp.tile, n_reads), dim3(stream ? 64 : 256), smem,
				 [&]() { halfband_chain_kernel(hp); });
		if (stream) {
			HalfbandStreamParams q;
			q.base = reads;
			q.read_off = offs.data();
			q.n_reads = n_reads;
			q.pairs = pairs;
			q.use_fir = hp.use_fir;
			q.f1 = hp.f1; q.f2 = hp.f2; q.f3 = hp.f3; q.f4 = hp.f4; q.f5 = hp.f5;
			q.out = img.data();
			q.out_stride = stride;
			q.l_len = l_len;
			q.sums = sums.data();
			q.span = g_hb_span;
			const long long threads = (long long)n_reads * ((M + q.span - 1) / q.span);
			const dim3 grid((unsigned)((threads + 127) / 128));
			switch (ds_p) {
			case 1: cuda_emu::launch(grid, dim3(128), 0, [&]() { halfband_stream_kernel<1>(q); }); break;
			case 2: cuda_emu::launch(grid, dim3(128), 0, [&]() { halfband_stream_kernel<2>(q); }); break;
			case 3: cuda_emu::launch(grid, dim3(128), 0, [&]() { halfband_stream_kernel<3>(q); }); break;
			case 4: cuda_emu::launch(grid, dim3(128), 0, [&]() { halfband_stream_kernel<4>(q); }); break;
			default: cuda_emu::launch(grid, dim3(128), 0, [&]() { halfband_stream_kernel<5>(q); }); break;
			}
		}
	} else {
		std::vector<c16> a((size_t)n_reads * (pairs / 2)), b((size_t)n_reads * (pairs / 4 + 4));
		const c16 *cur = nullptr;
		long long cur_stride = 0;
		int count = pairs;
		for (int j = 0; j < ds_p; j++) {
			HalfbandParams hp;
			c16 *dst = (j & 1) ? b.data() : a.data();
			long long dst_stride = (j & 1) ? (pairs / 4 + 4) : (pairs / 2);
			hp.in = j == 0 ? (const void *)reads : (const void *)cur;
			hp.read_off = offs.data();
			hp.in_stride = cur_stride;
			hp.out = dst;
			hp.out_stride = dst_stride;
			hp.n_out = count / 2;
			dim3 grid((hp.n_out + 255) / 256, n_reads);
			if (j == 0)
				cuda_emu::launch(grid, dim3(256), 0, [&]() { halfband_kernel<true>(hp); });
			else
				cuda_emu::launch(grid, dim3(256), 0, [&]() { halfband_kernel<false>(hp); });
			cur = dst;
			cur_stride = dst_stride;
			count /= 2;
		}
		FirParams f;
		f.in = cur;
		f.in_stride = cur_stride;
		f.out = img.data();
		f.out_stride = stride;
		f.count = count;
		f.use_fir = fir5 ? 1 : 0;
		f.f1 = fir5 ? fir5[0] : 0; f.f2 = fir5 ? fir5[1] : 0; f.f3 = fir5 ? fir5[2] : 0;
		f.f4 = fir5 ? fir5[3] : 0; f.f5 = fir5 ? fir5[4] : 0;
		cuda_emu::launch(dim3((count + 255) / 256, n_reads), dim3(256), 0, [&]() { fir9_kernel(f); });
	}
	if (mode != 0 && ds_p > 7) {
		DcSumParams dc;
		dc.img = img.data();
		dc.stride = stride;
		dc.l_len = l_len;
		dc.sums = sums.data();
		cuda_emu::launch(dim3(3, n_reads), dim3(256), 0, [&]() { dc_sums_c16_kernel(dc); });
	}
	if (image_out)
		memcpy(image_out, img.data(), (size_t)n_reads * stride * 4);
	if (sums_out)
		memcpy(sums_out, sums.data(), sums.size() * 8);

	SmallParams p;
	memset(&p, 0, sizeof(p));
	p.base = (const uint8_t *)img.data();
	p.read_off = nullptr;
	p.regular_stride = stride * 4;
	p.entry_base = 0;
	p.segs = (const int4 *)segs;
	p.n_segs = n_segs;
	std::vector<long long> smp(4096, 0);
	p.avg = avg;
	p.samples = smp.data();
	p.samples_per_read = 1;
	p.tw = t.tw.data();
	p.win = t.win.data();
	std::vector<int> ave((size_t)n_reads * 2, 0);
	DcFinalizeParams fz;
	fz.sums = sums.data();
	fz.ave = ave.data();
	fz.n = n_reads;
	fz.l_len = l_len;
	cuda_emu::launch(dim3((2 * n_reads + 255) / 256), dim3(256), 0, [&]() { dc_finalize_kernel(fz); });
	p.dc_ave = ave.data();
	p.l_len = l_len;
	p.n_blocks = shape.n_blocks;
	p.blocks_padded = shape.blocks_padded;
	p.twc = t.twc.data();
	p.tw0 = t.tw0;
	run_small(L, p, peak, 1);
}

static int g_emu_rms_warp = 0;
void emu_set_rms_warp(int v) { g_emu_rms_warp = v; }

void emu_rms(const uint8_t *reads, int n_reads, int buf_len, const int *hop_of, int peak, long long *avg)
{
	std::vector<long long> offs(n_reads);
	for (int i = 0; i < n_reads; i++)
		offs[i] = (long long)i * buf_len;
	RmsParams p;
	p.base = reads;
	p.read_off = offs.data();
	p.hop_of = hop_of;
	p.n_reads = n_reads;
	p.buf_len = buf_len;
	std::vector<long long> smp(4096, 0);
	p.peak = peak;
	p.avg = avg;
	p.samples = smp.data();
	if (buf_len == kRmsCtaBytes && !g_emu_rms_warp)
		cuda_emu::launch(dim3(n_reads > 3 ? 3 : 1), dim3(256), 0, [&]() { rms_cta_kernel(p); });
	else
		cuda_emu::launch(dim3((n_reads + 7) / 8 > 2 ? 2 : 1), dim3(256), 0, [&]() { rms_kernel(p); });
}

void emu_epilogue(const long long *avg, const int *samples, double *db, int bin_e, int i1, int i2, int rate, int hops)
{
	EpilogueParams p;
	memset(&p, 0, sizeof(p));
	std::vector<long long> smp(hops);
	std::vector<long long> avg_copy((size_t)hops << bin_e, -1);
	std::vector<int> smp_copy(hops, -1);
	for (int i = 0; i < hops; i++)
		smp[i] = samples[i];
	p.avg = avg;
	p.samples = smp.data();
	p.db = db;
	p.avg_out = avg_copy.data();
	p.samples_out = smp_copy.data();
	p.bin_e = bin_e;
	p.i1 = i1;
	p.i2 = i2;
	p.rate = rate;
	p.hop0 = 0;
	p.done = nullptr;
	p.avg_rw = nullptr;
	p.samples_rw = nullptr;
	int count = i2 - i1 + 2;
	int span = count > (1 << bin_e) ? count : (1 << bin_e);
	cuda_emu::launch(dim3((span + 255) / 256, hops), dim3(256), 0, [&]() { epilogue_kernel(p); });
	for (size_t i = 0; i < avg_copy.size(); i++)
		if (avg_copy[i] != avg[i])
			db[0] = -12345.0; /* flag a broken raw-bin copy */
	for (int i = 0; i < hops; i++)
		if (smp_copy[i] != samples[i])
			db[0] = -12345.0;
}

void emu_level_stats(const uint8_t *reads, int n_reads, int buf_len, const int *hop_of, unsigned long long *level)
{
	std::vector<long long> offs(n_reads);
	for (int i = 0; i < n_reads; i++)
		offs[i] = (long long)i * buf_len;
	LevelParams p;
	p.base = reads;
	p.read_off = offs.data();
	p.hop_of = hop_of;
	p.n_reads = n_reads;
	p.buf_len = buf_len;
	p.level = level;
	cuda_emu::launch(dim3(2), dim3(256), 0, [&]() { level_stats_kernel(p); });
}

/* fused boxcar + transform kernel: reads [n_reads][2*N*ds] */
void emu_fused_boxcar(int L, int peak, const uint8_t *reads, int n_reads, int ds, int slots, const int *segs,
		      int n_segs, const int16_t *sine, const int32_t *win, long long *avg, long long *samples)
{
	const int N = 1 << L;
	const Tables t(sine, win, L, L);
	std::vector<long long> offs(n_reads);
	for (int i = 0; i < n_reads; i++)
		offs[i] = (long long)i * 2 * N * ds;
	FusedBoxcarParams p;
	memset(&p, 0, sizeof(p));
	p.base = reads;
	p.read_off = offs.data();
	p.segs = (const int4 *)segs;
	p.n_segs = n_segs;
	p.ds = ds;
	p.slots = slots;
	p.avg = avg;
	p.samples = samples;
	p.twc = t.twc.data();
	p.win = t.win.data();
	p.tw0 = t.tw0;
#define FBS(LV, PK, NSV)                                                                              \
	cuda_emu::launch(dim3(n_segs), dim3(kThreads), FusedSmem<LV>::bytes(ds, NSV),                 \
			 [&]() { scan_boxcar_fused_kernel<LV, PK, NSV>(p); })
#define FB(LV)                                                                                        \
	do {                                                                                          \
		if (peak) {                                                                           \
			if (slots == 12) FBS(LV, true, 12); else if (slots == 6) FBS(LV, true, 6); else if (slots == 4) FBS(LV, true, 4); else if (slots == 3) FBS(LV, true, 3); else FBS(LV, true, 2); \
		} else {                                                                              \
			if (slots == 12) FBS(LV, false, 12); else if (slots == 6) FBS(LV, false, 6); else if (slots == 4) FBS(LV, false, 4); else if (slots == 3) FBS(LV, false, 3); else FBS(LV, false, 2); \
		}                                                                                     \
	} while (0)
	switch (L) {
	case 8: FB(8); break;
	case 9: FB(9); break;
	case 10: FB(10); break;
	case 11: FB(11); break;
	case 12: FB(12); break;
	}
#undef FBS
#undef FB
}

/* warp-specialised streaming variant of the same pipeline (producer / boxcar / transform roles) */
void emu_stream_boxcar(int L, int peak, int mode, const uint8_t *reads, int n_reads, int ds, int slots, int grid, const int *segs,
		       int n_segs, const int16_t *sine, const int32_t *win, long long *avg, long long *samples)
{
	const int N = 1 << L;
	const Tables t(sine, win, L, L);
	std::vector<long long> offs(n_reads);
	for (int i = 0; i < n_reads; i++)
		offs[i] = (long long)i * 2 * N * ds;
	FusedBoxcarParams p;
	memset(&p, 0, sizeof(p));
	p.base = reads;
	p.read_off = offs.data();
	p.segs = (const int4 *)segs;
	p.n_segs = n_segs;
	p.ds = ds;
	p.slots = slots;
	p.avg = avg;
	p.samples = samples;
	p.twc = t.twc.data();
	p.win = t.win.data();
	p.tw0 = t.tw0;
#define SBM(LV, PK, FG, BG)                                                                           \
	cuda_emu::launch(dim3(grid), dim3(StreamShape<FG, BG>::threads), StreamSmem<LV, FG>::bytes(ds, slots), \
			 [&]() { scan_boxcar_stream_kernel<LV, PK, FG, BG>(p); })
#define SB(LV)                                                                                        \
	do {                                                                                          \
		if (mode == 5) {                                                                      \
			if (peak)                                                                     \
				cuda_emu::launch(dim3(grid), dim3(kSymThreads), SymSmem<LV>::bytes(ds, slots), \
						 [&]() { scan_boxcar_sym_kernel<LV, true>(p); });     \
			else                                                                          \
				cuda_emu::launch(dim3(grid), dim3(kSymThreads), SymSmem<LV>::bytes(ds, slots), \
						 [&]() { scan_boxcar_sym_kernel<LV, false>(p); });    \
		} else if (mode == 1) {                                                                      \
			if (peak) SBM(LV, true, 1, 2); else SBM(LV, false, 1, 2);                     \
		} else if (mode == 3) {                                                               \
			if (peak) SBM(LV, true, 2, 2); else SBM(LV, false, 2, 2);                     \
		} else {                                                                              \
			if (peak) SBM(LV, true, 2, 1); else SBM(LV, false, 2, 1);                     \
		}                                                                                     \
	} while (0)
	switch (L) {
	case 8: SB(8); break;
	case 9: SB(9); break;
	case 10: SB(10); break;
	case 11: SB(11); break;
	case 12: SB(12); break;
	}
#undef SB
#undef SBM
}

#include "emu_large.inl"

} /* extern "C" */
