/*
 * TEST INFRASTRUCTURE ONLY -- the guard-bit kernels (rtlsdr_b200/csrc/scan_guard.cuh) and the guard dB epilogue on the
 * CPU through cuda_emu.h, with the library's own host tables (scan_host.cuh).  Built by tests/test_guard.py with
 *   g++ -std=c++20 -O2 -ffp-contract=off -DSCAN_EMU -Itests/emu -Irtlsdr_b200/csrc -shared -fPIC
 */
#include "scan_host.cuh"
#include "scan_kernels.cuh"
#include "scan_large.cuh"
#include "scan_guard.cuh"

#include <cstring>
#include <vector>

using namespace rscan;

namespace {

template <bool IN16, int MODE>
void run_guard_mode(GuardParams &p, int grid)
{
	cuda_emu::launch(dim3(grid), dim3(kThreads), 0, [&]() { guard_fft_a_kernel<IN16, MODE>(p); });
	if (p.L > 12)
		cuda_emu::launch(dim3(1u << (p.L - 12), p.b_groups), dim3(kThreads), 0, [&]() { guard_fft_b_kernel<MODE>(p); });
}

template <bool IN16>
void run_guard(GuardParams &p, int mode, int grid)
{
	if (mode == GUARD_SK)
		run_guard_mode<IN16, GUARD_SK>(p, grid);
	else if (mode == GUARD_PEAK)
		run_guard_mode<IN16, GUARD_PEAK>(p, grid);
	else
		run_guard_mode<IN16, GUARD_SUM>(p, grid);
}

struct Tables {
	std::vector<int2> tw;
	std::vector<uint16_t> win;
	Tables(const int16_t *sine, const int32_t *coefs, int L)
	{
		twiddles(sine, L, tw);
		win = window16(coefs, 1 << L);
	}
};

} // namespace

extern "C" {

/* u8 reads [n_reads][buf_len] (hop_of[i] = hop of read i) -> bins, sample counts, S2 (mode 2) as the library's guard
 * path computes them: dc_sums_u8_kernel, guard_fft_a_kernel over `grid` CTAs, and for N > 4096 guard_fft_b_kernel
 * over b_groups rows of CTAs.  Returns 0, or -1 for a configuration scan_shape() rejects. */
int emu_guard_u8(int L, const uint8_t *reads, int n_reads, int buf_len, const int *hop_of, int grid, int b_groups,
		 int mode, const int16_t *sine, const int32_t *win, long long *avg, long long *samples,
		 unsigned long long *s2)
{
	const rtlsdr_gpu_scan_cfg_t cfg = { .tune_count = 1, .bin_e = L, .buf_len = buf_len, .downsample = 1, .boxcar = 1,
					    .rate = 1, .flags = RTLSDR_GPU_FLAG_GUARD_BITS };
	ScanShape shape;
	if (scan_shape(cfg, &shape))
		return -1;
	const Tables t(sine, win, L);
	const long long N = 1ll << L;
	std::vector<long long> offs(n_reads), sums((size_t)n_reads * 2, 0);
	for (int i = 0; i < n_reads; i++)
		offs[i] = (long long)i * buf_len;
	std::vector<unsigned> tickets(n_reads, 0);
	std::vector<int2> consts(n_reads, int2{ -1, -1 });
	DcSumU8Params d;
	d.base = reads;
	d.read_off = offs.data();
	d.entry_base = 0;
	d.buf_len = buf_len;
	d.sums = sums.data();
	d.tickets = tickets.data();
	d.consts = consts.data();
	cuda_emu::launch(dim3(1, n_reads), dim3(256), 0, [&]() { dc_sums_u8_kernel(d); });
	std::vector<int2> scratch(L > 12 ? (size_t)n_reads * N : 1, int2{ 0x5EAD, 0x5EAD });
	GuardParams p;
	memset(&p, 0, sizeof(p));
	p.base = reads;
	p.read_off = offs.data();
	p.n_entries = n_reads;
	p.hop_of = hop_of;
	p.dc_u8 = consts.data();
	p.n_blocks = shape.n_blocks;
	p.L = L;
	p.tw = t.tw.data();
	p.win = t.win.data();
	p.scratch = scratch.data();
	p.avg = avg;
	p.samples = samples;
	p.samples_per_read = shape.samples_per_read;
	p.s2 = s2;
	p.b_groups = b_groups;
	run_guard<false>(p, mode, grid);
	return 0;
}

/* decimated images [n_reads][image_stride] c16 and their DC sums [n_reads][2] (what the decimators of a boxcar
 * (boxcar = 1, ds) or -F (boxcar = 0, ds = 2^ds_p) scan of buf_len-byte reads write) -> bins, counts, S2 */
int emu_guard_in16(int L, const uint32_t *images, const long long *sums, int n_reads, int buf_len, int ds, int ds_p,
		   int boxcar, const int *hop_of, int grid, int b_groups, int mode, const int16_t *sine,
		   const int32_t *win, long long *avg, long long *samples, unsigned long long *s2)
{
	const rtlsdr_gpu_scan_cfg_t cfg = { .tune_count = 1, .bin_e = L, .buf_len = buf_len, .downsample = ds,
					    .downsample_passes = ds_p, .boxcar = boxcar, .rate = 1,
					    .flags = RTLSDR_GPU_FLAG_GUARD_BITS };
	ScanShape shape;
	if (scan_shape(cfg, &shape))
		return -1;
	const Tables t(sine, win, L);
	const long long N = 1ll << L;
	std::vector<long long> sm(sums, sums + 2 * (size_t)n_reads);
	std::vector<int> ave((size_t)n_reads * 2, 0);
	DcFinalizeParams fz;
	fz.sums = sm.data();
	fz.ave = ave.data();
	fz.n = n_reads;
	fz.l_len = shape.l_len;
	cuda_emu::launch(dim3((2 * n_reads + 255) / 256), dim3(256), 0, [&]() { dc_finalize_kernel(fz); });
	std::vector<uint32_t> img(images, images + (size_t)n_reads * shape.image_stride);
	std::vector<int2> scratch(L > 12 ? (size_t)n_reads * N : 1, int2{ 0x5EAD, 0x5EAD });
	GuardParams p;
	memset(&p, 0, sizeof(p));
	p.base = (const uint8_t *)img.data();
	p.regular_stride = shape.image_stride * 4;
	p.n_entries = n_reads;
	p.hop_of = hop_of;
	p.dc_ave = ave.data();
	p.l_len = shape.l_len;
	p.n_blocks = shape.n_blocks;
	p.blocks_padded = shape.blocks_padded;
	p.L = L;
	p.tw = t.tw.data();
	p.win = t.win.data();
	p.scratch = scratch.data();
	p.avg = avg;
	p.samples = samples;
	p.samples_per_read = shape.samples_per_read;
	p.s2 = s2;
	p.b_groups = b_groups;
	run_guard<true>(p, mode, grid);
	return 0;
}

/* the guard dB rows of `hops` hops (epilogue_guard_kernel), db [hops][i2 - i1 + 2]; iir (may be NULL) is the -s iir
 * smoothing state [hops][i2 - i1 + 1] (NaN = no report yet) */
void emu_guard_epilogue_iir(const long long *avg, const long long *samples, double *db, int bin_e, int i1, int i2,
			    int rate, int hops, double *iir, double iir_alpha)
{
	EpilogueParams p;
	memset(&p, 0, sizeof(p));
	p.iir = iir;
	p.iir_alpha = iir_alpha;
	p.avg = avg;
	p.samples = samples;
	p.db = db;
	p.bin_e = bin_e;
	p.i1 = i1;
	p.i2 = i2;
	p.rate = rate;
	const int count = i2 - i1 + 2;
	cuda_emu::launch(dim3((count + 255) / 256, hops), dim3(256), 0, [&]() { epilogue_guard_kernel(p); });
}

void emu_guard_epilogue(const long long *avg, const long long *samples, double *db, int bin_e, int i1, int i2, int rate,
			int hops)
{
	emu_guard_epilogue_iir(avg, samples, db, bin_e, i1, i2, rate, hops, nullptr, 0.0);
}

} /* extern "C" */
