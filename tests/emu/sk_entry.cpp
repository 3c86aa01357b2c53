/*
 * TEST INFRASTRUCTURE ONLY -- the spectral-kurtosis pieces of the kernel source on the CPU through cuda_emu.h:
 * sk.cuh's conversion and estimator called directly (against gcc's unsigned __int128 conversion), and the SK
 * kernels (scan_small_sk_kernel, large_round_b_sk_kernel, large_round_c_sk_kernel) run end to end.  Built by
 * tests/test_sk.py with
 *   g++ -std=c++20 -O2 -ffp-contract=off -DSCAN_EMU -Itests/emu -Irtlsdr_b200/csrc -shared -fPIC
 */
#include "scan_host.cuh"
#include "scan_kernels.cuh"
#include "scan_large.cuh"
#include "sk.cuh"

#include <cstring>
#include <vector>

using namespace rscan;

namespace {

struct Tables {
	std::vector<int2> tw, twc;
	std::vector<uint16_t> win;
	PassTw tw0;
	Tables(const int16_t *sine, const int32_t *coefs, int L, int s_end)
	{
		twiddles(sine, L, tw);
		tw0 = first_stage_tw(tw, L);
		twc = compact_tw(tw, L, s_end);
		win = window16(coefs, 1 << L);
	}
};

template <int L>
void run_small_sk(const SmallParams &p, int in16, int grid, unsigned long long *s2)
{
	if (in16)
		cuda_emu::launch(dim3(grid), dim3(kThreads), SmallSmem<L>::bytes, [&]() { scan_small_sk_kernel<L, true>(p, s2); });
	else
		cuda_emu::launch(dim3(grid), dim3(kThreads), SmallSmem<L>::bytes, [&]() { scan_small_sk_kernel<L, false>(p, s2); });
}

void run_small_sk_l(int L, const SmallParams &p, int in16, int grid, unsigned long long *s2)
{
	switch (L) {
	case 1: run_small_sk<1>(p, in16, grid, s2); break;
	case 2: run_small_sk<2>(p, in16, grid, s2); break;
	case 3: run_small_sk<3>(p, in16, grid, s2); break;
	case 4: run_small_sk<4>(p, in16, grid, s2); break;
	case 5: run_small_sk<5>(p, in16, grid, s2); break;
	case 6: run_small_sk<6>(p, in16, grid, s2); break;
	case 7: run_small_sk<7>(p, in16, grid, s2); break;
	case 8: run_small_sk<8>(p, in16, grid, s2); break;
	case 9: run_small_sk<9>(p, in16, grid, s2); break;
	case 10: run_small_sk<10>(p, in16, grid, s2); break;
	case 11: run_small_sk<11>(p, in16, grid, s2); break;
	case 12: run_small_sk<12>(p, in16, grid, s2); break;
	}
}

} // namespace

extern "C" {

double emu_sk_u128_to_double(uint64_t lo, uint64_t hi) { return sk_u128_to_double(lo, hi); }

double emu_gcc_u128_to_double(uint64_t lo, uint64_t hi)
{
	return (double)(((unsigned __int128)hi << 64) | lo);
}

double emu_sk_from_moments(int64_t s1, uint64_t lo, uint64_t hi, int64_t m)
{
	return sk_from_moments(s1, lo, hi, m);
}

/* u8 path: reads [n_reads][16384] sorted by hop; `grid` CTAs share the working sets in equal runs */
void emu_sk_small_u8(int L, const uint8_t *reads, int n_reads, const int *hop_of, int grid, const int16_t *sine,
		     const int32_t *win, long long *avg, long long *samples, unsigned long long *s2)
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
	p.avg = avg;
	p.samples = samples;
	p.samples_per_read = kStageBytes / (2 << L);
	p.tw = t.tw.data();
	p.twc = t.twc.data();
	p.win = t.win.data();
	p.tw0 = t.tw0;
	run_small_sk_l(L, p, 0, grid, s2);
}

/* decimated images [n_reads][image_stride] c16 and their DC sums [n_reads][2] (what the decimators of a
 * boxcar (boxcar = 1, ds) or -F (boxcar = 0, ds = 2^ds_p) scan of buf_len-byte reads write) -> S1, S2 */
void emu_sk_small_in16(int L, const uint32_t *images, const long long *sums, int n_reads, int buf_len, int ds,
		       int ds_p, int boxcar, const int *segs, int n_segs, const int16_t *sine, const int32_t *win,
		       long long *avg, long long *samples, unsigned long long *s2)
{
	const rtlsdr_gpu_scan_cfg_t cfg = { .tune_count = 1, .bin_e = L, .buf_len = buf_len, .downsample = ds,
					    .downsample_passes = ds_p, .boxcar = boxcar, .rate = 1 };
	ScanShape shape;
	if (scan_shape(cfg, &shape))
		return;
	const Tables t(sine, win, L, L);
	std::vector<long long> sm(sums, sums + 2 * (size_t)n_reads);
	std::vector<int> ave((size_t)n_reads * 2, 0);
	DcFinalizeParams fz;
	fz.sums = sm.data();
	fz.ave = ave.data();
	fz.n = n_reads;
	fz.l_len = shape.l_len;
	cuda_emu::launch(dim3((2 * n_reads + 255) / 256), dim3(256), 0, [&]() { dc_finalize_kernel(fz); });
	std::vector<uint32_t> img(images, images + (size_t)n_reads * shape.image_stride);
	img.resize(img.size() + kWS, 0xDEADBEEFu); /* padding must not matter */
	SmallParams p;
	memset(&p, 0, sizeof(p));
	p.base = (const uint8_t *)img.data();
	p.regular_stride = shape.image_stride * 4;
	p.segs = (const int4 *)segs;
	p.n_segs = n_segs;
	p.avg = avg;
	p.samples = samples;
	p.samples_per_read = shape.samples_per_read;
	p.tw = t.tw.data();
	p.twc = t.twc.data();
	p.win = t.win.data();
	p.dc_ave = ave.data();
	p.l_len = shape.l_len;
	p.n_blocks = shape.n_blocks;
	p.blocks_padded = shape.blocks_padded;
	p.tw0 = t.tw0;
	run_small_sk_l(L, p, 1, n_segs, s2);
}

/* large path, u8 reads [n_reads][2N] sorted by hop: round A, then round B (SK, N <= 2^16) or the pipelined round B
 * and round C (SK) */
void emu_sk_large(int L, const uint8_t *reads, int n_reads, const int *hop_of, const int16_t *sine,
		  const int32_t *win, long long *avg, unsigned long long *s2)
{
	const size_t N = (size_t)1 << L;
	const Tables t(sine, win, L, 8);
	const std::vector<int2> twb = round_b_tw(t.tw, L);
	std::vector<long long> offs(n_reads);
	for (int i = 0; i < n_reads; i++)
		offs[i] = (long long)i * (long long)(2 * N);
	std::vector<c16> scratch((size_t)n_reads * N, 0xDEADBEEFu);
	std::vector<long long> sums((size_t)n_reads * 2, 0), smp(4096, 0);
	std::vector<unsigned> tickets(n_reads, 0);
	std::vector<int2> consts(n_reads, int2{ -1, -1 });
	LargeParams p;
	memset(&p, 0, sizeof(p));
	p.base = reads;
	p.read_off = offs.data();
	p.hop_of = hop_of;
	p.scratch = scratch.data();
	p.dc_sums = sums.data();
	p.dc_consts = consts.data();
	p.twc_a = t.twc.data();
	p.avg = avg;
	p.samples = smp.data();
	p.samples_per_read = 1;
	p.tw = t.tw.data();
	p.twb = twb.data();
	p.win = t.win.data();
	p.L = L;
	p.n_entries = n_reads;
	p.tw0 = t.tw0;
	p.tiles_log2 = L - 12;
	DcSumU8Params d;
	d.base = reads;
	d.read_off = offs.data();
	d.entry_base = 0;
	d.buf_len = (int)(2 * N);
	d.sums = sums.data();
	d.tickets = tickets.data();
	d.consts = consts.data();
	dim3 tiles((unsigned)(N / kWS), n_reads);
	cuda_emu::launch(dim3(1, n_reads), dim3(256), 0, [&]() { dc_sums_u8_kernel(d); });
	cuda_emu::launch(tiles, dim3(kThreads), kLargeSmemA, [&]() { large_round_a_kernel<false>(p); });
	switch (L) {
	case 13: cuda_emu::launch(tiles, dim3(kThreads), kLargeSmemB, [&]() { large_round_b_sk_kernel<5>(p, s2); }); return;
	case 14: cuda_emu::launch(tiles, dim3(kThreads), kLargeSmemB, [&]() { large_round_b_sk_kernel<6>(p, s2); }); return;
	case 15: cuda_emu::launch(tiles, dim3(kThreads), kLargeSmemB, [&]() { large_round_b_sk_kernel<7>(p, s2); }); return;
	case 16: cuda_emu::launch(tiles, dim3(kThreads), kLargeSmemB, [&]() { large_round_b_sk_kernel<8>(p, s2); }); return;
	}
	cuda_emu::launch(dim3(5), dim3(kThreads), kLargeSmemBP, [&]() { large_round_b_pipe_kernel(p); });
	p.c_reads = n_reads > 2 ? 2 : 1; /* more than one CTA row and a hop change inside a CTA's run */
	const int cta_x = 65536 / (kThreads * round_c_vec(L - 16));
	dim3 g(cta_x, (n_reads + p.c_reads - 1) / p.c_reads);
	switch (L - 16) {
	case 1: cuda_emu::launch(g, dim3(kThreads), 0, [&]() { large_round_c_sk_kernel<1, round_c_vec(1)>(p, s2); }); break;
	case 2: cuda_emu::launch(g, dim3(kThreads), 0, [&]() { large_round_c_sk_kernel<2, round_c_vec(2)>(p, s2); }); break;
	case 3: cuda_emu::launch(g, dim3(kThreads), 0, [&]() { large_round_c_sk_kernel<3, round_c_vec(3)>(p, s2); }); break;
	case 4: cuda_emu::launch(g, dim3(kThreads), 0, [&]() { large_round_c_sk_kernel<4, round_c_vec(4)>(p, s2); }); break;
	case 5: cuda_emu::launch(g, dim3(kThreads), 0, [&]() { large_round_c_sk_kernel<5, round_c_vec(5)>(p, s2); }); break;
	}
}

/* the SK rows of `hops` hops (sk_report_kernel) */
void emu_sk_report(const long long *avg, const long long *samples, const unsigned long long *s2, double *sk, int bin_e,
		   int i1, int i2, int ds, int hops)
{
	SkReportParams p;
	p.avg = avg;
	p.samples = samples;
	p.s2 = s2;
	p.sk = sk;
	p.bin_e = bin_e;
	p.i1 = i1;
	p.i2 = i2;
	p.downsample = ds;
	p.hop0 = 0;
	const int count = i2 - i1 + 2;
	cuda_emu::launch(dim3((count + 255) / 256, hops), dim3(256), 0, [&]() { sk_report_kernel(p); });
}

} /* extern "C" */
