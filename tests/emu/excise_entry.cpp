/*
 * TEST INFRASTRUCTURE ONLY -- the spectral-kurtosis excision pieces of the kernel source on the CPU: sk.cuh's
 * sk_sigma() and sk_from_moments() called directly, excise.cuh's fold and report kernels and csv_text.cuh's row
 * kernels run through cuda_emu.h.  Built by tests/test_excise.py with
 *   g++ -std=c++20 -O2 -ffp-contract=off -DSCAN_EMU -Itests/emu -Irtlsdr_b200/csrc -shared -fPIC
 */
#include "csv_text.cuh"
#include "excise.cuh"

#include <cstring>
#include <vector>

using namespace rscan;

extern "C" {

double emu_sk_sigma(int64_t m) { return sk_sigma(m); }

double emu_sk_from_moments(int64_t s1, uint64_t lo, uint64_t hi, int64_t m) { return sk_from_moments(s1, lo, hi, m); }

/* excise_fold_kernel over `hops` hops of 2^bin_e bins, on the grid the library launches */
void emu_excise_fold(const long long *avg, const long long *samples, const unsigned long long *s2, long long *snap_s1,
		     unsigned long long *snap_s2, long long *c1, int *b1, long long *snap_smp, unsigned *ticket,
		     double k_low, double k_high, int bin_e, int ds, int hops)
{
	ExciseFoldParams p;
	p.avg = avg;
	p.samples = samples;
	p.s2 = s2;
	p.snap_s1 = snap_s1;
	p.snap_s2 = snap_s2;
	p.c1 = c1;
	p.b1 = b1;
	p.snap_smp = snap_smp;
	p.ticket = ticket;
	p.k_low = k_low;
	p.k_high = k_high;
	p.bin_e = bin_e;
	p.downsample = ds;
	const int n = 1 << bin_e;
	cuda_emu::launch(dim3((n + 255) / 256, hops), dim3(256), 0, [&]() { excise_fold_kernel(p); });
}

/* excised_report_kernel<guard>; any output may be NULL */
void emu_excised_report(int guard, const long long *c1, const int *b1, const long long *snap_smp, int *samples_out,
			double *db, double *flagged, int bin_e, int i1, int i2, int rate, int ds, int hops)
{
	ExciseReportParams p;
	p.c1 = c1;
	p.b1 = b1;
	p.snap_smp = snap_smp;
	p.samples_out = samples_out;
	p.db = db;
	p.flagged = flagged;
	p.bin_e = bin_e;
	p.i1 = i1;
	p.i2 = i2;
	p.rate = rate;
	p.downsample = ds;
	const dim3 grid((i2 - i1 + 2 + 255) / 256, hops);
	if (guard)
		cuda_emu::launch(grid, dim3(256), 0, [&]() { excised_report_kernel<true>(p); });
	else
		cuda_emu::launch(grid, dim3(256), 0, [&]() { excised_report_kernel<false>(p); });
}

/* csv_rows_kernel (f4 = 0) or csv_sk_rows_kernel (f4 = 1) + csv_pack_kernel over rows [0, rows) of the table;
 * returns the packed length (-1 = a value outside the domain) */
long long emu_rows(int f4, const char *stamp, int rows, const double *vals, int db_count, const int *samples,
		   const int *low, const int *high, double step, char *text)
{
	const size_t stamp_len = strlen(stamp);
	const long long slot = (long long)(stamp_len + kCsvRowFixed + (size_t)(f4 ? kCsvSkValueMax : kCsvValueMax) * db_count);
	std::vector<int2> cols(rows);
	for (int i = 0; i < rows; i++)
		cols[i] = make_int2(low[i], high[i]);
	std::vector<char> slots((size_t)(slot * rows));
	std::vector<int> lens(rows);
	long long len = -2;
	CsvRowParams p;
	p.db = vals;
	p.db_stride = db_count;
	p.samples = samples;
	p.cols = cols.data();
	p.step = step;
	p.row_first = 0;
	p.db_count = db_count;
	p.slots = slots.data();
	p.slot_bytes = slot;
	p.lens = lens.data();
	p.stamp_len = (int)stamp_len;
	memcpy(p.stamp, stamp, stamp_len);
	if (f4)
		cuda_emu::launch(dim3(rows), dim3(kCsvThreads), 0, [&]() { csv_sk_rows_kernel(p); });
	else
		cuda_emu::launch(dim3(rows), dim3(kCsvThreads), 0, [&]() { csv_rows_kernel(p); });
	CsvPackParams q;
	q.slots = slots.data();
	q.slot_bytes = slot;
	q.lens = lens.data();
	q.text = text;
	q.len = &len;
	cuda_emu::launch(dim3(rows), dim3(kCsvThreads), 0, [&]() { csv_pack_kernel(q); });
	return len;
}

} /* extern "C" */
