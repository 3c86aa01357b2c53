/*
 * TEST INFRASTRUCTURE ONLY -- the spectral-kurtosis text and merge pieces of the kernel source on the CPU:
 * csv_text.cuh's %.4f formatter called directly and compared with glibc's printf, and csv_sk_rows_kernel +
 * csv_pack_kernel and sk.cuh's merge_sk_sets_kernel run through cuda_emu.h.  Built by tests/test_sk_text.py with
 *   g++ -std=c++20 -O2 -DSCAN_EMU -Itests/emu -Irtlsdr_b200/csrc -shared -fPIC
 */
#include "csv_text.cuh"
#include "sk.cuh"

#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

using namespace rscan;

extern "C" {

/* csv_fmt_f4 against snprintf("%.4f") -- "nan" for a NaN of either sign -- for v[0..n): mismatches (a value
 * outside the domain counts as one); *first = index of the first */
long long emu_csv_check_f4(const double *v, long long n, long long *first)
{
	long long bad = 0;
	*first = -1;
	for (long long i = 0; i < n; i++) {
		char got[32], want[400];
		const int g = csv_fmt_f4(v[i], got);
		const int w = std::isnan(v[i]) ? snprintf(want, sizeof(want), "nan")
					       : snprintf(want, sizeof(want), "%.4f", v[i]);
		if (g != w || memcmp(got, want, (size_t)w) != 0) {
			if (!bad)
				*first = i;
			bad++;
		}
	}
	return bad;
}

/* the formatter's text of one value (NUL-terminated), or -1 outside the domain */
int emu_csv_f4(double v, char *out)
{
	const int n = csv_fmt_f4(v, out);
	if (n >= 0)
		out[n] = '\0';
	return n;
}

/* csv_sk_rows_kernel + csv_pack_kernel for rows [row_first, row_first + rows) of the table (low, high, step); SK
 * row r at sk + r * sk_stride.  Returns the packed length (-1 = a value outside the domain); `text` must hold
 * rows * (stamp_len + kCsvRowFixed + kCsvSkValueMax * db_count) bytes. */
long long emu_sk_csv_rows(const char *stamp, int row_first, int rows, const double *sk, long long sk_stride,
			  const int *samples, const int *low, const int *high, int table_rows, double step, int db_count,
			  char *text)
{
	const size_t stamp_len = strlen(stamp);
	const long long slot = (long long)(stamp_len + kCsvRowFixed + (size_t)kCsvSkValueMax * db_count);
	std::vector<int2> cols(table_rows);
	for (int i = 0; i < table_rows; i++)
		cols[i] = make_int2(low[i], high[i]);
	std::vector<char> slots((size_t)(slot * rows));
	std::vector<int> lens(rows);
	long long len = -2;
	CsvRowParams p;
	p.db = sk;
	p.db_stride = sk_stride;
	p.samples = samples;
	p.cols = cols.data();
	p.step = step;
	p.row_first = row_first;
	p.db_count = db_count;
	p.slots = slots.data();
	p.slot_bytes = slot;
	p.lens = lens.data();
	p.stamp_len = (int)stamp_len;
	memcpy(p.stamp, stamp, stamp_len);
	cuda_emu::launch(dim3(rows), dim3(kCsvThreads), 0, [&]() { csv_sk_rows_kernel(p); });
	CsvPackParams q;
	q.slots = slots.data();
	q.slot_bytes = slot;
	q.lens = lens.data();
	q.text = text;
	q.len = &len;
	cuda_emu::launch(dim3(rows), dim3(kCsvThreads), 0, [&]() { csv_pack_kernel(q); });
	return len;
}

/* merge_sk_sets_kernel: `sets` external sets (S1 int64 [bins], counts int32 [hops], S2 u64 [bins][2] at
 * ext_* + s * stride bytes) into (avg, samples, s2) in place, on `grid` CTAs of 256 threads */
void emu_merge_sk(long long *avg, long long *samples, unsigned long long *s2, const void *ext_avg,
		  const void *ext_smp, const void *ext_s2, long long stride, long long bins, int hops, int sets, int grid)
{
	MergeSkParams p;
	p.avg = avg;
	p.samples = samples;
	p.s2 = s2;
	p.ext_avg = (const uint8_t *)ext_avg;
	p.ext_smp = (const uint8_t *)ext_smp;
	p.ext_s2 = (const uint8_t *)ext_s2;
	p.stride = stride;
	p.bins = bins;
	p.hops = hops;
	p.sets = sets;
	cuda_emu::launch(dim3(grid), dim3(256), 0, [&]() { merge_sk_sets_kernel(p); });
}

} /* extern "C" */
