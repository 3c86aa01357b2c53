/*
 * TEST INFRASTRUCTURE ONLY -- the CSV formatter of rtlsdr_b200/csrc/csv_text.cuh
 * on the CPU: the device functions called directly and compared with glibc's
 * printf here, and both row kernels run through cuda_emu.h.  Built by
 * tests/test_csv_text.py with
 *   g++ -std=c++20 -O2 -DSCAN_EMU -Itests/emu -Irtlsdr_b200/csrc -shared -fPIC
 */
#include "csv_text.cuh"

#include <cstdio>
#include <cstring>
#include <vector>

using namespace rscan;

extern "C" {

/* csv_fmt_f2 against snprintf("%.2f") for v[0..n): mismatches (a value outside the domain counts as one);
 * *first = index of the first */
long long emu_csv_check_f2(const double *v, long long n, long long *first)
{
	long long bad = 0;
	*first = -1;
	for (long long i = 0; i < n; i++) {
		char got[32], want[400];
		const int g = csv_fmt_f2(v[i], got);
		const int w = snprintf(want, sizeof(want), "%.2f", v[i]);
		if (g != w || memcmp(got, want, (size_t)w) != 0) {
			if (!bad)
				*first = i;
			bad++;
		}
	}
	return bad;
}

/* the formatter's text of one value (NUL-terminated), or -1 outside the domain */
int emu_csv_f2(double v, char *out)
{
	const int n = csv_fmt_f2(v, out);
	if (n >= 0)
		out[n] = '\0';
	return n;
}

long long emu_csv_check_i(const int *v, long long n, long long *first)
{
	long long bad = 0;
	*first = -1;
	for (long long i = 0; i < n; i++) {
		char got[16], want[16];
		const int g = csv_fmt_i(v[i], got);
		const int w = snprintf(want, sizeof(want), "%i", v[i]);
		if (g != w || memcmp(got, want, (size_t)w) != 0) {
			if (!bad)
				*first = i;
			bad++;
		}
	}
	return bad;
}

/* csv_rows_kernel + csv_pack_kernel for rows [row_first, row_first + rows) of the table (low, high, step);
 * db row r at db + r * db_stride.  Returns the packed length (-1 = a value outside the domain); `text` must
 * hold rows * (stamp_len + kCsvRowFixed + kCsvValueMax * db_count) bytes. */
long long emu_csv_rows(const char *stamp, int row_first, int rows, const double *db, long long db_stride,
		       const int *samples, const int *low, const int *high, int table_rows, double step, int db_count,
		       char *text)
{
	const size_t stamp_len = strlen(stamp);
	const long long slot = (long long)(stamp_len + kCsvRowFixed + (size_t)kCsvValueMax * db_count);
	std::vector<int2> cols(table_rows);
	for (int i = 0; i < table_rows; i++)
		cols[i] = make_int2(low[i], high[i]);
	std::vector<char> slots((size_t)(slot * rows));
	std::vector<int> lens(rows);
	long long len = -2;
	CsvRowParams p;
	p.db = db;
	p.db_stride = db_stride;
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
