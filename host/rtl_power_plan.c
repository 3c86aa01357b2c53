/* See rtl_power_plan.h.  Written against the reference's observable behaviour
 * (integer truncations included); cross-checked against the compiled reference
 * by tests/test_host_plan.py. */
#include "rtl_power_plan.h"

#include <ctype.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

static double suffix_scaled(const char *s, const char *suffixes, const double *scale)
{
	char tmp[64];
	size_t len = strlen(s), k;
	double v;
	if (len == 0)
		return 0.0;
	if (len >= sizeof(tmp))
		len = sizeof(tmp) - 1;
	memcpy(tmp, s, len);
	tmp[len] = '\0';
	for (k = 0; suffixes[k]; k++) {
		if (tolower((unsigned char)tmp[len - 1]) == suffixes[k]) {
			tmp[len - 1] = '\0';
			v = atof(tmp);
			return scale[k] * v;
		}
	}
	return atof(tmp);
}

double rp_atofs(const char *s)
{
	/* convenience.c:67-96 also strips trailing spaces before the suffix */
	static const double sc[] = { 1e3, 1e6, 1e9 };
	char tmp[64];
	size_t len = strlen(s);
	if (len >= sizeof(tmp))
		len = sizeof(tmp) - 1;
	memcpy(tmp, s, len);
	while (len > 1 && isspace((unsigned char)tmp[len - 1]))
		len--;
	tmp[len] = '\0';
	return suffix_scaled(tmp, "kmg", sc);
}

double rp_atoft(const char *s)
{
	static const double sc[] = { 1.0, 60.0, 3600.0 };
	return suffix_scaled(s, "smh", sc);
}

double rp_atofp(const char *s)
{
	static const double sc[] = { 0.01 };
	size_t len = strlen(s);
	if (len && s[len - 1] == '%')
		return suffix_scaled(s, "%", sc);
	return atof(s);
}

int rp_plan_range(const char *range, double crop, int boxcar, rp_plan_t *out)
{
	char field[3][64];
	const char *p = range, *q;
	int k, i, hops = 0, bw_seen = 0, bw_used = 0, bin_e = 0, ds = 1, ds_p = 0, buf_len;
	double bin_size = 0.0;

	if (!range || !out)
		return -1;
	for (k = 0; k < 3; k++) {
		size_t n;
		q = (k < 2) ? strchr(p, ':') : p + strlen(p);
		if (!q)
			return -1;
		n = (size_t)(q - p);
		if (n == 0 || n >= sizeof(field[k]))
			return -1;
		memcpy(field[k], p, n);
		field[k][n] = '\0';
		p = q + 1;
	}
	memset(out, 0, sizeof(*out));
	out->lower = (int)rp_atofs(field[0]);
	out->upper = (int)rp_atofs(field[1]);
	out->max_size = (int)rp_atofs(field[2]);

	/* evenly sized hops, each as close to the maximum rate as possible (:462-469) */
	for (i = 1; i < 1500; i++) {
		bw_seen = (out->upper - out->lower) / i;
		bw_used = (int)((double)bw_seen / (1.0 - crop));
		if (bw_used > RP_MAXIMUM_RATE)
			continue;
		hops = i;
		break;
	}
	if (hops == 0)
		return -2;
	/* narrow scans: one hop, decimate on the host side (:471-480) */
	if (bw_used < RP_MINIMUM_RATE) {
		if (bw_used <= 0)
			return -2;
		hops = 1;
		ds = RP_MAXIMUM_RATE / bw_used;
		bw_used = bw_used * ds;
	}
	if (!boxcar && ds > 1) {
		ds_p = (int)log2(ds);
		ds = 1 << ds_p;
		bw_used = (int)((double)(bw_seen * ds) / (1.0 - crop));
	}
	/* smallest power-of-two bin count whose bins are narrow enough (:483-488) */
	for (i = 1; i <= 21; i++) {
		bin_e = i;
		bin_size = (double)bw_used / (double)((1 << i) * ds);
		if (bin_size <= (double)out->max_size)
			break;
	}
	/* giant bins: one rms value per hop (:490-496) */
	if (out->max_size >= RP_MINIMUM_RATE) {
		bw_seen = out->max_size;
		bw_used = out->max_size;
		hops = (out->upper - out->lower) / bw_seen;
		bin_e = 0;
		crop = 0;
	}
	if (hops > RP_MAX_TUNES || hops <= 0)
		return -2;
	buf_len = 2 * (1 << bin_e) * ds;
	if (buf_len < RP_DEFAULT_BUF)
		buf_len = RP_DEFAULT_BUF;

	out->tune_count = hops;
	out->bin_e = bin_e;
	out->buf_len = buf_len;
	out->downsample = ds;
	out->downsample_passes = ds_p;
	out->rate = bw_used;
	out->bw_seen = bw_seen;
	out->crop = crop;
	out->bin_size = bin_size;
	for (i = 0; i < hops; i++)
		out->freq[i] = out->lower + i * bw_seen + bw_seen / 2;
	return 0;
}

void rp_plan_report(const rp_plan_t *p, void *file)
{
	FILE *f = (FILE *)file;
	const int bins = p->tune_count * (1 << p->bin_e);
	fprintf(f, "Number of frequency hops: %i\n", p->tune_count);
	fprintf(f, "Dongle bandwidth: %iHz\n", p->rate);
	fprintf(f, "Downsampling by: %ix\n", p->downsample);
	fprintf(f, "Cropping by: %0.2f%%\n", p->crop * 100);
	fprintf(f, "Total FFT bins: %i\n", bins);
	fprintf(f, "Logged FFT bins: %i\n", (int)((double)bins * (1.0 - p->crop)));
	fprintf(f, "FFT bin size: %0.2fHz\n", p->bin_size);
	fprintf(f, "Buffer size: %i bytes (%0.2fms)\n", p->buf_len,
		1000 * 0.5 * (float)p->buf_len / (float)p->rate);
}

int rp_db_count(const rp_plan_t *p)
{
	const int len = 1 << p->bin_e;
	const int i1 = 0 + (int)((double)len * p->crop * 0.5);
	const int i2 = (len - 1) - (int)((double)len * p->crop * 0.5);
	return i2 - i1 + 2;
}

void rp_csv_columns(const rp_plan_t *p, int hop, int *low, int *high, double *step)
{
	const int len = 1 << p->bin_e, ds = p->downsample;
	const int bin_count = (int)((double)len * (1.0 - p->crop));
	const int bw2 = (int)(((double)p->rate * (double)bin_count) / (len * 2 * ds));
	*low = p->freq[hop] - bw2;
	*high = p->freq[hop] + bw2;
	*step = (double)p->rate / (double)(len * ds);
}

int rp_csv_row(char *out, size_t cap, const rp_plan_t *p, int hop, int samples,
	       const double *db, int db_count)
{
	size_t used = 0;
	int i, n, low, high;
	double step;
	rp_csv_columns(p, hop, &low, &high, &step);
	n = snprintf(out, cap, "%i, %i, %.2f, %i, ", low, high, step, samples);
	if (n < 0 || (size_t)n >= cap)
		return -1;
	used = (size_t)n;
	for (i = 0; i < db_count; i++) {
		n = snprintf(out + used, cap - used, i + 1 < db_count ? "%.2f, " : "%.2f\n", db[i]);
		if (n < 0 || (size_t)n >= cap - used)
			return -1;
		used += (size_t)n;
	}
	return (int)used;
}
