/*
 * rtl_power_plan -- the caller side of the scan path kept semantically intact:
 * the hop planner (reference src/rtl_power.c:438-540, frequency_range), the
 * suffix parsers it uses (src/convenience/convenience.c:67-144) and the CSV row
 * formatter (src/rtl_power.c:739-760, 995-998).  Pure host code, no DSP.
 */
#ifndef RTL_POWER_PLAN_H
#define RTL_POWER_PLAN_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RP_MAX_TUNES    3000      /* rtl_power.c:113 */
#define RP_MAXIMUM_RATE 2800000   /* rtl_power.c:78 */
#define RP_MINIMUM_RATE 1000000   /* rtl_power.c:79 */
#define RP_DEFAULT_BUF  16384     /* rtl_power.c:74 */

typedef struct rp_plan {
	int tune_count;
	int bin_e;
	int buf_len;
	int downsample;
	int downsample_passes;
	int rate;        /* bw_used: sample rate requested from the dongle, tunes[i].rate */
	int bw_seen;     /* hop spacing */
	int lower, upper, max_size;
	double crop;     /* forced to 0 for >= 1 MHz bins (rtl_power.c:495) */
	double bin_size;
	int freq[RP_MAX_TUNES]; /* tunes[i].freq */
} rp_plan_t;

/* k/M/G, s/m/h and % suffix parsers (convenience.c:67-144); do not modify `s` */
double rp_atofs(const char *s);
double rp_atoft(const char *s);
double rp_atofp(const char *s);

/*
 * frequency_range(): range = "lower:upper:bin_size".  boxcar = 1 unless -F was
 * given.  Returns 0, -1 on a malformed range, -2 when no hop count fits or the
 * plan exceeds RP_MAX_TUNES ("Error: bandwidth too wide.").
 */
int rp_plan_range(const char *range, double crop, int boxcar, rp_plan_t *out);

/* the planner's stderr report (rtl_power.c:530-539) */
void rp_plan_report(const rp_plan_t *p, void *file /* FILE* */);

/*
 * One CSV row without the "date, time, " prefix (rtl_power.c:739-760):
 * "low, high, step, samples, dB, dB, ..., dB\n".  db[db_count] is what
 * rtlsdr_gpu_scan_collect() returns.  Returns characters written (excluding
 * NUL) or -1 if `cap` is too small.
 */
int rp_csv_row(char *out, size_t cap, const rp_plan_t *p, int hop, int samples,
	       const double *db, int db_count);

/* The first three columns of hop `hop`'s row (rtl_power.c:739-746): low and high edge in Hz and the
 * bin step.  rp_csv_row() prints these, and rtlsdr_gpu_scan_set_csv_columns() takes them. */
void rp_csv_columns(const rp_plan_t *p, int hop, int *low, int *high, double *step);

/* number of doubles per row = i2 - i1 + 2 (rtl_power.c:747-748) */
int rp_db_count(const rp_plan_t *p);

#ifdef __cplusplus
}
#endif
#endif
