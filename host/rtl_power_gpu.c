/*
 * rtl_power_gpu -- rtl_power's command line and CSV output with the scan
 * arithmetic done on a B200 through include/rtlsdr_gpu_scan.h.
 *
 * What is kept from the reference tool (src/rtl_power.c):
 *   - the option letters and their meaning            (:798-882)
 *   - the hop plan                                     (:438-540, rtl_power_plan.c)
 *   - the sweep order: for every hop, retune if the centre frequency differs
 *     (5 ms settle + a 4096-byte dump read), then ONE rtlsdr_read_sync of
 *     buf_len bytes                                    (:642-659, :542-552)
 *   - reporting once per interval, rows "date, time, low, high, step, samples,
 *     dB..." in hop order                              (:989-1003, :722-760)
 *   - SIGINT: first = finish the pass and exit, second = abort (:182-211, :651)
 * What is replaced: the DSP between the read and the row (:660-718, :730-764)
 * is rtlsdr_gpu_scan_submit() / rtlsdr_gpu_scan_collect_csv(), which also formats
 * the rows on the GPU (byte-identical to rp_csv_row's printf).
 *
 * Three items of the reference's TODO list (rtl_power.c:29-36) that the GPU makes cheap:
 *   -t workers   "multiple FFT workers": the hops are dealt in contiguous ranges to `workers`
 *                B200s (one rtlsdr_gpu_scan handle per device, first device RTLSDR_GPU_DEVICE,
 *                or the list RTLSDR_GPU_DEVICES=0,2,3); hops are independent (rtl_power.c:650-719),
 *                so the CSV bytes do not depend on the worker count.  With more workers than hops
 *                (single-hop scans) every worker owns all hops and takes every workers-th SWEEP; at a
 *                report their raw int64 accumulators are merged into worker 0's
 *                (rtlsdr_gpu_scan_merge_device: sums / -P maxima are exact in any grouping), same bytes
 *                again.  The reference parses -t and ignores it (:844-846); one worker is the default.
 *   -s iir       "continuous IIR smoothing" of the dB rows across reports (cfg.iir_alpha,
 *                RTL_POWER_IIR_ALPHA, default 0.25); -s avg = the reference's behaviour.
 *   -R seed      (extension) "randomized hopping": every sweep visits the hops in a fresh random
 *                order; bins are order-independent sums / maxima (rtl_power.c:708-716).
 *
 * The sample source is host/synth_source.c (no dongle on the GPU box); it is
 * configured through environment variables so that the command line stays the
 * reference's:
 *   RTLSDR_SYNTH_MODE   xorshift | counter | const | biased | tone | replay
 *   RTLSDR_SYNTH_SEED   integer      RTLSDR_SYNTH_PARAM  integer
 *   RTLSDR_SYNTH_REPLAY path of a recording: raw rtl_sdr output, rtl_sdr WAV, or a captured
 *                       rtl_tcp stream (host/replay_file.c)
 *   RTL_POWER_ASYNC     1 = fetch every hop visit through rtlsdr_read_async + callback
 *   RTL_POWER_PASSES    report after this many sweeps instead of by wall clock
 *   RTL_POWER_TIMESTAMP fixed "date, time" prefix (byte-reproducible output)
 *   RTL_POWER_REPORTS   exit after this many reports (with RTL_POWER_PASSES: a fixed amount of work)
 *   RTLSDR_GPU_DEVICE   first CUDA device ordinal      RTLSDR_GPU_DEVICES  explicit device list for -t
 *   RTL_POWER_IIR_ALPHA smoothing factor of -s iir (0 < a <= 1)
 */
#include <math.h>
#include <signal.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>

#include "replay_file.h"
#include "rtl_power_plan.h"
#include "rtlsdr_gpu_scan.h"
#include "synth_source.h"

#define SETTLE_DUMP_BYTES 4096 /* BUFFER_DUMP, rtl_power.c:76 */

static volatile sig_atomic_t stop_requests = 0;

static void on_signal(int signum)
{
	(void)signum;
	stop_requests++;
}

static void print_usage(void)
{
	fprintf(stderr,
		"rtl_power_gpu, rtl_power's FFT logger with the scan on a B200 GPU\n\n"
		"Use:\trtl_power_gpu -f freq_range [-options] [filename]\n"
		"\t-f lower:upper:bin_size [Hz]\n"
		"\t[-i integration_interval (default: 10 seconds)]\n"
		"\t[-1 enables single-shot mode (default: off)]\n"
		"\t[-e exit_timer (default: off/0)]\n"
		"\t[-d device_index] [-g tuner_gain] [-p ppm_error] [-T] [-O] [-D mode]\n"
		"\t\t(accepted for compatibility; the synthetic source ignores them)\n"
		"\t[-w window (default: rectangle)]\n"
		"\t\t(hamming, blackman, blackman-harris, hann-poisson, bartlett, youssef)\n"
		"\t[-c crop_percent (default: 0%%)]\n"
		"\t[-F fir_size (default: disabled)] (0 or 9; switches boxcar off)\n"
		"\t[-P enables peak hold (default: off)]\n"
		"\t[-s avg|iir (default: avg; iir smooths the dB rows across reports)]\n"
		"\t[-t workers (default: 1; hops -- or, with fewer hops than workers, sweeps -- are sharded over this many GPUs)]\n"
		"\t[-R seed (visit the hops of every sweep in a random order)]\n"
		"\t[-K sk_file (also write each bin's spectral kurtosis: rows like the power rows, %%.4f values,\n"
		"\t\t~1 for noise, > 1 for intermittent signals, < 1 for steady carriers; not with -P)]\n"
		"\tfilename (a '-' dumps samples to stdout, the default)\n");
	exit(1);
}

static int env_int(const char *name, int dflt)
{
	const char *v = getenv(name);
	return (v && *v) ? atoi(v) : dflt;
}

static int synth_mode_from_env(void)
{
	const char *v = getenv("RTLSDR_SYNTH_MODE");
	if (!v) return SYNTH_XORSHIFT;
	if (!strcmp(v, "counter")) return SYNTH_COUNTER;
	if (!strcmp(v, "const")) return SYNTH_CONST;
	if (!strcmp(v, "biased")) return SYNTH_BIASED;
	if (!strcmp(v, "tone")) return SYNTH_TONE;
	if (!strcmp(v, "replay")) return SYNTH_REPLAY;
	return SYNTH_XORSHIFT;
}

/* retune(): rtl_power.c:542-552 */
static void settle_on(rtlsdr_dev_t *dev, int freq)
{
	uint8_t dump[SETTLE_DUMP_BYTES];
	int got = 0;
	rtlsdr_set_center_freq(dev, (uint32_t)freq);
	if (!getenv("RTL_POWER_PASSES"))
		usleep(5000);
	rtlsdr_read_sync(dev, dump, SETTLE_DUMP_BYTES, &got);
	if (got != SETTLE_DUMP_BYTES)
		fprintf(stderr, "Error: bad retune.\n");
}

/* async variant of one hop visit: the callback contract of rtlsdr_read_async
 * (include/rtl-sdr.h:472-500): the library owns the buffer and re-arms it as soon as
 * the callback returns, so the callback hands the bytes to the GPU path (which copies
 * them) and cancels the stream after the one buffer rtl_power wants per visit */
struct visit_ctx {
	rtlsdr_dev_t *dev;
	rtlsdr_gpu_scan_t *gpu;
	int hop, rc, taken; /* hop = index inside the worker's shard */
	uint32_t want;
};

#define MAX_WORKERS 16

/* the GPU workers: worker w owns hops [first[w], first[w + 1]); with more workers than hops (by_pass) every
 * worker owns ALL hops and takes every count-th sweep instead -- the reads of a hop are then spread over the
 * workers and their raw accumulators are merged at report time (rtlsdr_gpu_scan_merge_device) */
struct workers {
	int count;
	int by_pass, cur;
	int first[MAX_WORKERS + 1];
	rtlsdr_gpu_scan_t *gpu[MAX_WORKERS];
};

static int worker_of(const struct workers *ws, int hop)
{
	int w = 0;
	if (ws->by_pass)
		return ws->cur;
	while (w + 1 < ws->count && hop >= ws->first[w + 1])
		w++;
	return w;
}

static uint64_t order_rng(uint64_t *s)
{
	*s ^= *s << 13;
	*s ^= *s >> 7;
	*s ^= *s << 17;
	return *s;
}

static void on_samples(unsigned char *buf, uint32_t len, void *ctx)
{
	struct visit_ctx *v = (struct visit_ctx *)ctx;
	if (v->taken)
		return;
	v->taken = 1;
	v->rc = (len == v->want) ? rtlsdr_gpu_scan_submit(v->gpu, v->hop, buf, len) : RTLSDR_GPU_ERR_LENGTH;
	rtlsdr_cancel_async(v->dev);
}

/* one sweep over all hops: the control flow of scanner(), rtl_power.c:642-659 */
static int sweep(rtlsdr_dev_t *dev, const struct workers *ws, const rp_plan_t *plan, uint8_t *buf8,
		 int *order, uint64_t *shuffle_state, int use_async)
{
	int i, hop, got, rc;
	if (shuffle_state) { /* -R: Fisher-Yates over the hop order of this sweep */
		for (i = plan->tune_count - 1; i > 0; i--) {
			int j = (int)(order_rng(shuffle_state) % (uint64_t)(i + 1)), t = order[i];
			order[i] = order[j];
			order[j] = t;
		}
	}
	for (i = 0; i < plan->tune_count; i++) {
		const int w = worker_of(ws, order[i]);
		rtlsdr_gpu_scan_t *gpu = ws->gpu[w];
		hop = order[i];
		if (stop_requests >= 2)
			return 0;
		if ((int)rtlsdr_get_center_freq(dev) != plan->freq[hop])
			settle_on(dev, plan->freq[hop]);
		if (use_async) {
			struct visit_ctx v = { dev, gpu, hop - ws->first[w], 0, 0, (uint32_t)plan->buf_len };
			rtlsdr_read_async(dev, on_samples, &v, 4, (uint32_t)plan->buf_len);
			if (v.rc) {
				fprintf(stderr, "rtlsdr_gpu_scan_submit: %s\n", rtlsdr_gpu_scan_strerror(v.rc));
				return v.rc;
			}
			continue;
		}
		got = 0;
		rtlsdr_read_sync(dev, buf8, plan->buf_len, &got);
		if (got != plan->buf_len)
			fprintf(stderr, "Error: dropped samples.\n");
		/* like the reference, the whole per-hop buffer is processed even after a short read
		 * (RTLSDR_GPU_FLAG_SHORT_READS keeps tunes[hop].buf8's stale tail inside the library) */
		rc = rtlsdr_gpu_scan_submit(gpu, hop - ws->first[w], buf8, (uint32_t)(got > 0 && got < plan->buf_len ? got : plan->buf_len));
		if (rc) {
			fprintf(stderr, "rtlsdr_gpu_scan_submit: %s (%s)\n", rtlsdr_gpu_scan_strerror(rc),
				rtlsdr_gpu_scan_last_cuda_error(gpu));
			return rc;
		}
	}
	return 0;
}

/* the row table of a worker: the plan's hops [first, first + rows) */
static int set_columns(rtlsdr_gpu_scan_t *gpu, const rp_plan_t *plan, int first, int rows)
{
	int32_t *low = (int32_t *)malloc(sizeof(int32_t) * (size_t)rows);
	int32_t *high = (int32_t *)malloc(sizeof(int32_t) * (size_t)rows);
	double step = 0.0;
	int i, l, h, rc = RTLSDR_GPU_ERR_NOMEM;
	if (low && high) {
		for (i = 0; i < rows; i++) {
			rp_csv_columns(plan, first + i, &l, &h, &step);
			low[i] = l;
			high[i] = h;
		}
		rc = rtlsdr_gpu_scan_set_csv_columns(gpu, rows, low, high, step);
	}
	free(low);
	free(high);
	return rc;
}

/* the device list of -t: RTLSDR_GPU_DEVICES=0,2,3 or RTLSDR_GPU_DEVICE, RTLSDR_GPU_DEVICE + 1, ... */
static int device_list(int workers, int *devices)
{
	const char *list = getenv("RTLSDR_GPU_DEVICES");
	int n = 0, first = env_int("RTLSDR_GPU_DEVICE", 0);
	if (list && *list) {
		char *copy = strdup(list), *save = NULL, *tok;
		for (tok = strtok_r(copy, ",", &save); tok && n < MAX_WORKERS; tok = strtok_r(NULL, ",", &save))
			devices[n++] = atoi(tok);
		free(copy);
		return n;
	}
	for (n = 0; n < workers && n < MAX_WORKERS; n++)
		devices[n] = first + n;
	return n;
}

int main(int argc, char **argv)
{
	const char *range = NULL, *window = "rectangle", *filename = "-", *sk_filename = NULL;
	const char *fixed_stamp = getenv("RTL_POWER_TIMESTAMP");
	int opt, interval = 10, single = 0, peak_hold = 0, boxcar = 1, comp_fir_size = 0;
	int passes_per_report = env_int("RTL_POWER_PASSES", 0), passes = 0, rc = 0, hop, w;
	int max_reports = env_int("RTL_POWER_REPORTS", 0), reports = 0;
	int want_workers = 1, smooth_iir = 0, shuffle = 0, devices[MAX_WORKERS];
	uint8_t *parts = NULL;      /* by_pass: raw bins + counts of workers 1.., pinned (device-readable) */
	size_t part_avg_bytes = 0, part_bytes = 0;
	const int use_async = getenv("RTL_POWER_ASYNC") != NULL;
	uint64_t shuffle_state = 0;
	long exit_after = 0;
	double crop = 0.0;
	time_t next_tick, exit_time = 0, now;
	rp_plan_t *plan;
	rtlsdr_dev_t *dev = NULL;
	struct workers ws;
	rtlsdr_gpu_scan_cfg_t cfg;
	int32_t *window_coefs = NULL;
	uint8_t *buf8, *replay = NULL;
	int *order;
	char *text, *sk_text = NULL, stamp[80];
	size_t text_cap = 0, text_len = 0, sk_cap = 0, sk_len = 0;
	FILE *out, *skf = NULL;
	struct sigaction sa;

	memset(&ws, 0, sizeof(ws));
	while ((opt = getopt(argc, argv, "f:i:s:t:d:g:p:e:w:c:F:1POhTD:R:K:")) != -1) {
		switch (opt) {
		case 'f': range = optarg; break;
		case 'i': interval = (int)round(rp_atoft(optarg)); break;
		case 'e': exit_after = (long)round(rp_atoft(optarg)); break;
		case 'w': window = optarg; break;
		case 'c': crop = rp_atofp(optarg); break;
		case 'F': boxcar = 0; comp_fir_size = atoi(optarg); break;
		case '1': single = 1; break;
		case 'P': peak_hold = 1; break;
		case 's': smooth_iir = strcmp("iir", optarg) == 0; break; /* avg | iir, rtl_power.c:820-825 */
		case 't': want_workers = atoi(optarg); break;             /* rtl_power.c:844-846 */
		case 'K': sk_filename = optarg; break;
		case 'R': shuffle = 1; shuffle_state = 0x9E3779B97F4A7C15ULL ^ (uint64_t)strtoull(optarg, NULL, 0); break;
		case 'd': case 'g': case 'p': case 'O': case 'T': case 'D':
			break; /* device housekeeping: no dongle behind the synthetic source */
		case 'h':
		default:
			print_usage();
		}
	}
	if (!range) {
		fprintf(stderr, "No frequency range provided.\n");
		return 1;
	}
	if (crop < 0.0 || crop > 1.0) {
		fprintf(stderr, "Crop value outside of 0 to 1.\n");
		return 1;
	}
	plan = (rp_plan_t *)calloc(1, sizeof(*plan));
	rc = rp_plan_range(range, crop, boxcar, plan);
	if (rc == -2) {
		fprintf(stderr, "Error: bandwidth too wide.\n");
		return 1;
	}
	if (rc || plan->tune_count == 0)
		print_usage();
	rp_plan_report(plan, stderr);
	if (optind < argc)
		filename = argv[optind];
	if (interval < 1)
		interval = 1;
	fprintf(stderr, "Reporting every %i seconds\n", interval);

	if (rtlsdr_open(&dev, 0) < 0) {
		fprintf(stderr, "Failed to open rtlsdr device #0.\n");
		return 1;
	}
	synth_configure(dev, synth_mode_from_env(), (uint64_t)env_int("RTLSDR_SYNTH_SEED", 0),
			env_int("RTLSDR_SYNTH_PARAM", 0));
	synth_set_hops(dev, plan->freq, plan->tune_count);
	synth_set_block_len(dev, (size_t)plan->buf_len);
	if (synth_mode_from_env() == SYNTH_REPLAY) {
		size_t n_reads = 0;
		const char *path = getenv("RTLSDR_SYNTH_REPLAY");
		replay_info_t rinfo;
		replay = path ? replay_load(path, (size_t)plan->buf_len, &n_reads, &rinfo) : NULL;
		if (!replay) {
			fprintf(stderr, "Failed to load replay file.\n");
			return 1;
		}
		synth_set_replay(dev, replay, (size_t)plan->buf_len, n_reads);
	}

	memset(&sa, 0, sizeof(sa));
	sa.sa_handler = on_signal;
	sigemptyset(&sa.sa_mask);
	sigaction(SIGINT, &sa, NULL);
	sigaction(SIGTERM, &sa, NULL);
	sigaction(SIGQUIT, &sa, NULL);
	sigaction(SIGPIPE, &sa, NULL);

	if (strcmp(filename, "-") == 0) {
		out = stdout;
	} else {
		out = fopen(filename, "wb");
		if (!out) {
			fprintf(stderr, "Failed to open %s\n", filename);
			return 1;
		}
	}

	rtlsdr_reset_buffer(dev);
	rtlsdr_set_sample_rate(dev, (uint32_t)plan->rate);

	/* host-built window table, rtl_power.c:985-988 */
	window_coefs = (int32_t *)malloc(sizeof(int32_t) << plan->bin_e);
	rtlsdr_gpu_scan_window(window, 1 << plan->bin_e, window_coefs);

	/* the GPU workers: contiguous, balanced hop ranges (sizes differ by at most one) */
	if (want_workers < 1)
		want_workers = 1;
	if (want_workers > MAX_WORKERS)
		want_workers = MAX_WORKERS;
	ws.count = device_list(want_workers, devices);
	if (ws.count > want_workers)
		ws.count = want_workers;
	/* fewer hops than workers (single-hop scans): shard the sweeps, not the hops */
	ws.by_pass = ws.count > plan->tune_count;
	if (sk_filename && ws.by_pass) {
		fprintf(stderr, "-K: the spectral kurtosis needs all reads of a hop on one worker (fewer hops than workers).\n");
		return 1;
	}
	if (sk_filename) {
		skf = fopen(sk_filename, "wb");
		if (!skf) {
			fprintf(stderr, "Failed to open %s\n", sk_filename);
			return 1;
		}
	}
	for (w = 0; w <= ws.count; w++) {
		const int base = plan->tune_count / ws.count, extra = plan->tune_count % ws.count;
		ws.first[w] = ws.by_pass ? (w < ws.count ? 0 : plan->tune_count) : w * base + (w < extra ? w : extra);
	}
	memset(&cfg, 0, sizeof(cfg));
	cfg.struct_size = sizeof(cfg);
	cfg.bin_e = plan->bin_e;
	cfg.buf_len = plan->buf_len;
	cfg.downsample = plan->downsample;
	cfg.downsample_passes = plan->downsample_passes;
	cfg.boxcar = boxcar;
	cfg.comp_fir_size = comp_fir_size;
	cfg.peak_hold = peak_hold;
	cfg.rate = plan->rate;
	cfg.crop = plan->crop;
	cfg.window_coefs = window_coefs;
	cfg.flags = RTLSDR_GPU_FLAG_SHORT_READS | (skf ? RTLSDR_GPU_FLAG_SPECTRAL_KURTOSIS : 0u);
	if (smooth_iir) {
		const char *a = getenv("RTL_POWER_IIR_ALPHA");
		cfg.iir_alpha = (a && *a) ? atof(a) : 0.25;
	}
	for (w = 0; w < ws.count; w++) {
		cfg.device = devices[w];
		cfg.tune_count = ws.by_pass ? plan->tune_count : ws.first[w + 1] - ws.first[w];
		rc = rtlsdr_gpu_scan_init(&cfg, &ws.gpu[w]);
		if (!rc)
			rc = set_columns(ws.gpu[w], plan, ws.first[w], cfg.tune_count);
		if (rc) {
			fprintf(stderr, "rtlsdr_gpu_scan_init (device %d): %s\n", devices[w], rtlsdr_gpu_scan_strerror(rc));
			return 1;
		}
		/* text buffer for the longest stamp this program prints */
		if ((size_t)rtlsdr_gpu_scan_csv_capacity(ws.gpu[w], cfg.tune_count, sizeof(stamp) - 1) > text_cap)
			text_cap = (size_t)rtlsdr_gpu_scan_csv_capacity(ws.gpu[w], cfg.tune_count, sizeof(stamp) - 1);
		if (skf && (size_t)rtlsdr_gpu_scan_sk_csv_capacity(ws.gpu[w], cfg.tune_count, sizeof(stamp) - 1) > sk_cap)
			sk_cap = (size_t)rtlsdr_gpu_scan_sk_csv_capacity(ws.gpu[w], cfg.tune_count, sizeof(stamp) - 1);
	}
	if (ws.count > 1 && ws.by_pass)
		fprintf(stderr, "GPU workers: %d (all %d hops each, every %d-th sweep; accumulators merged per report)\n",
			ws.count, plan->tune_count, ws.count);
	else if (ws.count > 1)
		fprintf(stderr, "GPU workers: %d (hops per worker: %d..%d)\n", ws.count,
			plan->tune_count / ws.count, (plan->tune_count + ws.count - 1) / ws.count);
	if (ws.by_pass) {
		part_avg_bytes = (sizeof(int64_t) << plan->bin_e) * (size_t)plan->tune_count;
		part_bytes = part_avg_bytes + ((sizeof(int) * (size_t)plan->tune_count + 7) & ~(size_t)7);
		parts = (uint8_t *)rtlsdr_gpu_scan_host_alloc(part_bytes * (size_t)(ws.count - 1));
		if (!parts) {
			fprintf(stderr, "Out of memory.\n");
			return 1;
		}
	}

	buf8 = (uint8_t *)malloc((size_t)plan->buf_len);
	/* report landing area: pinned, so every worker's device-to-host copy is plain DMA */
	text = (char *)rtlsdr_gpu_scan_host_alloc(text_cap);
	if (skf)
		sk_text = (char *)rtlsdr_gpu_scan_host_alloc(sk_cap);
	order = (int *)malloc(sizeof(int) * (size_t)plan->tune_count);
	if (!buf8 || !text || (skf && !sk_text) || !order) {
		fprintf(stderr, "Out of memory.\n");
		return 1;
	}
	for (hop = 0; hop < plan->tune_count; hop++)
		order[hop] = hop;
	next_tick = time(NULL) + interval;
	if (exit_after)
		exit_time = time(NULL) + exit_after;

	while (!stop_requests) {
		ws.cur = ws.by_pass ? passes % ws.count : 0;
		rc = sweep(dev, &ws, plan, buf8, order, shuffle ? &shuffle_state : NULL, use_async);
		if (rc)
			break;
		passes++;
		now = time(NULL);
		if (passes_per_report ? (passes % passes_per_report) != 0 : now < next_tick)
			continue;
		if (fixed_stamp) {
			snprintf(stamp, sizeof(stamp) - 2, "%s", fixed_stamp);
		} else {
			struct tm *cal = localtime(&now);
			strftime(stamp, sizeof(stamp) - 2, "%Y-%m-%d, %H:%M:%S", cal);
		}
		strcat(stamp, ", ");
		/* one report per worker (csv_dbm's reads and zeroing, rtl_power.c:730-764): the epilogue and the
		 * row formatter run on the worker's GPU, its rows' text is written out in hop order (:995-1000) */
		if (ws.by_pass) {
			/* the other workers' raw int64 bins and counts land in pinned memory, worker 0 folds them into its
			 * own accumulators (sums, or maxima under -P: exact in any grouping) and reports alone */
			for (w = 1; w < ws.count && !rc; w++)
				rc = rtlsdr_gpu_scan_collect_all(ws.gpu[w], (int64_t *)(parts + (size_t)(w - 1) * part_bytes),
								 (int *)(parts + (size_t)(w - 1) * part_bytes + part_avg_bytes), NULL);
			if (!rc)
				rc = rtlsdr_gpu_scan_merge_device(ws.gpu[0], parts, parts + part_avg_bytes, ws.count - 1,
								  (int64_t)part_bytes);
			if (!rc)
				rc = rtlsdr_gpu_scan_collect_csv(ws.gpu[0], stamp, text, text_cap, &text_len);
			if (!rc)
				fwrite(text, 1, text_len, out);
			if (rc)
				fprintf(stderr, "merging the workers' accumulators: %s (%s)\n", rtlsdr_gpu_scan_strerror(rc),
					rtlsdr_gpu_scan_last_cuda_error(ws.gpu[0]));
		}
		/* -K: the SK rows are formatted beside the power rows, with the same read-and-zero */
		for (w = 0; w < ws.count && !rc && !ws.by_pass; w++) {
			rc = skf ? rtlsdr_gpu_scan_collect_sk_csv(ws.gpu[w], stamp, text, text_cap, &text_len, sk_text, sk_cap,
								  &sk_len)
				 : rtlsdr_gpu_scan_collect_csv(ws.gpu[w], stamp, text, text_cap, &text_len);
			if (rc) {
				fprintf(stderr, "%s: %s (%s)\n", skf ? "rtlsdr_gpu_scan_collect_sk_csv" : "rtlsdr_gpu_scan_collect_csv",
					rtlsdr_gpu_scan_strerror(rc), rtlsdr_gpu_scan_last_cuda_error(ws.gpu[w]));
			} else {
				fwrite(text, 1, text_len, out);
				if (skf)
					fwrite(sk_text, 1, sk_len, skf);
			}
		}
		fflush(out);
		if (skf)
			fflush(skf);
		if (rc)
			break;
		while (time(NULL) >= next_tick)
			next_tick += interval;
		if (single || (max_reports && ++reports >= max_reports))
			break;
		if (exit_time && time(NULL) >= exit_time)
			break;
	}

	if (stop_requests)
		fprintf(stderr, "\nUser cancel, exiting...\n");
	else if (rc)
		fprintf(stderr, "\nLibrary error %d, exiting...\n", rc);
	if (out != stdout)
		fclose(out);
	if (skf)
		fclose(skf);
	for (w = 0; w < ws.count; w++)
		rtlsdr_gpu_scan_close(ws.gpu[w]);
	rtlsdr_close(dev);
	free(buf8);
	rtlsdr_gpu_scan_host_free(text);
	rtlsdr_gpu_scan_host_free(sk_text);
	rtlsdr_gpu_scan_host_free(parts);
	free(order);
	free(window_coefs);
	free(replay);
	free(plan);
	return rc ? 1 : 0;
}
