/*
 * rtlsdr_gpu_scan.h -- C ABI of the B200 (sm_100a) implementation of
 * rtl_power's per-hop scan pipeline.
 *
 * This is the drop-in boundary for ONE path of old-dab/rtlsdr: the body of
 * scanner()'s per-hop loop (reference src/rtl_power.c:660-718) and the reads of
 * tunes[i].avg / tunes[i].samples that csv_dbm() makes (src/rtl_power.c:730-764).
 * Everything the reference keeps in globals for that path -- tunes[],
 * tune_count, boxcar, comp_fir_size, peak_hold, window_coefs, Sinewave
 * (src/rtl_power.c:85-120) -- arrives through rtlsdr_gpu_scan_cfg_t.
 *
 * Conventions follow librtlsdr (include/rtl-sdr.h): opaque handle typedef
 * (rtl-sdr.h:37), `int` results with 0 = success and negative = error
 * (rtl-sdr.h:70-78, 466-470), extern "C" guards (rtl-sdr.h:23-25), explicit
 * symbol export with hidden default visibility (include/rtl-sdr_export.h,
 * CMakeLists.txt:54).  No CUDA or torch types appear in any signature: device
 * buffers and streams are passed as plain pointers.
 *
 * Threading: like the reference's scanner(), which is single threaded
 * (src/rtl_power.c:642-720), one handle must be driven by one thread at a
 * time.  submit() may be called from inside an rtlsdr_read_async callback
 * (include/rtl-sdr.h:472): it copies out of `buf` before returning, because
 * librtlsdr re-arms the transfer buffer as soon as the callback returns
 * (src/librtlsdr.c:2705-2707).
 *
 * There is no CPU fallback: every entry point that computes fails with
 * RTLSDR_GPU_ERR_CUDA / RTLSDR_GPU_ERR_NO_DEVICE when no sm_100 device or
 * driver is usable.
 */
#ifndef RTLSDR_GPU_SCAN_H
#define RTLSDR_GPU_SCAN_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define RTLSDR_GPU_API __attribute__((visibility("default")))
#else
#define RTLSDR_GPU_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* opaque, like rtlsdr_dev_t (include/rtl-sdr.h:37) */
typedef struct rtlsdr_gpu_scan rtlsdr_gpu_scan_t;

enum rtlsdr_gpu_scan_error {
	RTLSDR_GPU_OK            =  0,
	RTLSDR_GPU_ERR_NULL      = -1,  /* NULL handle / argument (librtlsdr returns -1 for !dev) */
	RTLSDR_GPU_ERR_CONFIG    = -2,  /* inconsistent or unsupported configuration */
	RTLSDR_GPU_ERR_HOP       = -3,  /* hop index outside [0, tune_count) */
	RTLSDR_GPU_ERR_LENGTH    = -4,  /* submit length != buf_len (short read, see submit), or a text buffer
	                                 * smaller than rtlsdr_gpu_scan_csv_capacity() */
	RTLSDR_GPU_ERR_NO_DEVICE = -5,  /* no CUDA device / device is not sm_100 */
	RTLSDR_GPU_ERR_CUDA      = -6,  /* a CUDA runtime call or kernel failed */
	RTLSDR_GPU_ERR_NOMEM     = -7,  /* host or device allocation failed */
	RTLSDR_GPU_ERR_ALIGN     = -8   /* device buffer not 16-byte aligned / stride not multiple of 16 */
};

/*
 * Configuration = the reference's per-scan state.  Field <- reference source:
 *   tune_count         <- tune_count                         rtl_power.c:116
 *   bin_e              <- tunes[0].bin_e  (scanner reads hop 0's) rtl_power.c:647
 *   buf_len            <- tunes[0].buf_len                   rtl_power.c:649, 501-504
 *   downsample         <- tunes[i].downsample   (same for all hops, :506-529)
 *   downsample_passes  <- tunes[i].downsample_passes
 *   boxcar             <- boxcar        (1 unless -F given)  rtl_power.c:118, 870-873
 *   comp_fir_size      <- comp_fir_size (-F argument)        rtl_power.c:119
 *   peak_hold          <- peak_hold     (-P)                 rtl_power.c:120, 853
 *   rate               <- tunes[i].rate  (dB scaling only)   rtl_power.c:751
 *   crop               <- tunes[i].crop  (dB/crop only)      rtl_power.c:741-748
 *   window_coefs       <- window_coefs[1<<bin_e], built on the host exactly
 *                         like rtl_power.c:985-988; NULL = rectangle (all 256).
 *                         Only used when bin_e > 0.
 *   sinewave           <- Sinewave[(1<<bin_e)*3/4] as built by sine_table()
 *                         rtl_power.c:247-261; NULL = the library builds it on
 *                         the host with the same expression.
 */
typedef struct rtlsdr_gpu_scan_cfg {
	uint32_t struct_size;       /* = sizeof(rtlsdr_gpu_scan_cfg_t), ABI versioning */
	int32_t  device;            /* CUDA device ordinal */
	int32_t  tune_count;
	int32_t  bin_e;
	int32_t  buf_len;
	int32_t  downsample;
	int32_t  downsample_passes;
	int32_t  boxcar;
	int32_t  comp_fir_size;
	int32_t  peak_hold;
	int32_t  rate;
	double   crop;
	const int32_t *window_coefs;
	const int16_t *sinewave;
	uint32_t ring_bytes;        /* pinned staging ring size per half, 0 = default (32 MiB) */
	uint32_t flags;             /* RTLSDR_GPU_FLAG_* */
	/* fields added after the first release: a caller that passes the shorter struct_size gets 0 */
	double   iir_alpha;         /* -s iir: 0 = off (plain per-interval averages, what the reference does),
	                             * 0 < a <= 1 = smoothing factor of the dB rows across reports, see collect() */
} rtlsdr_gpu_scan_cfg_t;

/* struct_size of the first release (up to and including `flags`) is still accepted */
#define RTLSDR_GPU_SCAN_CFG_V1_SIZE ((uint32_t)offsetof(rtlsdr_gpu_scan_cfg_t, iir_alpha))

/* cfg.flags: also count, per hop, the byte statistics librtlsdr's soft AGC looks at
 * (src/librtlsdr.c:3288-3306); read them with rtlsdr_gpu_scan_level_stats() */
#define RTLSDR_GPU_FLAG_LEVEL_STATS 1u
/* cfg.flags: rtlsdr_gpu_scan_collect_device() becomes asynchronous to the handle's stream: a second accumulator
 * set is allocated, the report of the current set runs on a separate stream
 * (rtlsdr_gpu_scan_get_report_stream()) behind everything submitted so far, and the next submits accumulate
 * into the other set at once -- back-to-back integration intervals with the report off the transform's
 * critical path (what rtl_power does between two reports, rtl_power.c:989-1003, without stalling the scanner).
 * The caller orders its use of the report buffers against the REPORT stream.  Host collects are unchanged. */
#define RTLSDR_GPU_FLAG_ASYNC_REPORT 2u
/* cfg.flags: rtlsdr_gpu_scan_submit() accepts len < buf_len like the reference accepts a short rtlsdr_read_sync
 * (rtl_power.c:657-659: it warns and processes the whole buffer): the handle keeps the reference's per-hop
 * tunes[i].buf8 (tune_count x buf_len host bytes, zero at init where the reference's malloc leaves garbage), a
 * short read replaces its first len bytes, the rest is the hop's previous read.  Costs one extra host copy per
 * submit; without the flag a short len is RTLSDR_GPU_ERR_LENGTH. */
#define RTLSDR_GPU_FLAG_SHORT_READS 4u
/* cfg.flags: spectral kurtosis per bin (Nita & Gary 2010), which tells stationary noise (SK ~ 1) from
 * intermittent interference (SK > 1) and steady carriers (SK < 1) in bins whose averaged power looks the same.
 * Per hop and bin the handle also accumulates S2 = sum pw^2, pw = re^2 + im^2 being the per-block value the
 * power bins (S1) sum, exactly as an unsigned 128-bit value; rtlsdr_gpu_scan_collect_sk() reports it with
 *   SK = (M+1)/(M-1) * (M * S2 / S1^2 - 1),   M = samples / downsample (FFT blocks of the interval),
 * evaluated in IEEE doubles in exactly this order without contraction (rtlsdr_b200/csrc/sk.cuh), a quiet NaN
 * when M < 2 or S1 = 0.  Not with peak_hold, bin_e = 0 (rms) or RTLSDR_GPU_FLAG_ASYNC_REPORT
 * (RTLSDR_GPU_ERR_CONFIG at init); on such a handle merge_device() and collect_device() return
 * RTLSDR_GPU_ERR_CONFIG (they do not carry S2): use collect_sk_device() and merge_sk_device(), which do, and
 * collect_sk_csv() / format_sk_csv_device() for the SK rows' text.  Every other collect also zeroes S2. */
#define RTLSDR_GPU_FLAG_SPECTRAL_KURTOSIS 8u

/* ---- lifecycle --------------------------------------------------------- */

/* Allocates device state for tune_count hops; all accumulators start at 0
 * like frequency_range() leaves tunes[i].avg (rtl_power.c:521-523). */
RTLSDR_GPU_API int rtlsdr_gpu_scan_init(const rtlsdr_gpu_scan_cfg_t *cfg, rtlsdr_gpu_scan_t **out);
RTLSDR_GPU_API void rtlsdr_gpu_scan_close(rtlsdr_gpu_scan_t *h);

/* ---- the hot path ------------------------------------------------------ */

/*
 * One hop visit: replaces rtl_power.c:660-718 for tunes[hop] given the bytes
 * rtlsdr_read_sync() delivered (rtl_power.c:657).  (buf, len) has the shape of
 * rtlsdr_read_async_cb_t (rtl-sdr.h:472).  The bytes are copied into a pinned,
 * double-buffered staging ring before returning; host-to-device copy and
 * kernels run asynchronously.  len must equal buf_len (the reference processes
 * the full buffer even after a short read, rtl_power.c:658-659, so callers pass
 * the whole buffer they own) unless RTLSDR_GPU_FLAG_SHORT_READS is set, which
 * reproduces that behaviour inside the library.
 */
RTLSDR_GPU_API int rtlsdr_gpu_scan_submit(rtlsdr_gpu_scan_t *h, int hop, const uint8_t *buf, uint32_t len);

/*
 * Many hop visits whose bytes already live in host memory obtained from
 * rtlsdr_gpu_scan_host_alloc() (pinned): read (pass p, hop hop_first + k) is at
 * buf + p * pass_stride + k * hop_stride, k < hop_count, p < passes.  The
 * bytes are copied to the device without the intermediate ring copy.
 *
 * Buffer lifetime: the call returns while its host-to-device copies are still
 * queued (on a copy stream of the handle, possibly behind the previous batch's
 * kernels).  `buf` must stay valid AND unmodified until rtlsdr_gpu_scan_sync() /
 * any collect() into host memory returns, or until an event the caller records
 * on rtlsdr_gpu_scan_get_stream() AFTER this call has completed (the handle's
 * stream waits for every copy before the kernel that consumes it).  Refilling
 * the same pinned buffer for the next interval without such a wait corrupts
 * the reads that have not crossed PCIe yet.
 */
RTLSDR_GPU_API int rtlsdr_gpu_scan_submit_batch(rtlsdr_gpu_scan_t *h, int hop_first, int hop_count,
		int passes, const uint8_t *buf, int64_t pass_stride, int64_t hop_stride);

/*
 * Hop visits in ANY order (randomised hopping, the reference's TODO list
 * src/rtl_power.c:29-36): read i is buf_len bytes at buf + i * stride and
 * belongs to hop hops[i]; a hop may appear any number of times.  Bins are
 * int64 sums / maxima (rtl_power.c:708-716), so the result does not depend on
 * the order.  `buf` is pinned host memory (rtlsdr_gpu_scan_host_alloc); same
 * lifetime rule as rtlsdr_gpu_scan_submit_batch.  `hops` is consumed before
 * the call returns.
 */
RTLSDR_GPU_API int rtlsdr_gpu_scan_submit_reads(rtlsdr_gpu_scan_t *h, int n_reads, const int32_t *hops,
		const uint8_t *buf, int64_t stride);

/* Same layout, but `dev_buf` is device memory on cfg.device (16-byte aligned,
 * strides multiples of 16).  Used for device-resident replay (roofline runs). */
RTLSDR_GPU_API int rtlsdr_gpu_scan_submit_device(rtlsdr_gpu_scan_t *h, int hop_first, int hop_count,
		int passes, const void *dev_buf, int64_t pass_stride, int64_t hop_stride);

/* Push everything staged so far to the device and launch it (asynchronous). */
RTLSDR_GPU_API int rtlsdr_gpu_scan_flush(rtlsdr_gpu_scan_t *h);
/* Block until all submitted work has finished on the device. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_sync(rtlsdr_gpu_scan_t *h);

/*
 * Report for one hop: replaces what csv_dbm() reads and resets
 * (rtl_power.c:730-764).  Blocks until all submitted work for the handle is
 * done.
 *   avg     [1<<bin_e]  raw int64 sums / peaks in natural FFT order, i.e.
 *                       tunes[hop].avg BEFORE csv_dbm's DC-nuke and half swap
 *                       (may be NULL)
 *   samples             tunes[hop].samples (may be NULL)
 *   db      [rtlsdr_gpu_scan_db_count()] the doubles csv_dbm prints after the
 *                       4-column prefix: bins i1..i2 of the swapped spectrum
 *                       followed by the re-associated duplicate of bin i2
 *                       (rtl_power.c:747-760) (may be NULL)
 * Afterwards the hop's accumulators and sample count are zero
 * (rtl_power.c:761-764).
 *
 * cfg.iir_alpha > 0 ("-s iir": the reference parses it, rtl_power.c:820-825, and lists
 * "continuous IIR smoothing" as a TODO, :29-36; it never defined it, so this is the
 * definition): `db` holds 10*log10(s), s being an exponential moving average across
 * reports of the linear value csv_dbm takes the logarithm of, d = avg / rate / samples:
 * s = d at a bin's first report, s += alpha * (d - s) afterwards, all in IEEE doubles
 * without contraction; a report of a hop without samples leaves s alone and prints d.
 * The duplicated last column repeats the smoothed last bin.  `avg` / `samples` are
 * never smoothed.
 */
RTLSDR_GPU_API int rtlsdr_gpu_scan_collect(rtlsdr_gpu_scan_t *h, int hop, int64_t *avg, int *samples, double *db);

/* All hops at once: avg [tune_count << bin_e], samples [tune_count],
 * db [tune_count * db_count]; any may be NULL.  Zeroes every hop. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_collect_all(rtlsdr_gpu_scan_t *h, int64_t *avg, int *samples, double *db);

/* collect_all() plus the spectral-kurtosis report of a RTLSDR_GPU_FLAG_SPECTRAL_KURTOSIS handle (any pointer may
 * be NULL): s2 [tune_count << bin_e][2] the raw 128-bit sums of pw^2 as (lo, hi) words in natural FFT order like
 * `avg`, sk [tune_count * db_count] the SK row of every hop in the dB row's layout -- bin 0 takes bin 1's
 * moments (csv_dbm's DC nuke), half swap, crop, duplicate of bin i2 -- so SK columns line up with dB columns
 * (never smoothed by iir_alpha).  Zeroes every hop.  RTLSDR_GPU_ERR_CONFIG on a handle without the flag. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_collect_sk(rtlsdr_gpu_scan_t *h, int64_t *avg, int *samples, double *db,
		uint64_t *s2, double *sk);

/* Same, into device buffers (for the per-interval NCCL gather); asynchronous
 * on the handle's stream, no host synchronisation. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_collect_device(rtlsdr_gpu_scan_t *h, void *dev_avg, void *dev_samples, void *dev_db);

/* collect_device() for a RTLSDR_GPU_FLAG_SPECTRAL_KURTOSIS handle: the same three outputs plus S2 (dev_s2, u64
 * [tune_count << bin_e][2] (lo, hi), 8-byte aligned) and the SK rows (dev_sk, double [tune_count][db_count]) as
 * collect_sk() writes them; any pointer may be NULL.  Read-and-zero of S1, the counts and S2.  Asynchronous on the
 * handle's stream, no host synchronisation; destinations may be peer-mapped memory of another GPU.
 * RTLSDR_GPU_ERR_CONFIG on a handle without the flag. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_collect_sk_device(rtlsdr_gpu_scan_t *h, void *dev_avg, void *dev_samples,
		void *dev_db, void *dev_s2, void *dev_sk);

/*
 * Reads of the SAME hops processed by several handles (e.g. one per GPU, each fed a share of the reads of a
 * single-hop scan): fold `sets` external accumulator sets into this handle's.  Set s is what
 * rtlsdr_gpu_scan_collect_device() wrote for a handle with the same configuration: raw bins int64
 * [tune_count << bin_e] at dev_avg + s * set_stride and sample counts int32 [tune_count] at
 * dev_samples + s * set_stride (bytes; 8-byte aligned).  Bins are added, or maximised under peak_hold; counts are
 * added -- exactly what the reference's accumulation does read by read (rtl_power.c:708-717), so a following
 * collect() of this handle returns bit-identical bins, counts and dB to ONE handle that had seen all the reads.
 * Asynchronous on the handle's stream; the external memory may be device memory, a peer mapping of another GPU
 * or pinned host memory from rtlsdr_gpu_scan_host_alloc() (what another handle's collect_all() filled), and must
 * stay valid until the work has run.  (iir_alpha: smoothing state is only updated by this handle's own collects.)
 */
RTLSDR_GPU_API int rtlsdr_gpu_scan_merge_device(rtlsdr_gpu_scan_t *h, const void *dev_avg, const void *dev_samples,
		int sets, int64_t set_stride);

/* merge_device() for a RTLSDR_GPU_FLAG_SPECTRAL_KURTOSIS handle: set s also has its S2 (what collect_sk_device()
 * wrote, u64 [tune_count << bin_e][2], 8-byte aligned) at dev_s2 + s * set_stride.  S1 and the counts are added like
 * merge_device() does, S2 as an exact unsigned 128-bit sum (a carry out of the low word goes into the high word), so
 * a following collect_sk() / collect_sk_csv() returns bit-identical bins, S2 and SK rows to ONE handle that had seen
 * all the reads.  Same argument and alignment checks as merge_device(); RTLSDR_GPU_ERR_CONFIG without the flag. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_merge_sk_device(rtlsdr_gpu_scan_t *h, const void *dev_avg, const void *dev_samples,
		const void *dev_s2, int sets, int64_t set_stride);

/*
 * Soft-AGC statistics of hop `hop` since its last collect (needs RTLSDR_GPU_FLAG_LEVEL_STATS):
 * overload = bytes equal to 0 or 255 (0 dBFS), high_level = bytes < 64 or > 191 (-6 dBFS), as
 * softagc() counts them per buffer (src/librtlsdr.c:3299-3306), bytes = bytes looked at.
 * Blocks until submitted work is done; collect() of the hop resets the counters.
 */
RTLSDR_GPU_API int rtlsdr_gpu_scan_level_stats(rtlsdr_gpu_scan_t *h, int hop, uint64_t *overload,
		uint64_t *high_level, uint64_t *bytes);

/* ---- CSV rows ------------------------------------------------------------ */

/*
 * The report as rtl_power prints it, formatted on the GPU: per row
 * "<stamp>low, high, step, samples, dB, ..., dB\n" (rtl_power.c:739-760, 995-998), byte-identical to the host's
 * printf("%i, %i, %.2f, %i, " "%.2f, " ... "%.2f\n") of the same values (host/rtl_power_plan.c rp_csv_row).
 * `stamp` is copied verbatim in front of every row (rtl_power prints "date, time, ", so pass it with the
 * separator); it is a NUL-terminated string of fewer than 128 bytes.
 *
 * The formatter prints what it is given: -inf for a bin of 0, nan / -nan with the sign bit of the NaN (a hop
 * without samples), -0.00 for values that round to zero from below.  A dB value whose text would be wider than
 * 7 characters (wider than "-999.99" or "9999.99") does not occur in a report, whose dB values lie in (-187, 190);
 * met in a caller's buffer it is an error, never text.
 */

/* The row table: row r prints low[r], high[r] and `step` (rtl_power_plan.c rp_csv_columns; 0 <= step < 2^31).
 * Copied to the device once.  collect_csv() prints rows [0, tune_count); the table may have more rows for
 * format_csv_device() (e.g. rank 0 of a sharded sweep prints every rank's hops).  Synchronous. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_set_csv_columns(rtlsdr_gpu_scan_t *h, int rows, const int32_t *low,
		const int32_t *high, double step);
/* Bytes that `rows` rows with a stamp of stamp_len bytes can take at most: the text buffer size collect_csv() and
 * format_csv_device() require.  rows * (stamp_len + 56 + 9 * db_count); negative = error. */
RTLSDR_GPU_API int64_t rtlsdr_gpu_scan_csv_capacity(const rtlsdr_gpu_scan_t *h, int rows, size_t stamp_len);
/*
 * collect_all()'s read-and-zero of every hop, returning the rows' text instead of the dB doubles: `text`
 * receives *len bytes (no NUL).  cap is checked against csv_capacity(tune_count) before anything is touched
 * (RTLSDR_GPU_ERR_LENGTH); without a table of at least tune_count rows the call is RTLSDR_GPU_ERR_CONFIG.  On
 * any error the accumulators are left as they were.  Blocks until the text is in `text`.
 */
RTLSDR_GPU_API int rtlsdr_gpu_scan_collect_csv(rtlsdr_gpu_scan_t *h, const char *stamp, char *text, size_t cap,
		size_t *len);
/*
 * The rows [row_first, row_first + rows) of the table for a report in device memory: dB row r at
 * dev_db + r * db_stride doubles (db_stride >= db_count, 8-byte aligned), its count at dev_samples[r] (int32) --
 * the layout collect_device() writes for a handle with the same configuration.  The text goes to dev_text
 * (cap >= csv_capacity(rows), else RTLSDR_GPU_ERR_LENGTH) and its length to *dev_len (int64, 8-byte aligned);
 * a value outside the formatter's domain makes *dev_len = -1 (all ones).  Asynchronous on the handle's stream;
 * the caller orders it after the writer of the report and before the reader of the text.
 */
RTLSDR_GPU_API int rtlsdr_gpu_scan_format_csv_device(rtlsdr_gpu_scan_t *h, const char *stamp, int row_first,
		int rows, const void *dev_db, int64_t db_stride, const void *dev_samples, void *dev_text, size_t cap,
		void *dev_len);

/*
 * The spectral-kurtosis rows of a RTLSDR_GPU_FLAG_SPECTRAL_KURTOSIS handle (RTLSDR_GPU_ERR_CONFIG without the flag):
 * per row the power row's prefix "<stamp>low, high, step, samples, ", then the SK values as printf("%.4f"), joined
 * by ", " and ended by "\n"; a NaN of either sign (SK undefined) prints "nan".  SK <= M + 1 < 2^31 + 1, so a value
 * takes at most 15 characters ("2147483649.0000"); a wider one met in a caller's buffer is an error, never text.
 */
/* Bytes of `rows` SK rows at their widest: rows * (stamp_len + 56 + 17 * db_count); negative = error. */
RTLSDR_GPU_API int64_t rtlsdr_gpu_scan_sk_csv_capacity(const rtlsdr_gpu_scan_t *h, int rows, size_t stamp_len);
/* format_csv_device() for SK rows: row r's values at dev_sk + r * sk_stride doubles (the layout collect_sk_device()
 * writes), its count at dev_samples[r]; cap >= sk_csv_capacity(rows), *dev_len = -1 for a value outside the
 * formatter's domain.  Asynchronous on the handle's stream. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_format_sk_csv_device(rtlsdr_gpu_scan_t *h, const char *stamp, int row_first,
		int rows, const void *dev_sk, int64_t sk_stride, const void *dev_samples, void *dev_text, size_t cap,
		void *dev_len);
/* collect_csv() plus the SK rows: the power rows' text to `text` (*len bytes, cap >= csv_capacity(tune_count)) and
 * the SK rows' text to `sk_text` (*sk_len bytes, sk_cap >= sk_csv_capacity(tune_count)), with the same read-and-zero
 * of S1, the counts and S2; only the text crosses PCIe.  On any error the accumulators are left as they were.  Blocks
 * until both texts are in host memory. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_collect_sk_csv(rtlsdr_gpu_scan_t *h, const char *stamp, char *text, size_t cap,
		size_t *len, char *sk_text, size_t sk_cap, size_t *sk_len);

/* ---- multi-GPU report hand-off ----------------------------------------- */

/*
 * With rtlsdr_gpu_scan_collect_device() every GPU's report epilogue can store straight into ONE GPU's memory
 * (NVLink peer mapping).  These two calls are the rest of the "gather": a 32-bit flag per (buffer, writer),
 * stored with system-scope release semantics by a one-thread kernel on `cuda_stream` (behind the epilogue), and a
 * wait for `count` consecutive flags to reach `value` (wrap-safe compare) by a kernel whose threads sleep between
 * polls, so it takes no issue slots from the transform kernels it runs beside.  The wait gives up after
 * timeout_ms (0 = 10 s) and then sets *dev_timed_out (may be NULL) instead of hanging the GPU.  Both launch on the
 * CURRENT device; flags may live in peer-mapped memory.  No reference counterpart (the reference has one device).
 * Caution (CUDA lazy module loading): while a wait is pending, the FIRST launch of any kernel the process has not
 * used yet may block until the wait ends; these two load each other before launching, callers should have run
 * whatever else the waited-for work needs (e.g. one submit + collect_device) at least once beforehand.
 */
RTLSDR_GPU_API int rtlsdr_gpu_scan_flag_signal(void *cuda_stream, void *dev_flag, uint32_t value);
/* the same value into up to 32 flags at unrelated addresses with ONE launch (dev_flags is a host array of device pointers) */
RTLSDR_GPU_API int rtlsdr_gpu_scan_flag_signal_many(void *cuda_stream, void *const *dev_flags, int count, uint32_t value);
RTLSDR_GPU_API int rtlsdr_gpu_scan_flag_wait(void *cuda_stream, const void *dev_flags, int count, uint32_t value,
		uint32_t timeout_ms, void *dev_timed_out);

/* ---- helpers ----------------------------------------------------------- */

/* Number of doubles per hop that collect() writes to `db` (= i2 - i1 + 2). */
RTLSDR_GPU_API int rtlsdr_gpu_scan_db_count(const rtlsdr_gpu_scan_t *h);
/* Pinned host memory for submit_batch() and fast collect(). */
RTLSDR_GPU_API void *rtlsdr_gpu_scan_host_alloc(size_t bytes);
RTLSDR_GPU_API void rtlsdr_gpu_scan_host_free(void *p);
/* Run the handle's work on a caller-owned CUDA stream (cudaStream_t passed as
 * void*); NULL restores the handle's own stream. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_set_stream(rtlsdr_gpu_scan_t *h, void *cuda_stream);
/* The stream the handle currently launches on (cudaStream_t as void*), e.g. to record events on it
 * or to make other streams wait for it. */
RTLSDR_GPU_API void *rtlsdr_gpu_scan_get_stream(rtlsdr_gpu_scan_t *h);
/* The stream rtlsdr_gpu_scan_collect_device() puts its report on: the handle's stream, or the separate report
 * stream of RTLSDR_GPU_FLAG_ASYNC_REPORT. */
RTLSDR_GPU_API void *rtlsdr_gpu_scan_get_report_stream(rtlsdr_gpu_scan_t *h);
/* Host table builders using the reference's expressions: Sinewave
 * (rtl_power.c:247-261; out[(1<<bin_e)*3/4]) and window_coefs for a -w name
 * (rtl_power.c:329-408, 826-843, 985-988; out[n]).  window returns -1 for an
 * unknown name (table is then rectangle, as the reference silently does). */
RTLSDR_GPU_API void rtlsdr_gpu_scan_sine_table(int bin_e, int16_t *out);
RTLSDR_GPU_API int rtlsdr_gpu_scan_window(const char *name, int n, int32_t *out);
/* Counters since init: kernels launched, bytes copied H2D / D2H. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_stats(const rtlsdr_gpu_scan_t *h, uint64_t *kernel_launches,
		uint64_t *h2d_bytes, uint64_t *d2h_bytes);
/* Device time in milliseconds of the main transform kernel(s) launched since
 * the previous call (CUDA events on the launching stream), and their count. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_kernel_time(rtlsdr_gpu_scan_t *h, double *ms, uint64_t *launches);
/* Time only every `every`-th transform (0 = off).  Event records between two kernels keep the
 * second from being launched programmatically dependent on the first, so long runs sample. */
RTLSDR_GPU_API int rtlsdr_gpu_scan_set_timing(rtlsdr_gpu_scan_t *h, int every);
RTLSDR_GPU_API const char *rtlsdr_gpu_scan_strerror(int err);
/* Text of the last CUDA error seen by this handle ("" if none). */
RTLSDR_GPU_API const char *rtlsdr_gpu_scan_last_cuda_error(const rtlsdr_gpu_scan_t *h);

#ifdef __cplusplus
}
#endif
#endif /* RTLSDR_GPU_SCAN_H */
