/*
 * scan_kernels.cuh -- sm_100a kernels for rtl_power's per-hop scan pipeline.
 *
 * Reference semantics reproduced bit-for-bit (file:line in /root/reference):
 *   u8 -> int16 minus 127                      src/rtl_power.c:666-668
 *   boxcar decimation                          src/rtl_power.c:671-681
 *   fifth_order x downsample_passes            src/rtl_power.c:554-579, 628-634, 683-685
 *   generic_fir (9-tap droop compensation)     src/rtl_power.c:598-626, 687-690
 *   remove_dc over the whole read buffer       src/rtl_power.c:581-596, 692-693
 *   window multiply (int16 truncation)         src/rtl_power.c:695-706
 *   fix_fft: Q15 radix-2 DIT, FIX_MPY rounding,
 *            halving on every stage             src/rtl_power.c:263-327
 *   |X|^2 int64 accumulate / peak hold         src/rtl_power.c:636-640, 708-716
 *   rms_power for 1-bin hops                   src/rtl_power.c:410-436
 *   csv_dbm numeric half (DC nuke, half swap,
 *            crop, dB)                          src/rtl_power.c:722-760
 *
 * Design (B200-first, no tensor cores: this is integer butterfly work):
 *  - A complex int16 sample is ONE 32-bit register (re low, im high), the same
 *    bytes as the reference's interleaved int16 buffer.
 *  - Each thread keeps 16 samples in registers and runs 4 consecutive radix-2
 *    stages on them ("register-blocked radix-16", with the reference's per-stage
 *    rounding, halving and int16 wrap intact -- no algebraic radix-4).  A CTA of
 *    256 threads therefore owns a 4096-sample working set; three passes with two
 *    padded shared-memory transposes cover 12 stages.
 *  - Input arrives with 16-byte cp.async (LDGSTS) copies into a double-buffered
 *    shared staging area; the next read is in flight while the current one is
 *    transformed.
 *  - |X|^2 is accumulated in registers across all the reads a CTA owns and
 *    flushed once with 64-bit atomics.
 */
#pragma once
#include "scan_compat.cuh"
#include "sk.cuh"

/* Micro-variants of the transform kernel, all measured on B200 (profiles/r02d_small_kernel_ab.txt, config 5):
 * window coefficients in registers +0.4 %, IDP.4A front end +0.8 %, packed "b" operands after a transpose +0.5 %,
 * together +1.9 %.  (Tried and measured slower: 16-byte transpose stores -1.2 %, DC partial sums hoisted in front of
 * the per-read barrier -0.5 %, IMAD.HI products: ptxas splits the chained form.)  tools/ab_run.sh builds both sides. */
#ifndef RSCAN_WIN_REGS
#define RSCAN_WIN_REGS 1
#endif
#ifndef RSCAN_FRONT_IDP
#define RSCAN_FRONT_IDP 1
#endif
#ifndef RSCAN_PACKED_B
#define RSCAN_PACKED_B 1
#endif

namespace rscan {

typedef uint32_t c16; /* packed complex int16: re = bits 0..15, im = bits 16..31 */

constexpr int kThreads = 256;                 /* threads per CTA */
constexpr int kPts     = 16;                  /* samples per thread */
constexpr int kWS      = kThreads * kPts;     /* 4096-sample working set */
constexpr int kStageBytes = 16384;            /* one staging slot */
constexpr int kXchWords   = kWS + kWS / 16;   /* transpose buffer, 1 pad word per 16 */

/* ---- packed helpers ---------------------------------------------------- */

SCAN_DEV int c16_re(c16 v) { return (int)(int16_t)(uint16_t)(v & 0xFFFFu); }
SCAN_DEV int c16_im(c16 v) { return ((int32_t)v) >> 16; }
SCAN_DEV c16 c16_pack(int re, int im) { return ((uint32_t)re & 0xFFFFu) | ((uint32_t)im << 16); }

/* FIX_MPY (rtl_power.c:263-269): ((a*b)>>14 ; (c>>1)+(c&1)) == (a*b + 2^14) >> 15 */
SCAN_DEV int fix_mpy(int w, int x) { return (w * x + 16384) >> 15; }

/*
 * One radix-2 DIT butterfly of fix_fft (rtl_power.c:309-321) on packed values.
 * (wr, wi) is the twiddle AFTER its halving (wr = Sinewave[j+N/4] >> 1,
 * wi = (-Sinewave[j]) >> 1, rtl_power.c:305-308).  tr/ti cannot leave int16
 * (|w| <= 16384); the four q +- t results wrap to int16 in c16_pack.
 * Reference form; the hot loops use the high-half form below.
 */
SCAN_DEV void butterfly(c16 &a, c16 &b, int wr, int wi)
{
	const int br = c16_re(b), bi = c16_im(b);
	const int tr = fix_mpy(wr, br) - fix_mpy(wi, bi);
	const int ti = fix_mpy(wr, bi) + fix_mpy(wi, br);
	const int qr = c16_re(a) >> 1, qi = c16_im(a) >> 1;
	b = c16_pack(qr - tr, qi - ti);
	a = c16_pack(qr + tr, qi + ti);
}

/*
 * High-half ("X") form used inside a pass: a component v lives in the TOP 16
 * bits of a 32-bit register, the low 16 bits are don't-care.  Then
 *   - the int16 wrap of q +- t is the natural mod-2^32 wrap of x + (t << 16),
 *   - the arithmetic halving q = v >> 1 is x >> 1 (the bit shifted out lands in
 *     the don't-care half and can never carry back up),
 *   - the sign-extended multiplicand is x >> 16.
 * Per butterfly: 4 IMAD + 4 (t<<16 +- q) on the FMA pipe, 2+2+2+2 shifts /
 * shift-adds on the ALU pipe: 8 + 8, balanced for the two half-rate integer
 * pipes of an sm_100 SM sub-partition (tools/ubench.cu measures both at 64
 * lanes/clk/SM and shows they dual-issue).
 */
struct X2 {
	int re, im;
};

SCAN_DEV X2 x_unpack(c16 v)
{
	X2 x;
	x.re = (int)(v << 16);
	x.im = (int)v; /* low half = re bits: don't care */
	return x;
}

SCAN_DEV c16 x_pack(X2 x)
{
	return __byte_perm((uint32_t)x.re, (uint32_t)x.im, 0x7632); /* one PRMT: bytes 2,3 of re | bytes 2,3 of im */
}

/* sign-extended low / high half of a packed value: one PRMT (sign-replicating selector) / one shift */
SCAN_DEV int c16_re_fast(c16 v)
{
#ifdef SCAN_EMU
	return (int)(int16_t)(uint16_t)(v & 0xFFFFu);
#else
	int r;
	asm("prmt.b32 %0, %1, 0, 0x9910;" : "=r"(r) : "r"(v));
	return r;
#endif
}

SCAN_DEV void butterfly_x(X2 &a, X2 &b, int wr, int wi);

/* the same butterfly when the lower ("b") element is still PACKED (first stage after a transpose):
 * its components are extracted straight from the packed word, the X-form unpack is skipped */
SCAN_DEV void butterfly_x_packed_b(X2 &a, X2 &b, c16 vb, int wr, int wi)
{
	const int br = c16_re_fast(vb), bi = ((int)vb) >> 16;
	const int tr = ((wr * br + 16384) >> 15) - ((wi * bi + 16384) >> 15);
	const int ti = ((wr * bi + 16384) >> 15) + ((wi * br + 16384) >> 15);
	const int hr = a.re >> 1, hi = a.im >> 1;
	b.re = hr - tr * 65536;
	b.im = hi - ti * 65536;
	a.re = hr + tr * 65536;
	a.im = hi + ti * 65536;
}

SCAN_DEV void butterfly_x(X2 &a, X2 &b, int wr, int wi)
{
	const int br = b.re >> 16, bi = b.im >> 16;
	const int tr = ((wr * br + 16384) >> 15) - ((wi * bi + 16384) >> 15);
	const int ti = ((wr * bi + 16384) >> 15) + ((wi * br + 16384) >> 15);
	const int hr = a.re >> 1, hi = a.im >> 1;
	b.re = hr - tr * 65536;
	b.im = hi - ti * 65536;
	a.re = hr + tr * 65536;
	a.im = hi + ti * 65536;
}

/* twiddle (wr, 0): first group of every stage (angle 0) */
SCAN_DEV void butterfly_x_re(X2 &a, X2 &b, int wr)
{
	const int tr = (wr * (b.re >> 16) + 16384) >> 15;
	const int ti = (wr * (b.im >> 16) + 16384) >> 15;
	const int hr = a.re >> 1, hi = a.im >> 1;
	b.re = hr - tr * 65536;
	b.im = hi - ti * 65536;
	a.re = hr + tr * 65536;
	a.im = hi + ti * 65536;
}

/* twiddle (0, wi): the quarter-turn group (Sinewave[N/2] = 0) */
SCAN_DEV void butterfly_x_im(X2 &a, X2 &b, int wi)
{
	const int tr = -((wi * (b.im >> 16) + 16384) >> 15);
	const int ti = (wi * (b.re >> 16) + 16384) >> 15;
	const int hr = a.re >> 1, hi = a.im >> 1;
	b.re = hr - tr * 65536;
	b.im = hi - ti * 65536;
	a.re = hr + tr * 65536;
	a.im = hi + ti * 65536;
}

/* real_conj + accumulate / peak hold (rtl_power.c:636-640, 708-716) on a register accumulator;
 * re^2 + im^2 <= 2^31 fits an unsigned 32-bit value.  (A mad.wide spelling with the 64-bit
 * accumulator as addend is split again by ptxas into multiply + add-with-carry: no gain.) */
template <bool PEAK>
SCAN_DEV void accumulate_power(unsigned long long &acc, int re, int im)
{
	const unsigned pw = (unsigned)(re * re) + (unsigned)(im * im);
	if constexpr (PEAK)
		acc = acc > pw ? acc : (unsigned long long)pw;
	else
		acc += pw;
}

/* ---- working-set geometry ---------------------------------------------- */

/* Position (0..4095) of register r of thread t while pass K is in registers:
 * r supplies bits [4K, 4K+4) of the position, t supplies the rest. */
template <int K>
SCAN_DEV int pos(int t, int r)
{
	constexpr int sh = 4 * K;
	return ((t >> sh) << (sh + 4)) | (r << sh) | (t & ((1 << sh) - 1));
}

SCAN_DEV int xch_idx(int p) { return p + (p >> 4); }

/* xch_idx(pos<K>(t, r)) == xch_idx(pos<K>(t, 0)) + xch_step<K>() * r for every t: the three fields of pos<K> are
 * disjoint, so p >> 4 splits over them, and r adds r << 4K to p and r << (4K - 4) to p >> 4 (nothing for K = 0).
 * exchange_pk addresses with one per-thread base plus a compile-time offset per register: pos<K> composes with `|`,
 * through which ptxas cannot distribute the padding term, and would rebuild every address. */
template <int K>
SCAN_DEV constexpr int xch_step()
{
	return K == 0 ? 1 : (1 << (4 * K)) + (1 << (4 * K - 4));
}

SCAN_DEV constexpr int brev4(int r)
{
	return ((r & 1) << 3) | ((r & 2) << 1) | ((r & 4) >> 1) | ((r & 8) >> 3);
}

SCAN_DEV int brev_bits(unsigned v, int bits)
{
	return bits <= 0 ? 0 : (int)(__brev(v) >> (32 - bits));
}

/*
 * Passes of the engine.  LE = number of radix-2 stages the engine runs on the
 * low LE bits of the position (LE <= 12).  Pass K covers stages
 * [4K, min(4K+4, LE)).  TW::get<K>(s, pa) returns the halved twiddle of stage s
 * for the butterfly whose upper ("a") element sits at position pa.
 * TW::kTrivial: pass-0 groups 0 and 2^(s-1) have twiddles (wr, 0) and (0, wi)
 * (true for every table sine_table() builds; checked by the host at init).
 */
template <int K, int LE, class TW>
SCAN_DEV void run_pass(X2 (&x)[kPts], int t, const TW &tw, const c16 *packed = nullptr)
{
	constexpr int s0 = 4 * K;
	constexpr int ns = (LE - s0) < 4 ? (LE - s0) : 4;
#pragma unroll
	for (int b = 0; b < ns; ++b) {
#pragma unroll
		for (int r = 0; r < kPts; ++r) {
			if ((r & (1 << b)) == 0) {
				const int2 w = tw.template get<K>(s0 + b, pos<K>(t, r));
				const int g = r & ((1 << b) - 1);
				if (RSCAN_PACKED_B && K > 0 && b == 0 && packed) /* x[r | 1] has not been unpacked: take it from the packed word */
					butterfly_x_packed_b(x[r], x[r | 1], packed[r | 1], w.x, w.y);
				else if (K == 0 && TW::kTrivial && g == 0)
					butterfly_x_re(x[r], x[r | (1 << b)], w.x);
				else if (K == 0 && TW::kTrivial && b > 0 && g == (1 << (b - 1)))
					butterfly_x_im(x[r], x[r | (1 << b)], w.y);
				else
					butterfly_x(x[r], x[r | (1 << b)], w.x, w.y);
			}
		}
	}
}

/*
 * Transpose through shared memory between two passes.  LEAD = true puts a
 * barrier in front (the buffer may still be read by slower threads).  The
 * streaming kernel instead alternates between two buffers on every exchange:
 * a buffer is rewritten only two exchanges later and the barrier of the
 * exchange in between already orders those accesses, so one barrier suffices.
 */
struct BlockBar { /* the 256 transform threads are the whole CTA */
	SCAN_DEV void sync() const { __syncthreads(); }
};
struct GroupBar { /* the transform threads are one role of a warp-specialised CTA: named barrier `id` */
	int id, count;
	SCAN_DEV void sync() const { named_bar_sync(id, count); }
};

/* tw_ = thread id whose pass-KA positions the registers hold, t = this thread's id in pass KB
 * (they differ only after a permuted front end, see front_thread_map) */
template <int KA, int KB, bool LEAD, class BAR = BlockBar>
SCAN_DEV void exchange(X2 (&x)[kPts], c16 *xch, int tw_, int t, const BAR &bar = BAR())
{
	/* the large path's transpose keeps per-register addresses: the base + offset form of exchange_pk measured 0.7 %
	 * slower on config 4 here */
	if (LEAD)
		bar.sync();
#pragma unroll
	for (int r = 0; r < kPts; ++r)
		xch[xch_idx(pos<KA>(tw_, r))] = x_pack(x[r]);
	bar.sync();
#pragma unroll
	for (int r = 0; r < kPts; ++r)
		x[r] = x_unpack(xch[xch_idx(pos<KB>(t, r))]);
}

/* Transpose whose odd registers stay packed in `pk` (they are the "b" elements of the next pass's first stage,
 * butterfly_x_packed_b extracts them without the X-form unpack); even registers are unpacked as usual. */
template <int KA, int KB, class BAR>
SCAN_DEV void exchange_pk(X2 (&x)[kPts], c16 (&pk)[kPts], c16 *xch, int tw_, int t, const BAR &bar)
{
	const int st = xch_idx(pos<KA>(tw_, 0)), ld = xch_idx(pos<KB>(t, 0));
#pragma unroll
	for (int r = 0; r < kPts; ++r)
		xch[st + xch_step<KA>() * r] = x_pack(x[r]);
	bar.sync();
#pragma unroll
	for (int r = 0; r < kPts; ++r) {
		pk[r] = xch[ld + xch_step<KB>() * r];
		if (!RSCAN_PACKED_B || (r & 1) == 0)
			x[r] = x_unpack(pk[r]);
	}
}

/*
 * Which samples a thread takes in the front end.  Natural choice: thread t holds positions
 * 16t + r, i.e. the samples n = (brev4(r) << (L-4)) + bitrev(t) -- but then the lanes of a warp
 * read 16-bit samples 16 bytes apart (4-way bank conflicts on every front-end load, 8-way on
 * the 32-bit loads of a decimated image).  For L = 12 the lanes instead take
 *   g = brev5(lane) << 3 | (brev5(lane)[4:3] ^ warp[1:0]) << 1 | warp[2]
 * as the low 8 sample bits: still a bijection, the 32 lanes now hit 32 different banks on the
 * sample and window loads, and the positions they hold, 16 * brev8(g) + r, are congruent to
 * 16 * lane + r modulo 512, so the first transpose's stores stay conflict-free.
 * Returns the low sample bits; t0 = the thread id whose natural positions this thread holds in pass 0.
 */
template <int L>
SCAN_DEV int front_thread_map(int t, int &t0)
{
	if constexpr (L == 12) {
		const int b = brev_bits((unsigned)(t & 31), 5), w = t >> 5;
		const int g = (b << 3) | ((((b >> 3) & 3) ^ (w & 3)) << 1) | (w >> 2);
		t0 = brev_bits((unsigned)g, 8);
		return g;
	} else {
		t0 = t;
		if constexpr (L >= 4)
			return brev_bits((unsigned)(t & ((1 << (L - 4)) - 1)), L - 4);
		return 0;
	}
}

/* Runs stages 0..LE-1; on return register r of thread t holds position
 * pos<(LE-1)/4>(t, r). */
template <int LE, class TW>
SCAN_DEV void engine_fft(X2 (&x)[kPts], c16 *xch, int t, const TW &tw)
{
	run_pass<0, LE>(x, t, tw);
	if constexpr (LE > 4) {
		exchange<0, 1, true>(x, xch, t, t);
		run_pass<1, LE>(x, t, tw);
	}
	if constexpr (LE > 8) {
		exchange<1, 2, true>(x, xch, t, t);
		run_pass<2, LE>(x, t, tw);
	}
}

/* Same, with two transpose buffers of kXchWords each; `flip` is the running
 * exchange parity (uniform across the CTA, carried across working sets). */
template <int LE, class TW, class BAR = BlockBar>
SCAN_DEV void engine_fft_db(X2 (&x)[kPts], c16 *xch2, int &flip, int t, const TW &tw, const BAR &bar = BAR(), int t0 = -1)
{
	if (t0 < 0)
		t0 = t; /* natural front end: the registers hold positions 16t + r */
	run_pass<0, LE>(x, t0, tw);
	c16 pk[kPts];
	if constexpr (LE > 4) {
		exchange_pk<0, 1, BAR>(x, pk, xch2 + flip * kXchWords, t0, t, bar);
		flip ^= 1;
		run_pass<1, LE>(x, t, tw, pk);
	}
	if constexpr (LE > 8) {
		exchange_pk<1, 2, BAR>(x, pk, xch2 + flip * kXchWords, t, t, bar);
		flip ^= 1;
		run_pass<2, LE>(x, t, tw, pk);
	}
}

template <int LE>
SCAN_DEV int last_pos(int t, int r)
{
	return pos<(LE - 1) / 4>(t, r);
}

/* ======================================================================== *
 *  Path 1: N <= 4096.  One CTA owns whole read buffers of one hop.          *
 * ======================================================================== */

struct PassTw {
	int2 w[15]; /* pass-0 twiddles: stage b, group g at w[(1<<b)-1+g] */
};

struct SmallParams {
	const uint8_t *base;        /* u8 reads, or (IN16) decimated c16 images */
	const long long *read_off;  /* byte offset of entry e from base; NULL = regular */
	long long regular_stride;   /* read_off == NULL: entry e at (e - entry_base) * regular_stride */
	int entry_base;             /* first entry of this launch (IN16 images / dc_sums are relative to it) */
	const int4 *segs;           /* IN16: (hop, first entry, entry count, -) */
	int n_segs;
	const int *hop_of;          /* u8 reads: hop of entry e, entries sorted by hop */
	int n_entries;              /* u8 reads: entries of this launch */
	int stagger_ns;             /* u8 reads: start delay of the second resident wave half (see the kernel) */
	long long *avg;             /* [tune_count << L] */
	long long *samples;         /* [tune_count] tunes[i].samples (rtl_power.c:717) */
	int samples_per_read;
	const int2 *tw;             /* [N/2] halved twiddles (wr, wi) */
	const int2 *twc;            /* [N-16] the same, per-stage compact: stage s >= 4, group m at (1<<s)-16+m */
	const uint16_t *win;        /* [N] low 16 bits of window_coefs */
	/* IN16 only: images of consecutive entries are contiguous, blocks_padded * N c16 each */
	const int *dc_ave;          /* [entry - entry_base][2]: int16 averages remove_dc subtracts (I, Q) */
	int l_len;                  /* buf_len / downsample (interleaved int16 count) */
	int n_blocks;               /* FFT blocks per read (rtl_power.c:695) */
	int blocks_padded;          /* >= n_blocks: image length / N (16-byte alignment padding for N = 2) */
	PassTw tw0;
};

template <int L>
struct SmallSmem {
	static constexpr int N = 1 << L;
	static constexpr int off_stage = 0;
	static constexpr int off_xch = 2 * kStageBytes;
	static constexpr int off_tw = off_xch + 2 * kXchWords * 4; /* two transpose buffers */
	static constexpr int tw_entries = N > 16 ? N - 16 : 1; /* stages 4..L-1, group m of stage s at (1<<s)-16+m */
	static constexpr int off_win = (off_tw + tw_entries * 8 + 15) & ~15; /* 16-byte aligned for cp.async */
	static constexpr int off_red = (off_win + N * 2 + 15) & ~15;
	static constexpr int off_dck = off_red + 16 * 8; /* after red[8 warps][2] */
	static constexpr int bytes = off_dck + 16;
};

template <int L>
struct TwSmall {
	static constexpr bool kTrivial = true;
	const int2 *tws;   /* shared: stage s >= 4, group m at (1<<s)-16+m -> consecutive lanes, consecutive words */
	const PassTw *tw0;
	template <int K>
	SCAN_DEV int2 get(int s, int pa) const
	{
		const int m = pa & ((1 << s) - 1);
		if constexpr (K == 0)
			return tw0->w[(1 << s) - 1 + m]; /* compile-time index: constant bank */
		else
			return tws[(1 << s) - 16 + m];
	}
};

/* the compact twiddles and the window -> shared memory, shared by the threads t = 0, 1, .. stride-1: asynchronous
 * 16-byte copies (the host pre-arranges the per-stage compact twiddle layout), so the caller's first input copies
 * overlap them; the caller waits for them and puts a barrier before the first use */
template <int L>
SCAN_DEV void load_tables(int2 *tws, uint16_t *wins, const int2 *twc, const uint16_t *win, int t, int stride)
{
	constexpr int N = 1 << L;
	if constexpr (N > 16) {
		for (int i = t; i < (N - 16) / 2; i += stride)
			cp_async16((uint8_t *)tws + 16 * i, (const uint8_t *)twc + 16 * i);
	}
	if constexpr (N >= 8) {
		for (int i = t; i < N / 8; i += stride)
			cp_async16((uint8_t *)wins + 16 * i, (const uint8_t *)win + 16 * i);
	} else {
		for (int i = t; i < N; i += stride)
			wins[i] = win[i];
	}
}

SCAN_DEV long long entry_offset(const SmallParams &prm, int e)
{
	return prm.read_off ? prm.read_off[e] : (long long)(e - prm.entry_base) * prm.regular_stride;
}

/* rtl_power.c:581-596 divides by the INTERLEAVED length and truncates toward 0 */
SCAN_DEV int dc_average(long long sum, int length)
{
	return (int)(int16_t)(sum / (long long)length);
}

/* ---- pieces shared by the two loops of scan_small_kernel ---------------- */

/* byte sums of I and Q over one staged 16 KiB read -> the constants (127 + int16 average) that the front end
 * subtracts from the raw bytes: remove_dc over the WHOLE read (rtl_power.c:581-596, 692-693), divisors B and B-1 */
SCAN_DEV void u8_read_dc(const uint8_t *st, int *red, int t, int &kI, int &kQ)
{
	unsigned sI = 0, sQ = 0;
#pragma unroll
	for (int i = 0; i < kStageBytes / (kThreads * 16); ++i) {
		const uint4 q = *(const uint4 *)(st + (i * kThreads + t) * 16);
		sI = __dp4a(q.x, 0x00010001u, sI);
		sQ = __dp4a(q.x, 0x01000100u, sQ);
		sI = __dp4a(q.y, 0x00010001u, sI);
		sQ = __dp4a(q.y, 0x01000100u, sQ);
		sI = __dp4a(q.z, 0x00010001u, sI);
		sQ = __dp4a(q.z, 0x01000100u, sQ);
		sI = __dp4a(q.w, 0x00010001u, sI);
		sQ = __dp4a(q.w, 0x01000100u, sQ);
	}
	sI = warp_sum(sI);
	sQ = warp_sum(sQ);
	if ((t & 31) == 0) {
		red[(t >> 5) * 2 + 0] = (int)sI;
		red[(t >> 5) * 2 + 1] = (int)sQ;
	}
	__syncthreads();
	int tI = 0, tQ = 0;
#pragma unroll
	for (int w = 0; w < kThreads / 32; ++w) {
		tI += red[w * 2];
		tQ += red[w * 2 + 1];
	}
	/* sum of (b - 127); int16 average, truncating division (rtl_power.c:589) */
	kI = 127 + (int)(int16_t)((tI - 127 * (kStageBytes / 2)) / kStageBytes);
	kQ = 127 + (int)(int16_t)((tQ - 127 * (kStageBytes / 2)) / (kStageBytes - 1));
}

/* sample index (inside its FFT block / inside the working set) that feeds register r */
template <int L>
SCAN_DEV void front_index(int r, int t, int trev, int blkbase, int &nblk, int &n)
{
	constexpr int N = 1 << L;
	if constexpr (L >= 4) {
		nblk = (brev4(r) << (L - 4)) + trev;
		n = blkbase + nblk;
	} else {
		nblk = brev_bits((unsigned)(r & (N - 1)), L);
		n = (t << 4) + (r & ~(N - 1)) + nblk;
	}
}

/* u8 -> int16 minus (127 + DC), window, bit-reversed placement (rtl_power.c:666-668, 594, 697-706) */

/* 4096 bins: a thread multiplies by the same 16 window coefficients in every working set (one FFT block per
 * working set, nblk depends on (t, r) only), so they live in 8 registers, two 16-bit coefficients each */
constexpr int kWinRegs = kPts / 2;

template <int L>
SCAN_DEV void load_window_regs(unsigned (&wreg)[kWinRegs], const uint16_t *wins, int t, int trev, int blkbase)
{
#pragma unroll
	for (int j = 0; j < kWinRegs; ++j) {
		int nblk0, nblk1, n;
		front_index<L>(2 * j, t, trev, blkbase, nblk0, n);
		front_index<L>(2 * j + 1, t, trev, blkbase, nblk1, n);
		wreg[j] = (unsigned)wins[nblk0] | ((unsigned)wins[nblk1] << 16);
	}
}

template <int L, bool WREG = false>
SCAN_DEV void front_u8(X2 (&x)[kPts], const uint8_t *st, int ws, int kI, int kQ, const uint16_t *wins, int t, int trev,
		       int blkbase, const unsigned *wreg = nullptr)
{
#pragma unroll
	for (int r = 0; r < kPts; ++r) {
		int nblk, n;
		front_index<L>(r, t, trev, blkbase, nblk, n);
		/* (byte - k) in one IDP.4A each, times the window coefficient already moved to the high half:
		 * the int16 truncation of the product (rtl_power.c:701, 705) is the natural mod-2^32 wrap */
		unsigned wx;
		if constexpr (WREG)
			wx = (r & 1) ? (wreg[r >> 1] & 0xFFFF0000u) : (wreg[r >> 1] << 16);
		else
			wx = (unsigned)wins[nblk] << 16;
		const unsigned raw = ((const uint16_t *)st)[ws * kWS + n];
#if RSCAN_FRONT_IDP
		x[r].re = (int)(__dp4a(raw, 0x00000001u, (unsigned)-kI) * wx);
		x[r].im = (int)(__dp4a(raw, 0x00000100u, (unsigned)-kQ) * wx);
#else
		x[r].re = (int)((unsigned)((int)(raw & 0xFFu) - kI) * wx);
		x[r].im = (int)((unsigned)((int)(raw >> 8) - kQ) * wx);
#endif
	}
}

/* one hop's sums / peaks of the kThreads transform threads synchronised by `bar` -> tunes[hop].avg (64-bit RED);
 * `bins` = N x u64 of shared memory that none of them is using (only touched when N < 4096, where several
 * registers share a bin) */
template <int L, bool PEAK, class BAR = BlockBar>
SCAN_DEV void flush_bins(unsigned long long (&acc)[kPts], long long *out, unsigned long long *bins, int t,
			 const BAR &bar = BAR())
{
	constexpr int N = 1 << L;
	if constexpr (L == 12) {
#pragma unroll
		for (int r = 0; r < kPts; ++r) {
			const int bin = last_pos<L>(t, r) & (N - 1);
			if constexpr (PEAK)
				atomicMax(out + bin, (long long)acc[r]);
			else
				atomicAdd((unsigned long long *)(out + bin), acc[r]);
		}
	} else {
		bar.sync();
		for (int i = t; i < N; i += kThreads)
			bins[i] = 0ull;
		bar.sync();
#pragma unroll
		for (int r = 0; r < kPts; ++r) {
			const int bin = last_pos<L>(t, r) & (N - 1);
			if constexpr (PEAK)
				atomicMax(bins + bin, acc[r]);
			else
				atomicAdd(bins + bin, acc[r]);
		}
		bar.sync();
		for (int i = t; i < N; i += kThreads) {
			if constexpr (PEAK)
				atomicMax(out + i, (long long)bins[i]);
			else
				atomicAdd((unsigned long long *)(out + i), bins[i]);
		}
		bar.sync();
	}
}

/* ---- spectral kurtosis: sum |X|^4 beside the power sums (sk.cuh) ----------- */

SCAN_DEV void sk_zero(unsigned long long (&lo)[kPts], unsigned (&hi)[kPts])
{
#pragma unroll
	for (int r = 0; r < kPts; ++r) {
		lo[r] = 0ull;
		hi[r] = 0u;
	}
}

/* accumulate_power<false> plus pw^2 into the 128-bit partial (lo, hi) */
SCAN_DEV void accumulate_power_sk(unsigned long long &acc, unsigned long long &lo, unsigned &hi, int re, int im)
{
	const unsigned pw = (unsigned)(re * re) + (unsigned)(im * im);
	acc += pw;
	sk_accumulate(lo, hi, pw);
}

/* flush_bins<L, false> for the S2 partials: out = the hop's [N][2] words; `bins` = 2N x u64 of idle shared memory */
template <int L>
SCAN_DEV void flush_s2(const unsigned long long (&lo)[kPts], const unsigned (&hi)[kPts], unsigned long long *out,
		       unsigned long long *bins, int t)
{
	constexpr int N = 1 << L;
	if constexpr (L == 12) {
#pragma unroll
		for (int r = 0; r < kPts; ++r) {
			const int bin = last_pos<L>(t, r) & (N - 1);
			sk_atomic_add(out + 2 * bin, lo[r], hi[r]);
		}
	} else {
		__syncthreads();
		for (int i = t; i < 2 * N; i += kThreads)
			bins[i] = 0ull;
		__syncthreads();
#pragma unroll
		for (int r = 0; r < kPts; ++r) {
			const int bin = last_pos<L>(t, r) & (N - 1);
			sk_atomic_add(bins + 2 * bin, lo[r], hi[r]);
		}
		__syncthreads();
		for (int i = t; i < N; i += kThreads)
			sk_atomic_add(out + 2 * i, bins[2 * i], bins[2 * i + 1]);
		__syncthreads();
	}
}

/*
 * u8 reads (IN16 = false): the launch's hop-sorted reads are cut into gridDim.x contiguous runs of equal
 * length, counted in 4096-sample working sets (half reads), so every CTA does the same amount of work whatever
 * the hop count; a CTA walks its run once, keeps the next read in flight across hop boundaries, and flushes
 * its register accumulators whenever the hop changes.  A run may begin or end in the middle of a read: that CTA
 * still stages the whole read (remove_dc needs all of it) and transforms only its half.
 * decimated images (IN16 = true): segment list, one CTA per segment (the decimating paths).
 */
template <int L, bool PEAK, bool IN16>
__global__ void __launch_bounds__(kThreads, 2)
scan_small_kernel(const SCAN_GRID_CONSTANT SmallParams prm)
{
	constexpr bool SK = false;
	[[maybe_unused]] unsigned long long *const s2 = nullptr;
#include "scan_small_body.inl"
}

/*
 * RTLSDR_GPU_FLAG_SPECTRAL_KURTOSIS: the same kernel with sum |X|^4 (sk.cuh) accumulated beside the power sums, into
 * s2 [tune_count << L][2] (lo, hi).  The 128-bit register partials take 48 more registers than scan_small_kernel's
 * 2-CTA budget of 128 allows, so this variant is compiled for one CTA per SM (no spills) instead of a shared-memory
 * S2 image: at N = 4096 the 48 KiB image would not leave room for a second CTA either.
 */
template <int L, bool IN16>
__global__ void __launch_bounds__(kThreads, 1)
scan_small_sk_kernel(const SCAN_GRID_CONSTANT SmallParams prm, unsigned long long *s2)
{
	constexpr bool SK = true, PEAK = false;
#include "scan_small_body.inl"
}

/* ======================================================================== *
 *  Decimating front ends (narrow scans): u8 reads -> c16 images             *
 * ======================================================================== */

struct DecimParams {
	const uint8_t *base;       /* u8 reads */
	const long long *read_off; /* byte offset of entry e */
	int n_reads;
	int pairs;                 /* buf_len / 2 complex samples per read */
	int ds;
	c16 *out;                  /* entry e at out + e * out_stride */
	long long out_stride;      /* in c16 units */
	int out_count;             /* c16 slots to write per entry */
	int l_len;                 /* buf_len / ds: interleaved int16 count remove_dc covers */
	long long *sums;           /* [entry][2], zeroed by the host */
};

/*
 * rtl_power.c:671-681 in closed form: slot k = wrap16(sum of inputs k*ds ..
 * k*ds+ds-1 that exist); slots past ceil(pairs/ds) are zero.  One thread per
 * output slot; VEC = widest load (bytes) that 2*ds bytes per slot stays aligned
 * to, all loads of a slot issued before they are summed (IDP.4A byte sums).
 * The DC sums the reference's remove_dc() takes over the decimated buffer
 * (I over even int16 indices < l_len, Q over odd ones, rtl_power.c:586-588,
 * 692-693) are reduced per CTA and added to prm.sums.
 */
template <int VEC>
SCAN_DEV void boxcar_accumulate(const uint8_t *p, int nbytes, int &sb_i, int &sb_q)
{
	unsigned si = 0, sq = 0;
	if constexpr (VEC == 16) {
		for (int o = 0; o < nbytes; o += 64) {
			uint4 q[4];
#pragma unroll
			for (int j = 0; j < 4; ++j)
				q[j] = (o + 16 * j < nbytes) ? __ldg((const uint4 *)(p + o + 16 * j)) : uint4{ 0, 0, 0, 0 };
#pragma unroll
			for (int j = 0; j < 4; ++j) {
				si = __dp4a(q[j].x, 0x00010001u, si); sq = __dp4a(q[j].x, 0x01000100u, sq);
				si = __dp4a(q[j].y, 0x00010001u, si); sq = __dp4a(q[j].y, 0x01000100u, sq);
				si = __dp4a(q[j].z, 0x00010001u, si); sq = __dp4a(q[j].z, 0x01000100u, sq);
				si = __dp4a(q[j].w, 0x00010001u, si); sq = __dp4a(q[j].w, 0x01000100u, sq);
			}
		}
	} else if constexpr (VEC == 8) {
		for (int o = 0; o < nbytes; o += 64) {
			uint2 q[8];
#pragma unroll
			for (int j = 0; j < 8; ++j)
				q[j] = (o + 8 * j < nbytes) ? __ldg((const uint2 *)(p + o + 8 * j)) : uint2{ 0, 0 };
#pragma unroll
			for (int j = 0; j < 8; ++j) {
				si = __dp4a(q[j].x, 0x00010001u, si); sq = __dp4a(q[j].x, 0x01000100u, sq);
				si = __dp4a(q[j].y, 0x00010001u, si); sq = __dp4a(q[j].y, 0x01000100u, sq);
			}
		}
	} else if constexpr (VEC == 4) {
		for (int o = 0; o < nbytes; o += 32) {
			unsigned q[8];
#pragma unroll
			for (int j = 0; j < 8; ++j)
				q[j] = (o + 4 * j < nbytes) ? __ldg((const unsigned *)(p + o + 4 * j)) : 0u;
#pragma unroll
			for (int j = 0; j < 8; ++j) {
				si = __dp4a(q[j], 0x00010001u, si);
				sq = __dp4a(q[j], 0x01000100u, sq);
			}
		}
	} else {
		for (int o = 0; o < nbytes; o += 2) {
			const unsigned raw = __ldg((const uint16_t *)(p + o));
			si += raw & 0xFFu;
			sq += raw >> 8;
		}
	}
	sb_i = (int)si;
	sb_q = (int)sq;
}

template <int VEC>
__global__ void __launch_bounds__(256)
boxcar_kernel(const SCAN_GRID_CONSTANT DecimParams prm)
{
	__shared__ long long red[2 * 8];
	const int e = blockIdx.y;
	const int k = blockIdx.x * blockDim.x + threadIdx.x;
	const uint8_t *src = prm.base + prm.read_off[e];
	const int outs = (prm.pairs + prm.ds - 1) / prm.ds;
	int si = 0, sq = 0;
	if (k < outs) {
		const int lo = k * prm.ds;
		const int cnt = (lo + prm.ds <= prm.pairs) ? prm.ds : prm.pairs - lo;
		int bi, bq;
		if (cnt == prm.ds)
			boxcar_accumulate<VEC>(src + 2ll * lo, 2 * cnt, bi, bq);
		else
			boxcar_accumulate<2>(src + 2ll * lo, 2 * cnt, bi, bq); /* partial tail group */
		si = bi - 127 * cnt; /* sum of (b - 127), rtl_power.c:666-668 */
		sq = bq - 127 * cnt;
	}
	const c16 v = c16_pack(si, sq);
	if (k < prm.out_count)
		prm.out[e * prm.out_stride + k] = v;
	/* remove_dc sees the wrapped int16 values at indices < l_len */
	long long dI = (2 * k < prm.l_len) ? (long long)c16_re(v) : 0;
	long long dQ = (2 * k + 1 < prm.l_len) ? (long long)c16_im(v) : 0;
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) {
		dI += __shfl_xor_sync(0xffffffffu, dI, o);
		dQ += __shfl_xor_sync(0xffffffffu, dQ, o);
	}
	if ((threadIdx.x & 31) == 0) {
		red[(threadIdx.x >> 5) * 2] = dI;
		red[(threadIdx.x >> 5) * 2 + 1] = dQ;
	}
	__syncthreads();
	if (threadIdx.x < 2) {
		long long t = 0;
		for (int w = 0; w < (int)(blockDim.x >> 5); ++w)
			t += red[2 * w + threadIdx.x];
		if (t != 0)
			atomicAdd((unsigned long long *)(prm.sums + 2 * e + threadIdx.x), (unsigned long long)t);
	}
}

/*
 * Same result, for ds <= 64: the 256 slots of a CTA cover 512*ds contiguous input
 * bytes.  They are fetched with fully coalesced 16-byte cp.async copies into
 * shared memory and summed from there, so DRAM sees only full-line streaming
 * reads (this is the HBM-bound regime of the pipeline: 2*ds input bytes per
 * decimated sample).
 */
constexpr int kBoxcarStageMaxDs = 64;

__global__ void __launch_bounds__(256)
boxcar_staged_kernel(const SCAN_GRID_CONSTANT DecimParams prm)
{
	SCAN_DYN_SMEM(smem);
	__shared__ long long red[2 * 8];
	const int e = blockIdx.y;
	const int t = threadIdx.x;
	const int k = blockIdx.x * blockDim.x + t;
	const uint8_t *src = prm.base + prm.read_off[e];
	const int outs = (prm.pairs + prm.ds - 1) / prm.ds;
	const int span0 = blockIdx.x * 512 * prm.ds;                 /* first input byte of this CTA */
	int span = 2 * prm.pairs - span0;                            /* bytes that exist */
	if (span > 512 * prm.ds)
		span = 512 * prm.ds;
	for (int o = t * 16; o < span; o += 256 * 16)               /* span0 and buf_len are multiples of 16 */
		cp_async16(smem + o, src + span0 + o);
	cp_async_commit();
	cp_async_wait_all();
	__syncthreads();
	int si = 0, sq = 0;
	if (k < outs) {
		const int lo = t * 2 * prm.ds;
		int nb = span - lo;
		if (nb > 2 * prm.ds)
			nb = 2 * prm.ds;
		unsigned ui = 0, uq = 0;
		if ((prm.ds & 1) == 0) {
			for (int o = 0; o < nb; o += 4) {
				const unsigned q = *(const unsigned *)(smem + lo + o);
				ui = __dp4a(q, 0x00010001u, ui);
				uq = __dp4a(q, 0x01000100u, uq);
			}
		} else {
			for (int o = 0; o < nb; o += 2) {
				const unsigned raw = *(const uint16_t *)(smem + lo + o);
				ui += raw & 0xFFu;
				uq += raw >> 8;
			}
		}
		si = (int)ui - 127 * (nb >> 1);
		sq = (int)uq - 127 * (nb >> 1);
	}
	const c16 v = c16_pack(si, sq);
	if (k < prm.out_count)
		prm.out[e * prm.out_stride + k] = v;
	long long dI = (2 * k < prm.l_len) ? (long long)c16_re(v) : 0;
	long long dQ = (2 * k + 1 < prm.l_len) ? (long long)c16_im(v) : 0;
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) {
		dI += __shfl_xor_sync(0xffffffffu, dI, o);
		dQ += __shfl_xor_sync(0xffffffffu, dQ, o);
	}
	if ((t & 31) == 0) {
		red[(t >> 5) * 2] = dI;
		red[(t >> 5) * 2 + 1] = dQ;
	}
	__syncthreads();
	if (t < 2) {
		long long s = 0;
		for (int w = 0; w < (int)(blockDim.x >> 5); ++w)
			s += red[2 * w + t];
		if (s != 0)
			atomicAdd((unsigned long long *)(prm.sums + 2 * e + t), (unsigned long long)s);
	}
}

struct HalfbandParams {
	const void *in;            /* u8 pairs (first pass) or c16 */
	const long long *read_off; /* first pass: byte offsets of the u8 reads */
	long long in_stride;       /* c16 units, later passes */
	c16 *out;
	long long out_stride;      /* c16 units */
	int n_out;                 /* outputs per entry = inputs / 2 */
};

template <bool FROM_U8>
SCAN_DEV void hb_sample(const HalfbandParams &prm, int e, int n, int &re, int &im)
{
	if constexpr (FROM_U8) {
		const uint16_t *src = (const uint16_t *)((const uint8_t *)prm.in + prm.read_off[e]);
		const unsigned raw = __ldg(src + n);
		re = (int)(raw & 0xFFu) - 127;
		im = (int)(raw >> 8) - 127;
	} else {
		const c16 raw = __ldg((const c16 *)prm.in + e * prm.in_stride + n);
		re = c16_re(raw);
		im = c16_im(raw);
	}
}

/*
 * One fifth_order pass (rtl_power.c:554-579) on both halves, stateless per read.
 * With s[n] the inputs of one half, output n is
 *   n=0: ((s0+s1)*10 + (s2+s3)*5 + s3 + s5) >> 4
 *   n=1: ((s1+s2)*10 + (s0+s3)*5 + s4 + s5) >> 4
 *   n=2: (s0 + (s1+s4)*5 + (s2+s3)*10 + s5) >> 4
 *   n>=3: (a + (b+e)*5 + (c+d)*10 + f) >> 4 with (a..f) =
 *        n=3: s2 s3 s4 s5 s5 s6   n=4: s4 s5 s5 s6 s7 s8   (the reference's ease-in)
 *        n>=5: s[2n-5] s[2n-4] s[2n-3] s[2n-2] s[2n-1] s[2n]
 */
template <bool FROM_U8>
__global__ void __launch_bounds__(256)
halfband_kernel(const SCAN_GRID_CONSTANT HalfbandParams prm)
{
	const int e = blockIdx.y;
	const int n = blockIdx.x * blockDim.x + threadIdx.x;
	if (n >= prm.n_out)
		return;
	int idx[6];
	if (n >= 5) {
		idx[0] = 2 * n - 5; idx[1] = 2 * n - 4; idx[2] = 2 * n - 3;
		idx[3] = 2 * n - 2; idx[4] = 2 * n - 1; idx[5] = 2 * n;
	} else if (n == 4) {
		idx[0] = 4; idx[1] = 5; idx[2] = 5; idx[3] = 6; idx[4] = 7; idx[5] = 8;
	} else if (n == 3) {
		idx[0] = 2; idx[1] = 3; idx[2] = 4; idx[3] = 5; idx[4] = 5; idx[5] = 6;
	} else {
		idx[0] = 0; idx[1] = 1; idx[2] = 2; idx[3] = 3; idx[4] = 4; idx[5] = 5;
	}
	int xr[6], xi[6];
#pragma unroll
	for (int i = 0; i < 6; ++i)
		hb_sample<FROM_U8>(prm, e, idx[i], xr[i], xi[i]);
	int re, im;
	if (n == 0) {
		re = ((xr[0] + xr[1]) * 10 + (xr[2] + xr[3]) * 5 + xr[3] + xr[5]) >> 4;
		im = ((xi[0] + xi[1]) * 10 + (xi[2] + xi[3]) * 5 + xi[3] + xi[5]) >> 4;
	} else if (n == 1) {
		re = ((xr[1] + xr[2]) * 10 + (xr[0] + xr[3]) * 5 + xr[4] + xr[5]) >> 4;
		im = ((xi[1] + xi[2]) * 10 + (xi[0] + xi[3]) * 5 + xi[4] + xi[5]) >> 4;
	} else if (n == 2) {
		re = (xr[0] + (xr[1] + xr[4]) * 5 + (xr[2] + xr[3]) * 10 + xr[5]) >> 4;
		im = (xi[0] + (xi[1] + xi[4]) * 5 + (xi[2] + xi[3]) * 10 + xi[5]) >> 4;
	} else {
		re = (xr[0] + (xr[1] + xr[4]) * 5 + (xr[2] + xr[3]) * 10 + xr[5]) >> 4;
		im = (xi[0] + (xi[1] + xi[4]) * 5 + (xi[2] + xi[3]) * 10 + xi[5]) >> 4;
	}
	prm.out[e * prm.out_stride + n] = c16_pack(re, im);
}

/*
 * The whole -F chain of one read tile in one kernel (downsample_passes <= 7):
 * fifth_order x P (rtl_power.c:554-579, 683-685) and the optional 9-tap
 * generic_fir (rtl_power.c:598-626, 687-690), with the decimated c16 image and
 * the remove_dc sums as output.  A CTA produces `tile` final samples; the input
 * span it needs (tile * 2^P samples plus a halo of 5 * (2^P - 1) + 9 * 2^P) is
 * read once with coalesced loads and all intermediate levels stay in shared
 * memory (int16 wrap at every level, like the reference's in-place buffer).
 */
struct HalfbandChainParams {
	const uint8_t *base;
	const long long *read_off;
	int pairs;                 /* complex samples per read */
	int passes;                /* P */
	int tile;                  /* final samples per CTA */
	int use_fir;
	int f1, f2, f3, f4, f5;
	c16 *out;
	long long out_stride;
	int l_len;
	long long *sums;
	int cap0;                  /* capacity (c16) of the level-0 buffer; level 1 buffer = cap0/2 + 8 */
};

/* one fifth_order output n from level buffer `src` whose element 0 is absolute index `lo` */
SCAN_DEV c16 halfband_output(const c16 *src, int lo, int n)
{
	int i0, i1, i2, i3, i4, i5;
	if (n >= 5) {
		i0 = 2 * n - 5; i1 = 2 * n - 4; i2 = 2 * n - 3; i3 = 2 * n - 2; i4 = 2 * n - 1; i5 = 2 * n;
	} else if (n == 4) {
		i0 = 4; i1 = 5; i2 = 5; i3 = 6; i4 = 7; i5 = 8;
	} else if (n == 3) {
		i0 = 2; i1 = 3; i2 = 4; i3 = 5; i4 = 5; i5 = 6;
	} else {
		i0 = 0; i1 = 1; i2 = 2; i3 = 3; i4 = 4; i5 = 5;
	}
	const c16 v0 = src[i0 - lo], v1 = src[i1 - lo], v2 = src[i2 - lo], v3 = src[i3 - lo], v4 = src[i4 - lo],
		  v5 = src[i5 - lo];
	const int r0 = c16_re(v0), r1 = c16_re(v1), r2 = c16_re(v2), r3 = c16_re(v3), r4 = c16_re(v4), r5 = c16_re(v5);
	const int q0 = c16_im(v0), q1 = c16_im(v1), q2 = c16_im(v2), q3 = c16_im(v3), q4 = c16_im(v4), q5 = c16_im(v5);
	int re, im;
	if (n == 0) {
		re = ((r0 + r1) * 10 + (r2 + r3) * 5 + r3 + r5) >> 4;
		im = ((q0 + q1) * 10 + (q2 + q3) * 5 + q3 + q5) >> 4;
	} else if (n == 1) {
		re = ((r1 + r2) * 10 + (r0 + r3) * 5 + r4 + r5) >> 4;
		im = ((q1 + q2) * 10 + (q0 + q3) * 5 + q4 + q5) >> 4;
	} else {
		re = (r0 + (r1 + r4) * 5 + (r2 + r3) * 10 + r5) >> 4;
		im = (q0 + (q1 + q4) * 5 + (q2 + q3) * 10 + q5) >> 4;
	}
	return c16_pack(re, im);
}

__global__ void __launch_bounds__(256)
halfband_chain_kernel(const SCAN_GRID_CONSTANT HalfbandChainParams prm)
{
	SCAN_DYN_SMEM(smem);
	__shared__ long long red[2 * 8];
	__shared__ int lo_s[12], hi_s[12];
	c16 *buf0 = (c16 *)smem;
	c16 *buf1 = buf0 + prm.cap0;
	const int e = blockIdx.y, t = threadIdx.x, P = prm.passes;
	const int nt = blockDim.x; /* 256 for full tiles, 64 for the 16-sample head tiles of the streaming path */
	const int M = prm.pairs >> P;
	const int k0 = blockIdx.x * prm.tile;
	const int k1 = (k0 + prm.tile < M) ? k0 + prm.tile : M;

	/* index ranges [lo_j, hi_j] needed at every level, top down */
	if (t == 0) {
		int lo = prm.use_fir ? (k0 >= 9 ? k0 - 9 : 0) : k0, hi = k1 - 1;
		lo_s[P] = lo;
		hi_s[P] = hi;
		for (int j = P; j >= 1; --j) {
			const int cnt = prm.pairs >> (j - 1);
			int nlo = 2 * lo - 5, nhi = 2 * hi;
			if (nlo < 0)
				nlo = 0;
			if (lo <= 4 && nhi < 8)
				nhi = 8; /* the eased-in outputs 0..4 read inputs 0..8 */
			if (nhi > cnt - 1)
				nhi = cnt - 1;
			lo = nlo;
			hi = nhi;
			lo_s[j - 1] = lo;
			hi_s[j - 1] = hi;
		}
	}
	__syncthreads();

	/* level 0: u8 pairs -> c16 minus 127 (rtl_power.c:666-668) */
	{
		const uint16_t *src = (const uint16_t *)(prm.base + prm.read_off[e]);
		const int lo = lo_s[0], n = hi_s[0] - lo + 1;
		for (int i = t; i < n; i += nt) {
			const unsigned raw = __ldg(src + lo + i);
			buf0[i] = c16_pack((int)(raw & 0xFFu) - 127, (int)(raw >> 8) - 127);
		}
	}
	__syncthreads();
	c16 *cur = buf0, *nxt = buf1;
	for (int j = 1; j <= P; ++j) {
		const int lo = lo_s[j], n = hi_s[j] - lo + 1, plo = lo_s[j - 1];
		for (int i = t; i < n; i += nt)
			nxt[i] = halfband_output(cur, plo, lo + i);
		__syncthreads();
		c16 *tmp = cur;
		cur = nxt;
		nxt = tmp;
	}

	/* droop-compensation FIR (or plain copy), image store, DC sums */
	long long dI = 0, dQ = 0;
	const int lo = lo_s[P];
	for (int k = k0 + t; k < k1; k += nt) {
		c16 o = cur[k - lo];
		if (prm.use_fir && k >= 9) {
			const c16 *hsrc = cur + (k - 9 - lo);
			int hr[9], hi[9];
#pragma unroll
			for (int i = 0; i < 9; ++i) {
				hr[i] = c16_re(hsrc[i]);
				hi[i] = c16_im(hsrc[i]);
			}
			unsigned sr = 0, si = 0;
			sr += (unsigned)(hr[0] + hr[8]) * (unsigned)prm.f1;
			sr += (unsigned)(hr[1] + hr[7]) * (unsigned)prm.f2;
			sr += (unsigned)(hr[2] + hr[6]) * (unsigned)prm.f3;
			sr += (unsigned)(hr[3] + hr[5]) * (unsigned)prm.f4;
			sr += (unsigned)hr[4] * (unsigned)prm.f5;
			si += (unsigned)(hi[0] + hi[8]) * (unsigned)prm.f1;
			si += (unsigned)(hi[1] + hi[7]) * (unsigned)prm.f2;
			si += (unsigned)(hi[2] + hi[6]) * (unsigned)prm.f3;
			si += (unsigned)(hi[3] + hi[5]) * (unsigned)prm.f4;
			si += (unsigned)hi[4] * (unsigned)prm.f5;
			o = c16_pack((int)sr >> 15, (int)si >> 15);
		}
		prm.out[e * prm.out_stride + k] = o;
		if (2 * k < prm.l_len)
			dI += c16_re(o);
		if (2 * k + 1 < prm.l_len)
			dQ += c16_im(o);
	}
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) {
		dI += __shfl_xor_sync(0xffffffffu, dI, o);
		dQ += __shfl_xor_sync(0xffffffffu, dQ, o);
	}
	if ((t & 31) == 0) {
		red[(t >> 5) * 2] = dI;
		red[(t >> 5) * 2 + 1] = dQ;
	}
	__syncthreads();
	if (t < 2) {
		long long s = 0;
		for (int w = 0; w < (nt >> 5); ++w)
			s += red[2 * w + t];
		if (s != 0)
			atomicAdd((unsigned long long *)(prm.sums + 2 * e + t), (unsigned long long)s);
	}
}

/*
 * The same -F chain as a register-resident streaming filter (downsample_passes <= 5): no shared
 * memory, no barriers, every intermediate sample is produced and consumed in registers.
 *
 * One thread owns `span` consecutive FINAL samples of one read and walks the input once,
 * 2^P samples per final sample.  Level 1 (half of all the chain's outputs) is computed
 * straight from the packed bytes: with W[m] the 32-bit word holding samples 2m and 2m+1
 * (bytes I, Q, I, Q), output n = (a + 5(b+e) + 10(c+d) + f) >> 4 over samples 2n-5 .. 2n
 * is four IDP.4A per component over W[n-3] .. W[n] with the coefficient words below, the
 * -127 offsets (rtl_power.c:666-668) folded into the addend (-127 * 32).  Levels >= 2 keep
 * the five newest samples of the level below as ints and take two new ones per output.
 * int16 wrap at every level like the reference's in-place buffer.
 *
 * Why outputs are exact although a thread starts in the middle of a read with zeroed
 * windows: a generic output n >= 5 of any level depends on samples 2n-5 .. 2n >= 5 of the
 * level below only, so garbage never spreads: after a warm-up of 16 final samples (level-0
 * reach 14 * 2^P - 5 samples incl. the 9 FIR taps) everything a thread stores is exact.  The
 * reference's eased-in outputs 0..4 of every level (rtl_power.c:567-577) only reach final
 * samples 0..13 (through the FIR); final samples [0, 16) of every read are therefore left to
 * halfband_chain_kernel (one 16-sample tile per read), which also adds their DC terms.
 */
struct HalfbandStreamParams {
	const uint8_t *base;
	const long long *read_off;
	int n_reads;
	int pairs;                 /* complex samples per read */
	int span;                  /* final samples per thread, a multiple of 4 */
	int use_fir;
	int f1, f2, f3, f4, f5;
	c16 *out;
	long long out_stride;
	int l_len;
	long long *sums;
};

constexpr int kHbStreamHead = 16; /* final samples [0, 16) come from the tile kernel */
constexpr int kHbStreamWarm = 16; /* final samples computed and discarded in front of a span */
constexpr int kHbStreamMaxPasses = 5;

/* Levels >= 2 keep the level below as PAIR words: samples 2m (low half) and 2m+1 (high half)
 * of one component, so that output n = a + 5(b+e) + 10(c+d) + f over samples 2n-5 .. 2n is four
 * IDP.2A (16-bit x 8-bit dot products) over pair words n-3 .. n; packing a pair (PRMT) is also
 * the int16 wrap of the reference's buffer. */
struct HbWin {
	unsigned r[3], i[3]; /* pair words n-3, n-2, n-1 of the level below */
};

template <int P>
struct HbState {
	unsigned wq[3];                   /* byte words W[n-3], W[n-2], W[n-1] */
	HbWin win[P > 1 ? P - 1 : 1];     /* win[j]: pair words of level j + 1, feeding level j + 2 */
};

constexpr unsigned kHbK1 = 0x0A050100u; /* bytes (0, 1 | 5, 10): _lo on pair n-3, _hi on pair n-2 */
constexpr unsigned kHbK2 = 0x0001050Au; /* bytes (10, 5 | 1, 0): _lo on pair n-1, _hi on pair n   */

/* level-1 output, NOT yet wrapped to int16 (the consumer's PRMT / the final sign extension does that) */
SCAN_DEV void hb_level1(unsigned (&wq)[3], unsigned w, int &re, int &im)
{
	unsigned sr = (unsigned)-4064, si = (unsigned)-4064; /* -127 * (1 + 5 + 10 + 10 + 5 + 1) */
	sr = __dp4a(wq[0], 0x00010000u, sr); si = __dp4a(wq[0], 0x01000000u, si); /* a = sample 2n-5 */
	sr = __dp4a(wq[1], 0x000A0005u, sr); si = __dp4a(wq[1], 0x0A000500u, si); /* 5 b + 10 c */
	sr = __dp4a(wq[2], 0x0005000Au, sr); si = __dp4a(wq[2], 0x05000A00u, si); /* 10 d + 5 e */
	sr = __dp4a(w, 0x00000001u, sr);     si = __dp4a(w, 0x00000100u, si);     /* f = sample 2n */
	re = (int)sr >> 4;
	im = (int)si >> 4;
	wq[0] = wq[1];
	wq[1] = wq[2];
	wq[2] = w;
}

/* output n of a level >= 2 (not yet wrapped) from the window and the new pair n of the level below */
SCAN_DEV void hb_combine(HbWin &w, int r0, int i0, int r1, int i1, int &re, int &im)
{
	const unsigned pr = __byte_perm((unsigned)r0, (unsigned)r1, 0x5410); /* low halves: int16 wrap */
	const unsigned pi = __byte_perm((unsigned)i0, (unsigned)i1, 0x5410);
	int sr = __dp2a_lo((int)w.r[0], (int)kHbK1, 0), si = __dp2a_lo((int)w.i[0], (int)kHbK1, 0);
	sr = __dp2a_hi((int)w.r[1], (int)kHbK1, sr);
	si = __dp2a_hi((int)w.i[1], (int)kHbK1, si);
	sr = __dp2a_lo((int)w.r[2], (int)kHbK2, sr);
	si = __dp2a_lo((int)w.i[2], (int)kHbK2, si);
	sr = __dp2a_hi((int)pr, (int)kHbK2, sr);
	si = __dp2a_hi((int)pi, (int)kHbK2, si);
	re = sr >> 4;
	im = si >> 4;
	w.r[0] = w.r[1]; w.r[1] = w.r[2]; w.r[2] = pr;
	w.i[0] = w.i[1]; w.i[1] = w.i[2]; w.i[2] = pi;
}

/* sample IDX (within the current macro step) of level J; level-1 sample m consumes word m */
template <int J, int IDX, int P, int NW>
SCAN_DEV void hb_produce(HbState<P> &st, const unsigned (&w)[NW], int &re, int &im)
{
	if constexpr (J == 1) {
		hb_level1(st.wq, w[IDX], re, im);
	} else {
		int r0, i0, r1, i1;
		hb_produce<J - 1, 2 * IDX, P, NW>(st, w, r0, i0);
		hb_produce<J - 1, 2 * IDX + 1, P, NW>(st, w, r1, i1);
		hb_combine(st.win[J - 2], r0, i0, r1, i1, re, im);
	}
}

template <int P>
__global__ void __launch_bounds__(128)
halfband_stream_kernel(const SCAN_GRID_CONSTANT HalfbandStreamParams prm)
{
	constexpr int LS = (1 << P) < 8 ? 8 : (1 << P); /* input samples per macro step */
	constexpr int NW = LS / 2, NV = NW / 4;         /* words / 16-byte loads per macro step */
	constexpr int OUTS = LS >> P;                   /* final samples per macro step */
	const int M = prm.pairs >> P;
	const int spans = (M + prm.span - 1) / prm.span;
	const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
	const int e = (int)(gid / spans), sp = (int)(gid % spans);
	if (e >= prm.n_reads)
		return;
	const int k0 = sp * prm.span;
	const int k1 = (k0 + prm.span < M) ? k0 + prm.span : M;
	const int kb = (k0 >= kHbStreamWarm) ? k0 - kHbStreamWarm : 0;
	const int first_store = (k0 > kHbStreamHead) ? k0 : kHbStreamHead;
	const uint4 *src = (const uint4 *)(prm.base + prm.read_off[e] + (long long)kb * (2 << P));

	HbState<P> st;
#pragma unroll
	for (int j = 0; j < 3; ++j)
		st.wq[j] = 0u;
#pragma unroll
	for (int j = 0; j < (P > 1 ? P - 1 : 1); ++j) {
#pragma unroll
		for (int q = 0; q < 3; ++q)
			st.win[j].r[q] = st.win[j].i[q] = 0u;
	}
	int hr[9], hi[9]; /* the nine final samples before the current one (generic_fir, rtl_power.c:598-626) */
#pragma unroll
	for (int q = 0; q < 9; ++q)
		hr[q] = hi[q] = 0;
	long long dI = 0, dQ = 0;
	c16 *dst = prm.out + e * prm.out_stride;

	uint4 nxt[NV];
#pragma unroll
	for (int j = 0; j < NV; ++j)
		nxt[j] = __ldg(src + j);
	for (int k = kb; k < k1; k += OUTS) {
		unsigned w[NW];
#pragma unroll
		for (int j = 0; j < NV; ++j) {
			w[4 * j] = nxt[j].x; w[4 * j + 1] = nxt[j].y; w[4 * j + 2] = nxt[j].z; w[4 * j + 3] = nxt[j].w;
		}
		src += NV;
		if (k + OUTS < k1) { /* next macro step's bytes, in flight during this one's arithmetic */
#pragma unroll
			for (int j = 0; j < NV; ++j)
				nxt[j] = __ldg(src + j);
		}
		int fr[OUTS], fi[OUTS];
		if constexpr (OUTS == 4) {
			hb_produce<P, 0, P, NW>(st, w, fr[0], fi[0]);
			hb_produce<P, 1, P, NW>(st, w, fr[1], fi[1]);
			hb_produce<P, 2, P, NW>(st, w, fr[2], fi[2]);
			hb_produce<P, 3, P, NW>(st, w, fr[3], fi[3]);
		} else if constexpr (OUTS == 2) {
			hb_produce<P, 0, P, NW>(st, w, fr[0], fi[0]);
			hb_produce<P, 1, P, NW>(st, w, fr[1], fi[1]);
		} else {
			hb_produce<P, 0, P, NW>(st, w, fr[0], fi[0]);
		}
#pragma unroll
		for (int o = 0; o < OUTS; ++o) {
			fr[o] = (int)(int16_t)fr[o]; /* the reference stores every level as int16 */
			fi[o] = (int)(int16_t)fi[o];
		}
#pragma unroll
		for (int o = 0; o < OUTS; ++o) {
			const int kk = k + o;
			int re = fr[o], im = fi[o];
			if (prm.use_fir) {
				/* the 9 samples BEFORE kk, int32 wrap-around arithmetic (all kk stored here are >= 16 > 9) */
				unsigned sr = 0, si = 0;
				sr += (unsigned)(hr[0] + hr[8]) * (unsigned)prm.f1;
				sr += (unsigned)(hr[1] + hr[7]) * (unsigned)prm.f2;
				sr += (unsigned)(hr[2] + hr[6]) * (unsigned)prm.f3;
				sr += (unsigned)(hr[3] + hr[5]) * (unsigned)prm.f4;
				sr += (unsigned)hr[4] * (unsigned)prm.f5;
				si += (unsigned)(hi[0] + hi[8]) * (unsigned)prm.f1;
				si += (unsigned)(hi[1] + hi[7]) * (unsigned)prm.f2;
				si += (unsigned)(hi[2] + hi[6]) * (unsigned)prm.f3;
				si += (unsigned)(hi[3] + hi[5]) * (unsigned)prm.f4;
				si += (unsigned)hi[4] * (unsigned)prm.f5;
				re = (int)(int16_t)((int)sr >> 15);
				im = (int)(int16_t)((int)si >> 15);
#pragma unroll
				for (int q = 0; q < 8; ++q) {
					hr[q] = hr[q + 1];
					hi[q] = hi[q + 1];
				}
				hr[8] = fr[o];
				hi[8] = fi[o];
			}
			if (kk >= first_store) {
				dst[kk] = c16_pack(re, im);
				if (2 * kk < prm.l_len)
					dI += re;
				if (2 * kk + 1 < prm.l_len)
					dQ += im;
			}
		}
	}
	if (dI != 0)
		atomicAdd((unsigned long long *)(prm.sums + 2 * e), (unsigned long long)dI);
	if (dQ != 0)
		atomicAdd((unsigned long long *)(prm.sums + 2 * e + 1), (unsigned long long)dQ);
}

struct FirParams {
	const c16 *in;
	long long in_stride;
	c16 *out;
	long long out_stride;
	int count;     /* samples per entry */
	int use_fir;   /* 0: plain copy */
	int f1, f2, f3, f4, f5; /* cic_9_tables[ds_p][1..5], rtl_power.c:219-232 */
};

/* generic_fir (rtl_power.c:598-626): samples 0..8 pass through, sample k >= 9 is
 * the 9-tap sum over inputs k-9..k-1, >> 15, int32 wrap-around arithmetic. */
__global__ void __launch_bounds__(256)
fir9_kernel(const SCAN_GRID_CONSTANT FirParams prm)
{
	const int e = blockIdx.y;
	const int k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= prm.count)
		return;
	const c16 *src = prm.in + e * prm.in_stride;
	c16 o = __ldg(src + k);
	if (prm.use_fir && k >= 9) {
		int hr[9], hi[9];
#pragma unroll
		for (int i = 0; i < 9; ++i) {
			const c16 x = __ldg(src + k - 9 + i);
			hr[i] = c16_re(x);
			hi[i] = c16_im(x);
		}
		unsigned sr = 0, si = 0;
		sr += (unsigned)(hr[0] + hr[8]) * (unsigned)prm.f1;
		sr += (unsigned)(hr[1] + hr[7]) * (unsigned)prm.f2;
		sr += (unsigned)(hr[2] + hr[6]) * (unsigned)prm.f3;
		sr += (unsigned)(hr[3] + hr[5]) * (unsigned)prm.f4;
		sr += (unsigned)hr[4] * (unsigned)prm.f5;
		si += (unsigned)(hi[0] + hi[8]) * (unsigned)prm.f1;
		si += (unsigned)(hi[1] + hi[7]) * (unsigned)prm.f2;
		si += (unsigned)(hi[2] + hi[6]) * (unsigned)prm.f3;
		si += (unsigned)(hi[3] + hi[5]) * (unsigned)prm.f4;
		si += (unsigned)hi[4] * (unsigned)prm.f5;
		o = c16_pack((int)sr >> 15, (int)si >> 15);
	}
	prm.out[e * prm.out_stride + k] = o;
}

struct DcSumParams {
	const c16 *img;
	long long stride;  /* c16 units */
	int l_len;         /* interleaved int16 length the reference's remove_dc sees */
	long long *sums;   /* [entry][2], zeroed by the host before launch */
};

/* Sums for remove_dc (rtl_power.c:586-588): I over even indices < l_len,
 * Q over odd indices < l_len. */
__global__ void __launch_bounds__(256)
dc_sums_c16_kernel(const SCAN_GRID_CONSTANT DcSumParams prm)
{
	const int e = blockIdx.y;
	const c16 *src = prm.img + e * prm.stride;
	const int nI = (prm.l_len + 1) >> 1, nQ = prm.l_len >> 1;
	long long sI = 0, sQ = 0;
	for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < nI; k += gridDim.x * blockDim.x) {
		const c16 x = __ldg(src + k);
		sI += c16_re(x);
		if (k < nQ)
			sQ += c16_im(x);
	}
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) {
		sI += __shfl_xor_sync(0xffffffffu, sI, o);
		sQ += __shfl_xor_sync(0xffffffffu, sQ, o);
	}
	if ((threadIdx.x & 31) == 0) {
		atomicAdd((unsigned long long *)(prm.sums + 2 * e), (unsigned long long)sI);
		atomicAdd((unsigned long long *)(prm.sums + 2 * e + 1), (unsigned long long)sQ);
	}
}

struct DcFinalizeParams {
	const long long *sums; /* [n][2] */
	int *ave;              /* [n][2] */
	int n;
	int l_len;
};

/* ave = (int16)(sum / length), C division; I over l_len, Q over l_len - 1 (rtl_power.c:589, 692-693) */
__global__ void __launch_bounds__(256)
dc_finalize_kernel(const SCAN_GRID_CONSTANT DcFinalizeParams prm)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= 2 * prm.n)
		return;
	prm.ave[i] = dc_average(prm.sums[i], prm.l_len - (i & 1));
}

/* ======================================================================== *
 *  Narrow scans, fused: boxcar decimation + DC + window + FFT + |X|^2 in one *
 *  kernel (the HBM-bound regime: 2*ds input bytes per transformed sample)    *
 * ======================================================================== */

struct FusedBoxcarParams {
	const uint8_t *base;        /* u8 reads of 2 * N * ds bytes (one FFT block per read) */
	const long long *read_off;
	const int4 *segs;           /* IN16: (hop, first entry, entry count, -) */
	int n_segs;
	const int *hop_of;          /* u8 reads: hop of entry e, entries sorted by hop */
	int n_entries;              /* u8 reads: entries of this launch */
	int stagger_ns;             /* u8 reads: start delay of the second resident wave half (see the kernel) */
	int ds;
	int slots;                  /* staging ring depth, 2..4 chunks of 512 * ds bytes */
	long long *avg;
	long long *samples;
	const int2 *twc;
	const uint16_t *win;
	PassTw tw0;
};

template <int L>
struct FusedSmem {
	static constexpr int N = 1 << L;
	static constexpr int off_image = 0;                          /* 4096 c16 decimated samples */
	static constexpr int off_xch = kWS * 4;                      /* two transpose buffers */
	static constexpr int off_tw = off_xch + 2 * kXchWords * 4;
	static constexpr int off_win = off_tw + (N - 16) * 8;
	static constexpr int off_red = (off_win + N * 2 + 15) & ~15; /* [8 warps][2] long long */
	static constexpr int off_stage = off_red + 128;              /* `slots` chunks of 512 * ds bytes */
	static int bytes(int ds, int slots) { return off_stage + slots * 512 * ds; }
};

/* producer lane of a warp-specialised narrow-scan kernel: the CPR chunks of each of the n reads first, first + 1, ..
 * go into the ring of nslots slots in order, one bulk copy each; (slot, ph) is the ring position and phase */
template <int CPR>
SCAN_DEV void produce_reads(const FusedBoxcarParams &prm, int first, int n, uint8_t *stage, uint64_t *full,
			    uint64_t *empty, int chunk_bytes, int nslots, int &slot, unsigned &ph)
{
	long long off = prm.read_off[first];
	for (int rd = 0; rd < n; ++rd) {
		const uint8_t *src = prm.base + off;
		if (rd + 1 < n)
			off = prm.read_off[first + rd + 1]; /* in flight while this read's copies are issued */
		for (int c = 0; c < CPR; ++c) {
			mbar_wait(empty + slot, ph ^ 1u);
			mbar_arrive_expect_tx(full + slot, (unsigned)chunk_bytes);
			bulk_copy_g2s(stage + slot * chunk_bytes, src + (long long)c * chunk_bytes, (unsigned)chunk_bytes,
				      full + slot);
			if (++slot == nslots) {
				slot = 0;
				ph ^= 1u;
			}
		}
	}
}

/*
 * Requirements (checked by the host): boxcar, 2 <= ds <= 64, buf_len = 2 * N * ds (so every
 * read is exactly one FFT block and remove_dc covers all of it), 256 <= N <= 4096.
 * A CTA walks a segment of reads of one hop.  The input is streamed through two 512*ds-byte
 * shared-memory slots with 16-byte cp.async copies (the next slot is in flight while the
 * current one is summed); 256 slots of a chunk are summed per thread with IDP.4A (rtl_power.c
 * :671-681 in closed form); 4096 / N reads fill the working set, each with its own DC average
 * (rtl_power.c:581-596, 692-693); then the same register-blocked transform as scan_small_kernel.
 */
template <int L, bool PEAK, int NS>
__global__ void __launch_bounds__(kThreads, 2)
scan_boxcar_fused_kernel(const SCAN_GRID_CONSTANT FusedBoxcarParams prm)
{
	SCAN_DYN_SMEM(smem);
	typedef FusedSmem<L> SM;
	constexpr int N = 1 << L;
	constexpr int RPW = kWS / N;      /* reads per working set */
	constexpr int CPR = N / kThreads; /* 256-slot chunks per read */
	c16 *image = (c16 *)(smem + SM::off_image);
	c16 *xch = (c16 *)(smem + SM::off_xch);
	int2 *tws = (int2 *)(smem + SM::off_tw);
	uint16_t *wins = (uint16_t *)(smem + SM::off_win);
	long long *red = (long long *)(smem + SM::off_red);
	uint8_t *stage = smem + SM::off_stage;

	const int t = threadIdx.x, ds = prm.ds;
	const int chunk_bytes = 512 * ds;
	load_tables<L>(tws, wins, prm.twc, prm.win, t, kThreads);

	TwSmall<L> tw;
	tw.tws = tws;
	tw.tw0 = &prm.tw0;
	int t0;
	const int trev = front_thread_map<L>(t, t0);
	const int myblk = t >> (L - 4);
	const int blkbase = myblk << L;
	int flip = 0;

	for (int seg = blockIdx.x; seg < prm.n_segs; seg += gridDim.x) {
		const int4 sg = prm.segs[seg];
		const int hop = sg.x, first = sg.y, count = sg.z;
		const int total_chunks = count * CPR;
		unsigned long long acc[kPts];
#pragma unroll
		for (int r = 0; r < kPts; ++r)
			acc[r] = 0ull;

		/* chunk q of the segment = chunk (q % CPR) of read first + q / CPR; a ring of `slots`
		 * staging slots keeps slots-1 chunks in flight (one copy group per chunk, possibly empty) */
		constexpr int ns = NS; /* compile time: slot index and wait depth cost no division / branch */
#pragma unroll
		for (int q0 = 0; q0 < ns - 1; ++q0) {
			if (q0 < total_chunks) {
				const uint8_t *src = prm.base + prm.read_off[first + q0 / CPR] + (long long)(q0 % CPR) * chunk_bytes;
				uint8_t *dst = stage + (q0 % ns) * chunk_bytes;
				for (int o = t * 16; o < chunk_bytes; o += kThreads * 16)
					cp_async16(dst + o, src + o);
			}
			cp_async_commit();
		}
		int kI = 0, kQ = 0;
		long long dI = 0, dQ = 0;
		for (int q = 0; q < total_chunks; ++q) {
			cp_async_wait_group<NS - 2>();
			__syncthreads(); /* chunk q landed; the slot of chunk q-1 is free */
			{
				const int qn = q + ns - 1;
				if (qn < total_chunks) {
					const uint8_t *src = prm.base + prm.read_off[first + qn / CPR] + (long long)(qn % CPR) * chunk_bytes;
					uint8_t *dst = stage + (qn % ns) * chunk_bytes;
					for (int o = t * 16; o < chunk_bytes; o += kThreads * 16)
						cp_async16(dst + o, src + o);
				}
				cp_async_commit();
			}
			const int rd = q / CPR;          /* read within the segment */
			const int rw = rd % RPW;         /* read within the working set */
			const int c = q % CPR;
			/* ---- boxcar: slot = sum of ds samples, minus 127 each (rtl_power.c:666-681) ---- */
			{
				const uint8_t *p = stage + (q % ns) * chunk_bytes + t * 2 * ds;
				unsigned ui = 0, uq = 0;
				if ((ds & 1) == 0) {
					int o = 0;
					for (; o + 16 <= 2 * ds; o += 16) {
						const unsigned w0 = *(const unsigned *)(p + o), w1 = *(const unsigned *)(p + o + 4),
							       w2 = *(const unsigned *)(p + o + 8), w3 = *(const unsigned *)(p + o + 12);
						ui = __dp4a(w0, 0x00010001u, ui); uq = __dp4a(w0, 0x01000100u, uq);
						ui = __dp4a(w1, 0x00010001u, ui); uq = __dp4a(w1, 0x01000100u, uq);
						ui = __dp4a(w2, 0x00010001u, ui); uq = __dp4a(w2, 0x01000100u, uq);
						ui = __dp4a(w3, 0x00010001u, ui); uq = __dp4a(w3, 0x01000100u, uq);
					}
					for (; o < 2 * ds; o += 4) {
						const unsigned w4 = *(const unsigned *)(p + o);
						ui = __dp4a(w4, 0x00010001u, ui);
						uq = __dp4a(w4, 0x01000100u, uq);
					}
				} else {
					for (int o = 0; o < 2 * ds; o += 2) {
						const unsigned raw = *(const uint16_t *)(p + o);
						ui += raw & 0xFFu;
						uq += raw >> 8;
					}
				}
				const c16 v = c16_pack((int)ui - 127 * ds, (int)uq - 127 * ds);
				image[rw * N + c * kThreads + t] = v;
				dI += c16_re(v); /* remove_dc sums the wrapped int16 values */
				dQ += c16_im(v);
			}
			if (c == CPR - 1) {
				/* ---- the read is complete: its DC averages (divisors 2N and 2N-1) ---- */
#pragma unroll
				for (int o = 16; o > 0; o >>= 1) {
					dI += __shfl_xor_sync(0xffffffffu, dI, o);
					dQ += __shfl_xor_sync(0xffffffffu, dQ, o);
				}
				long long *rr = red; /* the two barriers below order its reuse */
				if ((t & 31) == 0) {
					rr[(t >> 5) * 2] = dI;
					rr[(t >> 5) * 2 + 1] = dQ;
				}
				__syncthreads();
				if (myblk == rw) {
					long long sI = 0, sQ = 0;
#pragma unroll
					for (int w = 0; w < kThreads / 32; ++w) {
						sI += rr[2 * w];
						sQ += rr[2 * w + 1];
					}
					kI = dc_average(sI, 2 * N);
					kQ = dc_average(sQ, 2 * N - 1);
				}
				dI = dQ = 0;
				__syncthreads(); /* red may be rewritten by the next read */
			}
			const bool ws_done = (c == CPR - 1) && (rw == RPW - 1 || rd == count - 1);
			if (!ws_done)
				continue;
			const int nvalid = rw + 1;

			/* ---- DC, window, bit-reversed placement, transform, |X|^2 ---- */
			X2 x[kPts];
#pragma unroll
			for (int r = 0; r < kPts; ++r) {
				const int nblk = (brev4(r) << (L - 4)) + trev;
				const c16 raw = image[blkbase + nblk];
				const int wv = wins[nblk];
				x[r].re = ((c16_re(raw) - kI) * wv) << 16;
				x[r].im = ((c16_im(raw) - kQ) * wv) << 16;
			}
			engine_fft_db<L>(x, xch, flip, t, tw, BlockBar(), t0);
#pragma unroll
			for (int r = 0; r < kPts; ++r) {
				const int re = x[r].re >> 16, im = x[r].im >> 16;
				if ((last_pos<L>(t, r) >> L) < nvalid)
					accumulate_power<PEAK>(acc[r], re, im);
			}
			__syncthreads(); /* the image is rewritten by the next working set */
		}

		pdl_wait();
		if (t == 0)
			atomicAdd((unsigned long long *)(prm.samples + hop), (unsigned long long)((long long)count * ds));
		/* the transpose buffers are idle here: 2 * kXchWords * 4 >= N * 8 */
		flush_bins<L, PEAK>(acc, prm.avg + ((long long)hop << L), (unsigned long long *)xch, t);
	}
}

/*
 * The same narrow-scan pipeline, warp specialised (one CTA per SM, three roles):
 *   - warp 16, one lane: the producer.  It walks the CTA's segments and issues one
 *     bulk asynchronous copy (cp.async.bulk, the TMA engine's 1-D form) per 512*ds-byte
 *     chunk into a ring of `slots` shared-memory slots; full[]/empty[] transaction
 *     barriers hand the slots back and forth.  The copies never stop while the other
 *     roles compute, which the single-role kernel above cannot do (its CTAs alternate
 *     between a streaming phase and a transform phase: measured time = sum of both).
 *   - warps 8..15: the boxcar role, two groups of four warps that take alternate chunks.
 *     256 output slots per chunk, two per thread, summed from shared memory with IDP.4A
 *     (rtl_power.c:666-681 in closed form) into one of TWO 4096-sample images; per read
 *     the DC averages (rtl_power.c:581-596, 692-693).  (One group was the bottleneck:
 *     a lone warp per scheduler runs this dependent code at 0.19 instructions per clock.)
 *   - warps 0..7: the transform role.  It waits for a complete image, applies DC and
 *     window, hands the image back at once (img_empty) and runs the register-blocked
 *     fix_fft + |X|^2 with its own named barrier while the other image fills.
 * Same requirements as scan_boxcar_fused_kernel; the host picks this kernel when the
 * streaming side dominates (large ds) and the ring fits.
 */
constexpr int kStreamFftThreads = kThreads;  /* 8 warps per transform group */
constexpr int kStreamBoxGroup = 128;         /* 4 warps: two slots of a chunk per thread */
constexpr int kStreamMaxSlots = 16;

/* FG transform groups (alternate working sets), BG boxcar groups (alternate chunks):
 * (1, 2) when the streaming side dominates, (2, 1) when the transform does (small ds). */
template <int FG, int BG>
struct StreamShape {
	static constexpr int fft_threads = FG * kStreamFftThreads;
	static constexpr int box_threads = BG * kStreamBoxGroup;
	static constexpr int threads = fft_threads + box_threads + 32;
};

template <int L, int FG>
struct StreamSmem {
	static constexpr int N = 1 << L;
	static constexpr int off_image = 0;                          /* 2 x 4096 c16 */
	static constexpr int off_xch = 2 * kWS * 4;                  /* two transpose buffers per transform group */
	static constexpr int off_tw = off_xch + FG * 2 * kXchWords * 4;
	static constexpr int off_win = off_tw + (N - 16) * 8;
	static constexpr int off_dc = (off_win + N * 2 + 15) & ~15;  /* [2 images][16 reads][2] int */
	static constexpr int off_red = off_dc + 2 * 16 * 2 * 4;      /* [2][8 warps][2] int */
	static constexpr int off_bar = off_red + 2 * 8 * 2 * 4;      /* full[16] empty[16] img_full[2] img_empty[2] */
	static constexpr int off_stage = (off_bar + (2 * kStreamMaxSlots + 4) * 8 + 127) & ~127;
	static int bytes(int ds, int slots) { return off_stage + slots * 512 * ds; }
};

/*
 * Byte sums of two boxcar slots at once: I = bytes at even addresses, Q = bytes at odd
 * addresses of [p0, p0 + nbytes) and [p1, p1 + nbytes); both pointers aligned to ALIGN,
 * nbytes a multiple of ALIGN.  Eight independent IDP.4A chains and all loads of an
 * iteration issued before they are consumed: the boxcar role is four warps only.
 */
template <int ALIGN>
SCAN_DEV void boxcar_two_slot_sums(const uint8_t *p0, const uint8_t *p1, int nbytes, unsigned &i0, unsigned &q0,
				   unsigned &i1, unsigned &q1)
{
	unsigned a0 = 0, a1 = 0, b0 = 0, b1 = 0, c0 = 0, c1 = 0, d0 = 0, d1 = 0;
	if constexpr (ALIGN == 16) {
#pragma unroll 2
		for (int o = 0; o < nbytes; o += 16) {
			const uint4 q = *(const uint4 *)(p0 + o), r = *(const uint4 *)(p1 + o);
			a0 = __dp4a(q.x, 0x00010001u, a0); b0 = __dp4a(q.x, 0x01000100u, b0);
			c0 = __dp4a(r.x, 0x00010001u, c0); d0 = __dp4a(r.x, 0x01000100u, d0);
			a1 = __dp4a(q.y, 0x00010001u, a1); b1 = __dp4a(q.y, 0x01000100u, b1);
			c1 = __dp4a(r.y, 0x00010001u, c1); d1 = __dp4a(r.y, 0x01000100u, d1);
			a0 = __dp4a(q.z, 0x00010001u, a0); b0 = __dp4a(q.z, 0x01000100u, b0);
			c0 = __dp4a(r.z, 0x00010001u, c0); d0 = __dp4a(r.z, 0x01000100u, d0);
			a1 = __dp4a(q.w, 0x00010001u, a1); b1 = __dp4a(q.w, 0x01000100u, b1);
			c1 = __dp4a(r.w, 0x00010001u, c1); d1 = __dp4a(r.w, 0x01000100u, d1);
		}
	} else if constexpr (ALIGN == 8) {
#pragma unroll 4
		for (int o = 0; o < nbytes; o += 8) {
			const uint2 q = *(const uint2 *)(p0 + o), r = *(const uint2 *)(p1 + o);
			a0 = __dp4a(q.x, 0x00010001u, a0); b0 = __dp4a(q.x, 0x01000100u, b0);
			c0 = __dp4a(r.x, 0x00010001u, c0); d0 = __dp4a(r.x, 0x01000100u, d0);
			a1 = __dp4a(q.y, 0x00010001u, a1); b1 = __dp4a(q.y, 0x01000100u, b1);
			c1 = __dp4a(r.y, 0x00010001u, c1); d1 = __dp4a(r.y, 0x01000100u, d1);
		}
	} else if constexpr (ALIGN == 4) {
#pragma unroll 4
		for (int o = 0; o < nbytes; o += 4) {
			const unsigned q = *(const unsigned *)(p0 + o), r = *(const unsigned *)(p1 + o);
			a0 = __dp4a(q, 0x00010001u, a0); b0 = __dp4a(q, 0x01000100u, b0);
			c0 = __dp4a(r, 0x00010001u, c0); d0 = __dp4a(r, 0x01000100u, d0);
		}
	} else {
#pragma unroll 4
		for (int o = 0; o < nbytes; o += 2) {
			const unsigned q = *(const uint16_t *)(p0 + o), r = *(const uint16_t *)(p1 + o);
			a0 += q & 0xFFu; b0 += q >> 8;
			c0 += r & 0xFFu; d0 += r >> 8;
		}
	}
	i0 = a0 + a1;
	q0 = b0 + b1;
	i1 = c0 + c1;
	q1 = d0 + d1;
}

template <int L, bool PEAK, int FG, int BG>
__global__ void __launch_bounds__((StreamShape<FG, BG>::threads), 1)
scan_boxcar_stream_kernel(const SCAN_GRID_CONSTANT FusedBoxcarParams prm)
{
	SCAN_DYN_SMEM(smem);
	typedef StreamSmem<L, FG> SM;
	typedef StreamShape<FG, BG> SH;
	constexpr int N = 1 << L;
	constexpr int RPW = kWS / N;      /* reads per working set */
	constexpr int CPR = N / kThreads; /* 256-slot chunks per read */
	c16 *image = (c16 *)(smem + SM::off_image);
	int2 *tws = (int2 *)(smem + SM::off_tw);
	uint16_t *wins = (uint16_t *)(smem + SM::off_win);
	int *dc = (int *)(smem + SM::off_dc);
	int *red = (int *)(smem + SM::off_red);
	uint64_t *full = (uint64_t *)(smem + SM::off_bar);
	uint64_t *empty = full + kStreamMaxSlots;
	uint64_t *img_full = empty + kStreamMaxSlots;
	uint64_t *img_empty = img_full + 2;
	uint8_t *stage = smem + SM::off_stage;

	const int t = threadIdx.x, ds = prm.ds, nslots = prm.slots;
	const int chunk_bytes = 512 * ds;
	if (t == 0) {
		for (int s = 0; s < nslots; ++s) {
			mbar_init(full + s, 1);
			mbar_init(empty + s, kStreamBoxGroup / 32);
		}
		for (int b = 0; b < 2; ++b) {
			mbar_init(img_full + b, SH::box_threads);
			mbar_init(img_empty + b, kStreamFftThreads);
		}
		mbar_fence_init();
	}
	__syncthreads();

	if (t >= SH::fft_threads + SH::box_threads) {
		/* ================= producer ================= */
		if (t != SH::fft_threads + SH::box_threads)
			return;
		int slot = 0;
		unsigned ph = 0;
		for (int seg = blockIdx.x; seg < prm.n_segs; seg += gridDim.x) {
			const int4 sg = prm.segs[seg];
			produce_reads<CPR>(prm, sg.y, sg.z, stage, full, empty, chunk_bytes, nslots, slot, ph);
		}
		return;
	}

	if (t >= SH::fft_threads) {
		/* ================= boxcar role ================= */
		const int bt = (t - SH::fft_threads) & (kStreamBoxGroup - 1); /* thread within its group */
		const int grp = (t - SH::fft_threads) / kStreamBoxGroup;
		const int bw = (t - SH::fft_threads) >> 5;                    /* warp within the role */
		int slot = 0, wsn = 0, par = 0, seq = 0;
		unsigned ph = 0;
		for (int seg = blockIdx.x; seg < prm.n_segs; seg += gridDim.x) {
			const int4 sg = prm.segs[seg];
			const int count = sg.z;
			for (int rd = 0; rd < count; ++rd) {
				const int rw = rd % RPW;
				const int buf = wsn & 1;
				if (rw == 0)
					mbar_wait(img_empty + buf, ((unsigned)(wsn >> 1) & 1u) ^ 1u); /* transform role has read it */
				c16 *img = image + buf * kWS + rw * N;
				int dI = 0, dQ = 0; /* |sum| <= N * 32768 / threads: fits */
				for (int c = 0; c < CPR; ++c, ++seq) {
					if ((seq & (BG - 1)) == grp) {
						mbar_wait(full + slot, ph);
						const uint8_t *p0 = stage + slot * chunk_bytes + bt * 2 * ds;
						const uint8_t *p1 = p0 + kStreamBoxGroup * 2 * ds;
						unsigned i0, q0, i1, q1;
						if ((ds & 7) == 0)
							boxcar_two_slot_sums<16>(p0, p1, 2 * ds, i0, q0, i1, q1);
						else if ((ds & 3) == 0)
							boxcar_two_slot_sums<8>(p0, p1, 2 * ds, i0, q0, i1, q1);
						else if ((ds & 1) == 0)
							boxcar_two_slot_sums<4>(p0, p1, 2 * ds, i0, q0, i1, q1);
						else
							boxcar_two_slot_sums<2>(p0, p1, 2 * ds, i0, q0, i1, q1);
						const c16 v0 = c16_pack((int)i0 - 127 * ds, (int)q0 - 127 * ds);
						const c16 v1 = c16_pack((int)i1 - 127 * ds, (int)q1 - 127 * ds);
						img[c * kThreads + bt] = v0;
						img[c * kThreads + bt + kStreamBoxGroup] = v1;
						dI += c16_re(v0) + c16_re(v1); /* remove_dc sums the wrapped int16 values */
						dQ += c16_im(v0) + c16_im(v1);
						warp_sync();
						if ((bt & 31) == 0)
							mbar_arrive(empty + slot); /* this warp is done with the slot */
					}
					if (++slot == nslots) {
						slot = 0;
						ph ^= 1u;
					}
				}
				/* ---- the read is complete: its DC averages (divisors 2N and 2N-1) ---- */
#pragma unroll
				for (int o = 16; o > 0; o >>= 1) {
					dI += __shfl_xor_sync(0xffffffffu, dI, o);
					dQ += __shfl_xor_sync(0xffffffffu, dQ, o);
				}
				int *rr = red + par * 16; /* alternating: rewritten two reads later, one barrier in between */
				par ^= 1;
				if ((bt & 31) == 0) {
					rr[bw * 2] = dI;
					rr[bw * 2 + 1] = dQ;
				}
				named_bar_sync(4, SH::box_threads);
				if (t == SH::fft_threads) {
					long long sI = 0, sQ = 0;
#pragma unroll
					for (int w = 0; w < SH::box_threads / 32; ++w) {
						sI += rr[2 * w];
						sQ += rr[2 * w + 1];
					}
					dc[(buf * 16 + rw) * 2] = dc_average(sI, 2 * N);
					dc[(buf * 16 + rw) * 2 + 1] = dc_average(sQ, 2 * N - 1);
				}
				if (rw == RPW - 1 || rd == count - 1) {
					mbar_arrive(img_full + buf); /* release: image and averages are visible to the waiters */
					++wsn;
				}
			}
		}
		return;
	}

	/* ================= transform role ================= */
	/* group fg takes the working sets with number = fg (mod FG); its threads are tf = 0..255 */
	const int fg = t / kStreamFftThreads, tf = t % kStreamFftThreads;
	c16 *xch = (c16 *)(smem + SM::off_xch) + fg * 2 * kXchWords;
	for (int i = t; i < (N - 16) / 2; i += SH::fft_threads)
		cp_async16((uint8_t *)tws + 16 * i, (const uint8_t *)prm.twc + 16 * i);
	for (int i = t; i < N / 8; i += SH::fft_threads)
		cp_async16((uint8_t *)wins + 16 * i, (const uint8_t *)prm.win + 16 * i);
	cp_async_commit();
	cp_async_wait_all();
	named_bar_sync(3, SH::fft_threads); /* tables complete for every transform thread */

	TwSmall<L> tw;
	tw.tws = tws;
	tw.tw0 = &prm.tw0;
	int t0;
	const int trev = front_thread_map<L>(tf, t0);
	const int myblk = tf >> (L - 4);
	const int blkbase = myblk << L;
	int flip = 0, wsn = 0;
	const GroupBar fft_bar = { 1 + fg, kStreamFftThreads };

	for (int seg = blockIdx.x; seg < prm.n_segs; seg += gridDim.x) {
		const int4 sg = prm.segs[seg];
		const int hop = sg.x, count = sg.z;
		unsigned long long acc[kPts];
#pragma unroll
		for (int r = 0; r < kPts; ++r)
			acc[r] = 0ull;

		for (int rd0 = 0; rd0 < count; rd0 += RPW, ++wsn) {
			if (FG > 1 && (wsn & (FG - 1)) != fg)
				continue;
			const int nvalid = (count - rd0 < RPW) ? count - rd0 : RPW;
			const int buf = wsn & 1;
			mbar_wait(img_full + buf, (unsigned)(wsn >> 1) & 1u);
			const c16 *img = image + buf * kWS;
			const int kI = dc[(buf * 16 + myblk) * 2], kQ = dc[(buf * 16 + myblk) * 2 + 1];

			/* ---- DC, window, bit-reversed placement ---- */
			X2 x[kPts];
#pragma unroll
			for (int r = 0; r < kPts; ++r) {
				const int nblk = (brev4(r) << (L - 4)) + trev;
				const c16 raw = img[blkbase + nblk];
				const int wv = wins[nblk];
				x[r].re = ((c16_re(raw) - kI) * wv) << 16;
				x[r].im = ((c16_im(raw) - kQ) * wv) << 16;
			}
			mbar_arrive(img_empty + buf); /* the boxcar role may refill this image */

			engine_fft_db<L, TwSmall<L>, GroupBar>(x, xch, flip, tf, tw, fft_bar, t0);
#pragma unroll
			for (int r = 0; r < kPts; ++r) {
				const int re = x[r].re >> 16, im = x[r].im >> 16;
				if ((last_pos<L>(tf, r) >> L) < nvalid)
					accumulate_power<PEAK>(acc[r], re, im);
			}
		}

		pdl_wait();
		if (t == 0)
			atomicAdd((unsigned long long *)(prm.samples + hop), (unsigned long long)((long long)count * ds));
		/* both transpose buffers are idle here (2 * kXchWords * 4 >= N * 8): every transform thread is past its
		 * last exchange read once it has passed the first barrier in flush_bins */
		flush_bins<L, PEAK, GroupBar>(acc, prm.avg + ((long long)hop << L), (unsigned long long *)xch, tf, fft_bar);
	}
}

/*
 * Symmetric variant of the warp-specialised narrow-scan kernel: instead of dedicated boxcar and
 * transform roles two pipelines share the CTA (and the twiddle / window tables), each with its
 * own producer lane, its own ring and a WORKER group of 8 warps that owns alternate working sets
 * end to end -- sum the working set's chunks out of the ring into a
 * private 4096-sample image (one output slot per thread and chunk), take the DC averages, then
 * run the register-blocked transform on it.  While one group transforms, the other sums; no warp
 * idles in a role that has nothing to do (in the three-role kernel the transform role waits for
 * images 58 % of its time at ds = 28 while the boxcar warps are the limit), and no image hand-off
 * barriers are needed.  544 threads, so the transform keeps its 117 registers.
 */
constexpr int kSymGroups = 2;
constexpr int kSymThreads = kSymGroups * kThreads + kSymGroups * 32; /* + one producer warp per pipeline */

template <int L>
struct SymSmem {
	static constexpr int N = 1 << L;
	static constexpr int off_image = 0;                                   /* one 4096 c16 image per group */
	static constexpr int off_xch = kSymGroups * kWS * 4;                  /* two transpose buffers per group */
	static constexpr int off_tw = off_xch + kSymGroups * 2 * kXchWords * 4;
	static constexpr int off_win = off_tw + (N - 16) * 8;
	static constexpr int off_red = (off_win + N * 2 + 15) & ~15;          /* [group][2][8 warps][2] int */
	static constexpr int off_bar = off_red + kSymGroups * 2 * 16 * 4;     /* full[group][16] empty[group][16] */
	static constexpr int off_stage = (off_bar + 2 * kSymGroups * kStreamMaxSlots * 8 + 127) & ~127;
	static int bytes(int ds, int slots) { return off_stage + kSymGroups * slots * 512 * ds; } /* slots per group */
};

/* byte sums of one boxcar slot: I = even addresses, Q = odd addresses of [p, p + nbytes) */
template <int ALIGN>
SCAN_DEV void boxcar_one_slot_sums(const uint8_t *p, int nbytes, unsigned &si, unsigned &sq)
{
	unsigned a0 = 0, a1 = 0, a2 = 0, a3 = 0, b0 = 0, b1 = 0, b2 = 0, b3 = 0;
	if constexpr (ALIGN == 16) {
#pragma unroll 2
		for (int o = 0; o < nbytes; o += 16) {
			const uint4 q = *(const uint4 *)(p + o);
			a0 = __dp4a(q.x, 0x00010001u, a0); b0 = __dp4a(q.x, 0x01000100u, b0);
			a1 = __dp4a(q.y, 0x00010001u, a1); b1 = __dp4a(q.y, 0x01000100u, b1);
			a2 = __dp4a(q.z, 0x00010001u, a2); b2 = __dp4a(q.z, 0x01000100u, b2);
			a3 = __dp4a(q.w, 0x00010001u, a3); b3 = __dp4a(q.w, 0x01000100u, b3);
		}
	} else if constexpr (ALIGN == 8) {
#pragma unroll 4
		for (int o = 0; o < nbytes; o += 8) {
			const uint2 q = *(const uint2 *)(p + o);
			a0 = __dp4a(q.x, 0x00010001u, a0); b0 = __dp4a(q.x, 0x01000100u, b0);
			a1 = __dp4a(q.y, 0x00010001u, a1); b1 = __dp4a(q.y, 0x01000100u, b1);
		}
	} else if constexpr (ALIGN == 4) {
#pragma unroll 4
		for (int o = 0; o < nbytes; o += 4) {
			const unsigned q = *(const unsigned *)(p + o);
			a0 = __dp4a(q, 0x00010001u, a0);
			b0 = __dp4a(q, 0x01000100u, b0);
		}
	} else {
#pragma unroll 4
		for (int o = 0; o < nbytes; o += 2) {
			const unsigned q = *(const uint16_t *)(p + o);
			a0 += q & 0xFFu;
			b0 += q >> 8;
		}
	}
	si = (a0 + a1) + (a2 + a3);
	sq = (b0 + b1) + (b2 + b3);
}

template <int L, bool PEAK>
__global__ void __launch_bounds__(kSymThreads, 1)
scan_boxcar_sym_kernel(const SCAN_GRID_CONSTANT FusedBoxcarParams prm)
{
	SCAN_DYN_SMEM(smem);
	typedef SymSmem<L> SM;
	constexpr int N = 1 << L;
	constexpr int RPW = kWS / N;      /* reads per working set */
	constexpr int CPR = N / kThreads; /* 256-slot chunks per read */
	int2 *tws = (int2 *)(smem + SM::off_tw);
	uint16_t *wins = (uint16_t *)(smem + SM::off_win);

	/* prm.slots = ring depth PER GROUP: each group has its own ring and its own producer lane, so every
	 * transaction barrier has exactly one consumer group, which sees every phase of it in order (a parity
	 * wait may never skip a phase) */
	const int t = threadIdx.x, ds = prm.ds, nslots = prm.slots;
	const int chunk_bytes = 512 * ds;
	const int role = t / kThreads; /* 0, 1: worker groups; 2: the producer warps */
	const int pg = role < kSymGroups ? role : (t - kSymGroups * kThreads) / 32; /* pipeline this thread belongs to */
	uint64_t *full = (uint64_t *)(smem + SM::off_bar) + pg * kStreamMaxSlots;
	uint64_t *empty = full + kSymGroups * kStreamMaxSlots;
	uint8_t *stage = smem + SM::off_stage + pg * nslots * chunk_bytes;
	if (t == 0) {
		for (int g = 0; g < kSymGroups; ++g)
			for (int s = 0; s < nslots; ++s) {
				mbar_init((uint64_t *)(smem + SM::off_bar) + g * kStreamMaxSlots + s, 1);
				mbar_init((uint64_t *)(smem + SM::off_bar) + (kSymGroups + g) * kStreamMaxSlots + s, kThreads / 32);
			}
		mbar_fence_init();
	}
	__syncthreads();

	if (role >= kSymGroups) {
		/* ================= producers: one lane per pipeline ================= */
		if ((t & 31) != 0)
			return;
		int slot = 0, wsn = 0;
		unsigned ph = 0;
		for (int seg = blockIdx.x; seg < prm.n_segs; seg += gridDim.x) {
			const int4 sg = prm.segs[seg];
			for (int rd0 = 0; rd0 < sg.z; rd0 += RPW, ++wsn) {
				if ((wsn & (kSymGroups - 1)) != pg)
					continue;
				const int nvalid = (sg.z - rd0 < RPW) ? sg.z - rd0 : RPW;
				produce_reads<CPR>(prm, sg.y + rd0, nvalid, stage, full, empty, chunk_bytes, nslots, slot, ph);
			}
		}
		return;
	}

	/* ================= worker groups ================= */
	const int fg = t / kThreads, tf = t % kThreads;
	c16 *image = (c16 *)(smem + SM::off_image) + fg * kWS;
	c16 *xch = (c16 *)(smem + SM::off_xch) + fg * 2 * kXchWords;
	int *red = (int *)(smem + SM::off_red) + fg * 32;
	const GroupBar bar = { 1 + fg, kThreads };
	load_tables<L>(tws, wins, prm.twc, prm.win, t, kSymGroups * kThreads);
	cp_async_commit();
	cp_async_wait_all();
	named_bar_sync(3, kSymGroups * kThreads); /* tables complete for every worker */

	TwSmall<L> tw;
	tw.tws = tws;
	tw.tw0 = &prm.tw0;
	int t0;
	const int trev = front_thread_map<L>(tf, t0);
	const int myblk = tf >> (L - 4);
	const int blkbase = myblk << L;
	int flip = 0, wsn = 0, par = 0;
	int slot = 0; /* position in this group's own ring */
	unsigned ph = 0;

	for (int seg = blockIdx.x; seg < prm.n_segs; seg += gridDim.x) {
		const int4 sg = prm.segs[seg];
		const int hop = sg.x, count = sg.z;
		unsigned long long acc[kPts];
#pragma unroll
		for (int r = 0; r < kPts; ++r)
			acc[r] = 0ull;

		for (int rd0 = 0; rd0 < count; rd0 += RPW, ++wsn) {
			const int nvalid = (count - rd0 < RPW) ? count - rd0 : RPW;
			if ((wsn & (kSymGroups - 1)) != fg)
				continue; /* the other pipeline's working set */
			int kI = 0, kQ = 0;
			/* ---- boxcar: sum this working set's chunks out of the ring (rtl_power.c:666-681) ---- */
			for (int rw = 0; rw < nvalid; ++rw) {
				int dI = 0, dQ = 0; /* |sum| <= N * 32768 / 256 per thread: fits */
				for (int c = 0; c < CPR; ++c) {
					mbar_wait(full + slot, ph);
					const uint8_t *p = stage + slot * chunk_bytes + tf * 2 * ds;
					unsigned ui, uq;
					if ((ds & 7) == 0)
						boxcar_one_slot_sums<16>(p, 2 * ds, ui, uq);
					else if ((ds & 3) == 0)
						boxcar_one_slot_sums<8>(p, 2 * ds, ui, uq);
					else if ((ds & 1) == 0)
						boxcar_one_slot_sums<4>(p, 2 * ds, ui, uq);
					else
						boxcar_one_slot_sums<2>(p, 2 * ds, ui, uq);
					const c16 v = c16_pack((int)ui - 127 * ds, (int)uq - 127 * ds);
					image[rw * N + c * kThreads + tf] = v;
					dI += c16_re(v); /* remove_dc sums the wrapped int16 values */
					dQ += c16_im(v);
					warp_sync();
					if ((tf & 31) == 0)
						mbar_arrive(empty + slot); /* this warp is done with the slot */
					if (++slot == nslots) {
						slot = 0;
						ph ^= 1u;
					}
				}
				/* the read is complete: its DC averages (divisors 2N and 2N-1, rtl_power.c:581-596) */
#pragma unroll
				for (int o = 16; o > 0; o >>= 1) {
					dI += __shfl_xor_sync(0xffffffffu, dI, o);
					dQ += __shfl_xor_sync(0xffffffffu, dQ, o);
				}
				int *rr = red + par * 16; /* alternating: rewritten two reads later, one barrier in between */
				par ^= 1;
				if ((tf & 31) == 0) {
					rr[(tf >> 5) * 2] = dI;
					rr[(tf >> 5) * 2 + 1] = dQ;
				}
				bar.sync(); /* also: the image rows of this read are complete */
				if (myblk == rw) {
					long long sI = 0, sQ = 0;
#pragma unroll
					for (int w = 0; w < kThreads / 32; ++w) {
						sI += rr[2 * w];
						sQ += rr[2 * w + 1];
					}
					kI = dc_average(sI, 2 * N);
					kQ = dc_average(sQ, 2 * N - 1);
				}
			}

			/* ---- DC, window, bit-reversed placement, transform, |X|^2 ---- */
			X2 x[kPts];
#pragma unroll
			for (int r = 0; r < kPts; ++r) {
				const int nblk = (brev4(r) << (L - 4)) + trev;
				const c16 raw = image[blkbase + nblk];
				const int wv = wins[nblk];
				x[r].re = ((c16_re(raw) - kI) * wv) << 16;
				x[r].im = ((c16_im(raw) - kQ) * wv) << 16;
			}
			engine_fft_db<L, TwSmall<L>, GroupBar>(x, xch, flip, tf, tw, bar, t0);
#pragma unroll
			for (int r = 0; r < kPts; ++r) {
				const int re = x[r].re >> 16, im = x[r].im >> 16;
				if ((last_pos<L>(tf, r) >> L) < nvalid)
					accumulate_power<PEAK>(acc[r], re, im);
			}
		}

		pdl_wait();
		if (t == 0)
			atomicAdd((unsigned long long *)(prm.samples + hop), (unsigned long long)((long long)count * ds));
		/* the group's transpose buffers are idle here: 2 * kXchWords * 4 >= N * 8 */
		flush_bins<L, PEAK, GroupBar>(acc, prm.avg + ((long long)hop << L), (unsigned long long *)xch, tf, bar);
	}
}

/* ======================================================================== *
 *  rms_power: 1-bin hops (rtl_power.c:410-436)                              *
 * ======================================================================== */

struct RmsParams {
	const uint8_t *base;
	const long long *read_off;
	const int *hop_of;   /* hop of entry e */
	int n_reads;
	int buf_len;
	int peak;
	long long *avg;      /* [tune_count] */
	long long *samples;  /* [tune_count], += 1 per read (rtl_power.c:435) */
};

/* One warp per read: 512-byte coalesced rows, 8 x LDG.128 in flight per lane,
 * sum(b) and sum(b*b) with IDP.4A, everything else exact int64 per read. */
__global__ void __launch_bounds__(256)
rms_kernel(const SCAN_GRID_CONSTANT RmsParams prm)
{
	const int lane = threadIdx.x & 31;
	const int warps = (gridDim.x * blockDim.x) >> 5;
	for (int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < prm.n_reads; e += warps) {
		const uint8_t *src = prm.base + prm.read_off[e];
		unsigned sb = 0, sbb = 0; /* per lane <= 2^21/32 bytes: fits */
		for (int i = lane * 16; i < prm.buf_len; i += 32 * 16 * 8) {
			uint4 q[8];
#pragma unroll
			for (int j = 0; j < 8; ++j)
				q[j] = (i + j * 512 < prm.buf_len) ? __ldg((const uint4 *)(src + i + j * 512)) : uint4{ 0, 0, 0, 0 };
#pragma unroll
			for (int j = 0; j < 8; ++j) {
				sb = __dp4a(q[j].x, 0x01010101u, sb); sbb = __dp4a(q[j].x, q[j].x, sbb);
				sb = __dp4a(q[j].y, 0x01010101u, sb); sbb = __dp4a(q[j].y, q[j].y, sbb);
				sb = __dp4a(q[j].z, 0x01010101u, sb); sbb = __dp4a(q[j].z, q[j].z, sbb);
				sb = __dp4a(q[j].w, 0x01010101u, sb); sbb = __dp4a(q[j].w, q[j].w, sbb);
			}
		}
		long long tb = sb, tbb = sbb;
#pragma unroll
		for (int o = 16; o > 0; o >>= 1) {
			tb += __shfl_xor_sync(0xffffffffu, tb, o);
			tbb += __shfl_xor_sync(0xffffffffu, tbb, o);
		}
		if (lane == 0) {
			/* s = b - 127:  sum s = sum b - 127 n,  sum s^2 = sum b^2 - 254 sum b + 127^2 n */
			const long long n = prm.buf_len;
			const long long t = tb - 127 * n;
			long long p = tbb - 254 * tb + 16129 * n;
			/* same IEEE double operations, in the reference's order, no FMA contraction */
			const double dn = (double)prm.buf_len;
			const double dc = __ddiv_rn((double)t, dn);
			const double err = __dsub_rn(__dmul_rn((double)(t * 2), dc), __dmul_rn(__dmul_rn(dc, dc), dn));
			p -= (long long)round(err);
			pdl_wait(); /* the accumulators may still be read by the previous interval's report epilogue */
			atomicAdd((unsigned long long *)(prm.samples + prm.hop_of[e]), 1ull);
			long long *dst = prm.avg + prm.hop_of[e];
			if (prm.peak)
				atomicMax(dst, p);
			else
				atomicAdd((unsigned long long *)dst, (unsigned long long)p);
		}
	}
}

/*
 * The same result with one CTA per read (the planner's rms reads are always 16384 bytes): 256 threads x 4 x 16 bytes
 * = one read in flight per CTA plus the next one already requested while this one is reduced, i.e. ~1200 long
 * sequential streams on the device instead of ~9500 warp-private ones, and one barrier per read (the per-warp
 * partials alternate between two buffers; thread 0 finishes read e while the others already sum read e+1).
 */
constexpr int kRmsCtaBytes = 16384;

__global__ void __launch_bounds__(256)
rms_cta_kernel(const SCAN_GRID_CONSTANT RmsParams prm)
{
	__shared__ unsigned part[2][8][2];
	const int t = threadIdx.x, lane = t & 31, w = t >> 5;
	int e = blockIdx.x;
	if (e >= prm.n_reads)
		return;
	uint4 cur[4], nxt[4];
	{
		const uint8_t *src = prm.base + prm.read_off[e];
#pragma unroll
		for (int j = 0; j < 4; ++j)
			cur[j] = __ldg((const uint4 *)(src + (t + 256 * j) * 16));
	}
	int par = 0;
	bool waited = false;
	for (; e < prm.n_reads; e += gridDim.x) {
		const int en = e + gridDim.x;
		if (en < prm.n_reads) {
			const uint8_t *src = prm.base + prm.read_off[en];
#pragma unroll
			for (int j = 0; j < 4; ++j)
				nxt[j] = __ldg((const uint4 *)(src + (t + 256 * j) * 16));
		}
		unsigned sb = 0, sbb = 0; /* per warp <= 2048 bytes: 2048 * 255^2 fits */
#pragma unroll
		for (int j = 0; j < 4; ++j) {
			sb = __dp4a(cur[j].x, 0x01010101u, sb); sbb = __dp4a(cur[j].x, cur[j].x, sbb);
			sb = __dp4a(cur[j].y, 0x01010101u, sb); sbb = __dp4a(cur[j].y, cur[j].y, sbb);
			sb = __dp4a(cur[j].z, 0x01010101u, sb); sbb = __dp4a(cur[j].z, cur[j].z, sbb);
			sb = __dp4a(cur[j].w, 0x01010101u, sb); sbb = __dp4a(cur[j].w, cur[j].w, sbb);
		}
#pragma unroll
		for (int o = 16; o > 0; o >>= 1) {
			sb += __shfl_xor_sync(0xffffffffu, sb, o);
			sbb += __shfl_xor_sync(0xffffffffu, sbb, o);
		}
		if (lane == 0) {
			part[par][w][0] = sb;
			part[par][w][1] = sbb;
		}
		__syncthreads();
		if (t == 0) {
			long long tb = 0, tbb = 0;
#pragma unroll
			for (int k = 0; k < 8; ++k) {
				tb += part[par][k][0];
				tbb += part[par][k][1];
			}
			/* s = b - 127:  sum s = sum b - 127 n,  sum s^2 = sum b^2 - 254 sum b + 127^2 n */
			const long long n = kRmsCtaBytes;
			const long long ts = tb - 127 * n;
			long long p = tbb - 254 * tb + 16129 * n;
			/* same IEEE double operations, in the reference's order, no FMA contraction (rtl_power.c:410-436) */
			const double dn = (double)kRmsCtaBytes;
			const double dc = __ddiv_rn((double)ts, dn);
			const double err = __dsub_rn(__dmul_rn((double)(ts * 2), dc), __dmul_rn(__dmul_rn(dc, dc), dn));
			p -= (long long)round(err);
			if (!waited)
				pdl_wait(); /* the accumulators may still be read by the previous interval's report epilogue */
			waited = true;
			atomicAdd((unsigned long long *)(prm.samples + prm.hop_of[e]), 1ull);
			long long *dst = prm.avg + prm.hop_of[e];
			if (prm.peak)
				atomicMax(dst, p);
			else
				atomicAdd((unsigned long long *)dst, (unsigned long long)p);
		}
		par ^= 1;
#pragma unroll
		for (int j = 0; j < 4; ++j)
			cur[j] = nxt[j];
	}
}

/* ======================================================================== *
 *  Soft-AGC byte statistics (src/librtlsdr.c:3288-3306), optional            *
 * ======================================================================== */

struct LevelParams {
	const uint8_t *base;
	const long long *read_off;
	const int *hop_of;
	int n_reads;
	int buf_len;
	unsigned long long *level; /* [tune_count][2]: overload, high level */
};

/* one warp per read; four bytes per compare with the SIMD-in-a-word intrinsics */
__global__ void __launch_bounds__(256)
level_stats_kernel(const SCAN_GRID_CONSTANT LevelParams prm)
{
	const int lane = threadIdx.x & 31;
	const int warps = (gridDim.x * blockDim.x) >> 5;
	for (int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < prm.n_reads; e += warps) {
		const uint8_t *src = prm.base + prm.read_off[e];
		unsigned over = 0, high = 0;
		for (int i = lane * 16; i < prm.buf_len; i += 32 * 16) {
			const uint4 q = __ldg((const uint4 *)(src + i));
			const unsigned w[4] = { q.x, q.y, q.z, q.w };
#pragma unroll
			for (int j = 0; j < 4; ++j) {
				over += __popc(__vcmpeq4(w[j], 0u) | __vcmpeq4(w[j], 0xFFFFFFFFu)) >> 3;   /* u == 0 || u == 255 */
				high += __popc(__vcmpltu4(w[j], 0x40404040u) | __vcmpgtu4(w[j], 0xBFBFBFBFu)) >> 3; /* u < 64 || u > 191 */
			}
		}
#pragma unroll
		for (int o = 16; o > 0; o >>= 1) {
			over += __shfl_xor_sync(0xffffffffu, over, o);
			high += __shfl_xor_sync(0xffffffffu, high, o);
		}
		if (lane == 0) {
			atomicAdd(prm.level + 2 * prm.hop_of[e], (unsigned long long)over);
			atomicAdd(prm.level + 2 * prm.hop_of[e] + 1, (unsigned long long)high);
		}
	}
}

/* ======================================================================== *
 *  Report epilogue: DC nuke, half swap, crop, dB (rtl_power.c:722-760)      *
 * ======================================================================== */

struct EpilogueParams {
	const long long *avg;     /* [hops << bin_e] natural order */
	const long long *samples; /* [hops] */
	double *db;               /* [hops][db_count], indexed from hop0 */
	long long *avg_out;       /* optional copy of the raw bins, indexed from hop0 */
	int *samples_out;         /* optional, indexed from hop0 */
	int bin_e;
	int i1, i2;               /* first / last printed bin of the swapped spectrum */
	int rate;
	int hop0;                 /* first hop to process */
	unsigned *done;           /* optional [hops]: blocks finished per hop; the last one zeroes the hop */
	long long *avg_rw;        /* same memory as avg when `done` is set */
	long long *samples_rw;
	double *iir;              /* optional [hops][db_count - 1] smoothing state (-s iir), NaN = no report yet */
	double iir_alpha;
};

/* the bin as the dB chain's first double: (double)avg, times 2^-8 (exact) for guard-bit bins */
template <bool GUARD>
SCAN_DEV double epilogue_value(long long v)
{
	if constexpr (GUARD)
		return __dmul_rn((double)v, 0x1p-8);
	else
		return (double)v;
}

/* one launch per report: dB row, raw-bin copy and sample count of every hop */
__global__ void __launch_bounds__(256)
epilogue_kernel(const SCAN_GRID_CONSTANT EpilogueParams prm)
{
	constexpr bool GUARD = false;
#include "epilogue_body.inl"
}

/* the same for a RTLSDR_GPU_FLAG_GUARD_BITS handle */
__global__ void __launch_bounds__(256)
epilogue_guard_kernel(const SCAN_GRID_CONSTANT EpilogueParams prm)
{
	constexpr bool GUARD = true;
#include "epilogue_body.inl"
}

/* ======================================================================== *
 *  Merging accumulator sets (reads of ONE hop sharded over several GPUs)     *
 * ======================================================================== */

/*
 * tunes[i].avg is a sum (or, with -P, a maximum) of per-read |X|^2 and tunes[i].samples a sum of per-read counts
 * (rtl_power.c:708-717): both are associative and exact in int64, so the reads of one hop can be split over
 * several handles / GPUs and their raw accumulators combined afterwards -- the report computed from the merged
 * integers is bit-identical to a single handle's.  `sets` external sets (raw bins as rtlsdr_gpu_scan_collect_device
 * writes them, int32 sample counts) are folded into the handle's accumulators; the external memory may be a peer
 * mapping (the slots the other GPUs' epilogues stored into over NVLink).
 */
struct MergeParams {
	long long *avg;          /* [bins] this handle's accumulators */
	long long *samples;      /* [hops] */
	const uint8_t *ext_avg;  /* set s: int64 [bins] at ext_avg + s * stride */
	const uint8_t *ext_smp;  /* set s: int32 [hops] at ext_smp + s * stride */
	long long stride;
	long long bins;
	int hops;
	int sets;
	int peak;
};

__global__ void __launch_bounds__(256)
merge_sets_kernel(const SCAN_GRID_CONSTANT MergeParams prm)
{
	const long long step = (long long)gridDim.x * blockDim.x;
	const long long first = (long long)blockIdx.x * blockDim.x + threadIdx.x;
	for (long long i = first; i < prm.bins; i += step) {
		long long v = prm.avg[i];
		for (int s = 0; s < prm.sets; ++s) {
			const long long e = ((const long long *)(prm.ext_avg + s * prm.stride))[i];
			v = prm.peak ? (e > v ? e : v) : v + e;
		}
		prm.avg[i] = v;
	}
	for (long long i = first; i < prm.hops; i += step) {
		long long v = prm.samples[i];
		for (int s = 0; s < prm.sets; ++s)
			v += ((const int *)(prm.ext_smp + s * prm.stride))[i];
		prm.samples[i] = v;
	}
}

/* ======================================================================== *
 *  Device-side flags for the per-interval report exchange (multi-GPU)       *
 * ======================================================================== */

/*
 * The report epilogue of every rank stores straight into rank 0's memory (NVLink peer mapping).  What is left of
 * a "gather" is telling rank 0 that a slot is complete and telling the writers that rank 0 has consumed it: one
 * 32-bit flag per (buffer, rank), written with a system-scope release store by a one-thread kernel behind the
 * epilogue, and awaited by a kernel whose threads SLEEP between polls -- a waiter that spins (or a collective's
 * CTAs) takes issue slots from the transform CTAs of the SM it lands on, and with the transform's static
 * equal-run schedule one slowed SM delays the whole launch (measured at 8 GPUs: transform 545 us per interval
 * with a spinning barrier kernel, 513 us without).
 */
__global__ void flag_signal_kernel(unsigned *flag, unsigned value)
{
#ifdef SCAN_EMU
	*flag = value;
#else
	__threadfence_system();
	asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(value) : "memory");
#endif
}

/* the same for up to 32 flags at different addresses (rank 0 raising "interval consumed" in every rank's memory) */
constexpr int kFlagSignalMax = 32;
struct FlagList {
	unsigned *flag[kFlagSignalMax];
};

__global__ void flag_signal_many_kernel(const FlagList list, int count, unsigned value)
{
	const int i = threadIdx.x;
	if (i >= count)
		return;
#ifdef SCAN_EMU
	*list.flag[i] = value;
#else
	__threadfence_system();
	asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(list.flag[i]), "r"(value) : "memory");
#endif
}

/* thread i waits until flags[i] - value >= 0 (wrap-safe); gives up after about `timeout_ns` and reports it */
__global__ void flag_wait_kernel(const unsigned *flags, int count, unsigned value, unsigned long long timeout_ns,
				 unsigned *timed_out)
{
	const int i = threadIdx.x;
	if (i >= count)
		return;
#ifdef SCAN_EMU
	(void)flags; (void)value; (void)timeout_ns; (void)timed_out;
#else
	unsigned long long t0;
	asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
	unsigned sleep_ns = 64;
	for (;;) {
		unsigned v;
		asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + i) : "memory");
		if ((int)(v - value) >= 0)
			break;
		__nanosleep(sleep_ns);
		if (sleep_ns < 2048)
			sleep_ns *= 2;
		unsigned long long t1;
		asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
		if (t1 - t0 > timeout_ns) {
			if (timed_out)
				atomicExch(timed_out, 1u);
			break;
		}
	}
#endif
}

} // namespace rscan
