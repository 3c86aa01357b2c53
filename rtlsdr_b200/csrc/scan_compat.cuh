/*
 * scan_compat.cuh -- the handful of CUDA spellings the scan kernels use.
 *
 * Product builds (nvcc, sm_100a) take the first branch.  tests/emu/ compiles the
 * very same kernel source with g++ -DSCAN_EMU against tests/emu/cuda_emu.h (one
 * OS thread per CUDA thread, barriers for __syncthreads) so that the index math
 * of every kernel can be parity-checked on the GPU-less build box.  The emulator
 * is test infrastructure only; nothing in the shipped library can reach it.
 */
#pragma once
#include <stdint.h>

#ifdef SCAN_EMU
#include "cuda_emu.h"
#define SCAN_DYN_SMEM(name) unsigned char *name = ::cuda_emu::dyn_smem()
#define SCAN_GRID_CONSTANT
#else
#include <cuda_runtime.h>
#define SCAN_DYN_SMEM(name) extern __shared__ __align__(16) unsigned char name[]
#define SCAN_GRID_CONSTANT __grid_constant__
#endif

#define SCAN_DEV __device__ __forceinline__

namespace rscan {

/* 16-byte asynchronous global->shared copy (LDGSTS), commit and drain. */
SCAN_DEV void cp_async16(void *smem_dst, const void *gmem_src)
{
#ifdef SCAN_EMU
	::cuda_emu::copy16(smem_dst, gmem_src);
#else
	unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
	asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src) : "memory");
#endif
}

/* 8-byte form (LDGSTS.64): destinations that are only 8-byte aligned (swizzled tile rows of the large path) */
SCAN_DEV void cp_async8(void *smem_dst, const void *gmem_src)
{
#ifdef SCAN_EMU
	::cuda_emu::copy8(smem_dst, gmem_src);
#else
	unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
	asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem_src) : "memory");
#endif
}

SCAN_DEV void cp_async_commit()
{
#ifndef SCAN_EMU
	asm volatile("cp.async.commit_group;\n" ::: "memory");
#endif
}

SCAN_DEV void cp_async_wait_all()
{
#ifndef SCAN_EMU
	asm volatile("cp.async.wait_group 0;\n" ::: "memory");
#endif
}

/* wait until at most `pending` of the most recently committed copy groups are still in flight */
SCAN_DEV void cp_async_wait_pending(int pending)
{
#ifndef SCAN_EMU
	switch (pending) {
	case 0: asm volatile("cp.async.wait_group 0;\n" ::: "memory"); break;
	case 1: asm volatile("cp.async.wait_group 1;\n" ::: "memory"); break;
	case 2: asm volatile("cp.async.wait_group 2;\n" ::: "memory"); break;
	default: asm volatile("cp.async.wait_group 3;\n" ::: "memory"); break;
	}
#else
	(void)pending;
#endif
}

template <int PENDING>
SCAN_DEV void cp_async_wait_group()
{
#ifndef SCAN_EMU
	asm volatile("cp.async.wait_group %0;\n" ::"n"(PENDING) : "memory");
#endif
}

/*
 * Programmatic dependent launch (sm_90+): a kernel launched with the
 * programmatic-stream-serialization attribute may start while the previous
 * kernel in the stream is still running; pdl_wait() blocks until that kernel
 * has completed and its writes are visible, pdl_launch_dependents() lets the
 * next kernel start early.  Both are no-ops for ordinary launches.
 */
SCAN_DEV void pdl_wait()
{
#ifndef SCAN_EMU
	asm volatile("griddepcontrol.wait;\n" ::: "memory");
#endif
}

SCAN_DEV void pdl_launch_dependents()
{
#ifndef SCAN_EMU
	asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
#endif
}

/*
 * Transaction barriers (mbarrier), bulk asynchronous copies (the 1-D form of the
 * TMA engine) and named barriers: the producer / consumer plumbing of the
 * warp-specialised streaming kernel.  A wait on parity p returns once the phase
 * with that parity has completed; waiting for parity 1 on a freshly initialised
 * barrier returns at once (the "previous" phase counts as complete).
 */
SCAN_DEV void mbar_init(uint64_t *bar, int count)
{
#ifdef SCAN_EMU
	::cuda_emu::mbar_init(bar, count);
#else
	unsigned s = (unsigned)__cvta_generic_to_shared(bar);
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(s), "r"(count) : "memory");
#endif
}

/* make the initialised barriers visible to the async proxy (bulk copies) */
SCAN_DEV void mbar_fence_init()
{
#ifndef SCAN_EMU
	asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
	asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
#endif
}

SCAN_DEV void mbar_arrive(uint64_t *bar)
{
#ifdef SCAN_EMU
	::cuda_emu::mbar_arrive(bar, 0);
#else
	unsigned s = (unsigned)__cvta_generic_to_shared(bar);
	asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared::cta.b64 st, [%0];\n}\n" ::"r"(s) : "memory");
#endif
}

SCAN_DEV void mbar_arrive_expect_tx(uint64_t *bar, unsigned bytes)
{
#ifdef SCAN_EMU
	::cuda_emu::mbar_arrive(bar, bytes);
#elif defined(RSCAN_RACECHECK_COPY)
	(void)bar; (void)bytes; /* debug build: the producer's one arrival happens AFTER its copy, in bulk_copy_g2s */
#else
	unsigned s = (unsigned)__cvta_generic_to_shared(bar);
	asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n}\n" ::"r"(s), "r"(bytes)
		     : "memory");
#endif
}

SCAN_DEV void mbar_wait(uint64_t *bar, unsigned parity)
{
#ifdef SCAN_EMU
	::cuda_emu::mbar_wait(bar, parity);
#else
	unsigned s = (unsigned)__cvta_generic_to_shared(bar);
	asm volatile("{\n"
		     ".reg .pred p;\n"
		     "MBAR_WAIT:\n"
		     "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
		     "@p bra MBAR_DONE;\n"
		     "bra MBAR_WAIT;\n"
		     "MBAR_DONE:\n"
		     "}\n" ::"r"(s),
		     "r"(parity)
		     : "memory");
#endif
}

/* global -> shared bulk copy (16-byte aligned, size a multiple of 16); completion is
 * counted on `bar` as `bytes` transaction bytes */
SCAN_DEV void bulk_copy_g2s(void *smem_dst, const void *gmem_src, unsigned bytes, uint64_t *bar)
{
#ifdef SCAN_EMU
	::cuda_emu::bulk_copy(smem_dst, gmem_src, bytes, bar);
#elif defined(RSCAN_RACECHECK_COPY)
	/* Debug build for compute-sanitizer racecheck (tools/racecheck_stream.sh), never shipped: racecheck does not
	 * model the async proxy's writes completing through complete_tx, so it flags every staged read of the real
	 * build.  Here the SAME producer lane moves the chunk with ordinary loads / stores and then makes the ONE
	 * arrival the full[] barrier expects (arrive.expect_tx + complete_tx of the real build collapse into a
	 * plain arrive after the data is written): the full / empty protocol and every consumer are unchanged,
	 * only the copy engine and the arrival are ones the tool may understand. */
	{
		const uint4 *s = (const uint4 *)gmem_src;
		uint4 *d = (uint4 *)smem_dst;
		for (unsigned i = 0; i < bytes / 16; ++i)
			d[i] = s[i];
		__threadfence_block();
		mbar_arrive(bar);
	}
#else
	unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
	unsigned b = (unsigned)__cvta_generic_to_shared(bar);
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(d),
		     "l"(gmem_src), "r"(bytes), "r"(b)
		     : "memory");
#endif
}

/* barrier `id` (1..15) over `count` threads of the CTA (a multiple of 32) */
SCAN_DEV void named_bar_sync(int id, int count)
{
#ifdef SCAN_EMU
	::cuda_emu::named_bar_sync(id, count);
#else
	asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(count) : "memory");
#endif
}

/* sum (mod 2^32) over the 32 lanes of a full warp, returned to every lane: one REDUX instead of five
 * shuffle + add rounds */
SCAN_DEV unsigned warp_sum(unsigned v)
{
#ifdef SCAN_EMU
	for (int o = 16; o > 0; o >>= 1)
		v += __shfl_xor_sync(0xffffffffu, v, o);
	return v;
#else
	return __reduce_add_sync(0xffffffffu, v);
#endif
}

SCAN_DEV void warp_sync()
{
#ifdef SCAN_EMU
	::cuda_emu::warp_sync();
#else
	__syncwarp();
#endif
}

} // namespace rscan
