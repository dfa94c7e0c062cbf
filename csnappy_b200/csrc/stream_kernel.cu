// stream_kernel.cu -- parallel decoder of ONE long Snappy raw stream for sm_100a.
//
// csnappy_decompress_noheader (/root/reference/csnappy_decompress.c:319-387) walks one stream tag by tag:
// tag k+1 starts where tag k ends and a back-reference reads what earlier tags wrote, so a single stream
// offers no block-level parallelism and a warp that walks it serially (decompress_kernel.cu, global
// path) runs at ~30 MB/s.  This decoder breaks both chains:
//
//   1. TAG STARTS by speculation + pointer jumping.  Every input byte is parsed as if a tag started
//      there: next(p) = p + tag bytes, O(p) = output bytes.  The real tags are the orbit of 0 under next.
//      A CTA owns a chunk of kChunk input bytes in shared memory and doubles next/O synchronously
//      (Wyllie list ranking) until every position knows where it LEAVES the chunk and how many output
//      bytes that takes (exit_kernel).  A single thread then hops from chunk to chunk (chain_kernel:
//      n / kChunk dependent loads) and records where the real chain enters each chunk and at which
//      output offset.
//   2. TAGS of a chunk from its entry point (expand_kernel): the same doubling, stopped after 6 rounds,
//      gives jumps of exactly 64 tags; one thread walks those (<= 33 steps), 33 threads walk 64 single
//      steps each, and the chunk's tag list with output offsets is complete.  Warps then run the tags:
//      literals are copied input -> output at once; for every output byte of a copy only its SOURCE
//      index is recorded: S[o] = o - offset (S[o] = o for literal bytes).
//   3. BACK-REFERENCES by pointer jumping over the output (resolve_kernel, cooperative launch):
//      S[o] <- S[S[o]] until every chain ends at a literal byte -- log2(depth) rounds, a run of
//      offset-1 copies over a megabyte needs 20 -- then out[o] = out[S[o]].
//
// Errors keep the reference's order: every real tag is checked where its output offset is known (offset
// == 0 or > produced: -5, then space: -3; literal: payload cut off: -5, then space: -3; header cut off by
// the end of input: -5, defined here) and the failing tag with the smallest input position wins
// (atomicMin on position * 4 + rank).  Nothing is written at or past `cap`.
// Tables: 8 bytes per input byte (exit table) + 8 per chunk, 4 bytes per output byte (S).
#include <cooperative_groups.h>

#include "device_common.cuh"
#include "kernels.h"

namespace cg = cooperative_groups;

namespace csb {

constexpr uint32_t kChunk = 4096;      // input bytes per CTA
constexpr int kSThreads = 512;	       // kChunk / 8 positions per thread
constexpr uint32_t kPer = kChunk / kSThreads;
constexpr uint32_t kTerminal = 0xffffffffu;  // "the chain ends at this tag with an error"
constexpr uint32_t kNone = 0xffffffffu;
constexpr uint32_t kTagSlots = kChunk / 2 + 64;   // a tag is at least 2 bytes long
constexpr uint32_t kSpineSlots = kChunk / 128 + 2;  // one entry per 64 tags
constexpr size_t kExpandSmem = 8 * (2 * kChunk + kTagSlots + kSpineSlots) + kChunk + 8;
constexpr int S_OK = 0, S_OUTPUT_OVERRUN = -3, S_DATA_MALFORMED = -5;

struct StreamCtl {  // device-side control block (aux_in + 0)
	unsigned long long err_key;  // min over failing tags of position * 4 + rank (rank 0: -5, 1: -3)
	uint32_t end_pos;	     // where the chain stopped: n, or kTerminal
	uint32_t total;		     // output bytes of the whole chain (saturated)
	uint32_t flags[40];	     // per-round "something changed" words of resolve_kernel
};

__device__ __forceinline__ uint32_t sat_add(uint32_t a, uint32_t b)
{
	const uint32_t s = a + b;
	return s < a ? 0xffffffffu : s;
}

// One speculative tag at absolute position p (local index q of the staged chunk `sm`, which holds 8 bytes of
// lookahead): -> (next position | kTerminal, output bytes).  csnappy_decompress.c:345-382 without the copies.
__device__ __forceinline__ uint2 tag_step(const uint8_t *sm, uint32_t q, uint32_t p, uint32_t n)
{
	const uint32_t tag = sm[q], kind = tag & 3u, lf = tag >> 2, avail = n - p;
	if (kind == 0) {
		uint32_t len = lf + 1, hdr = 1;
		if (lf >= 60) {
			const uint32_t nb = lf - 59;
			if (avail - 1 < nb)
				return make_uint2(kTerminal, 0);
			uint32_t v = 0;
			for (uint32_t b = 0; b < nb; ++b)
				v |= (uint32_t)sm[q + 1 + b] << (8 * b);
			len = v + 1;
			hdr = 1 + nb;
		}
		if ((int32_t)len < 0 || avail - hdr < len)
			return make_uint2(kTerminal, 0);
		return make_uint2(p + hdr + len, len);
	}
	const uint32_t hdr = kind == 1 ? 2u : (kind == 2 ? 3u : 5u);
	if (avail < hdr)
		return make_uint2(kTerminal, 0);
	return make_uint2(p + hdr, kind == 1 ? ((lf & 7u) + 4u) : (lf + 1u));
}

// stage chunk c (+ 8 bytes of lookahead) and fill J[q] = tag_step(q)
__device__ __forceinline__ void stage_and_parse(const uint8_t *in, uint32_t n, uint32_t start, uint32_t clen, uint8_t *sm_in,
						uint2 *J)
{
	const uint32_t want = min(clen + 8u, n - start);
	for (uint32_t i = threadIdx.x; i < want; i += kSThreads)
		sm_in[i] = in[start + i];
	for (uint32_t i = want + threadIdx.x; i < kChunk + 8; i += kSThreads)
		sm_in[i] = 0;
	__syncthreads();
	for (uint32_t q = threadIdx.x; q < clen; q += kSThreads)
		J[q] = tag_step(sm_in, q, start + q, n);
	__syncthreads();
}

// one synchronous doubling round over J (every position jumps twice as far, unless it has left the chunk)
__device__ __forceinline__ bool double_round(uint2 *J, uint32_t start, uint32_t clen)
{
	uint2 nv[kPer];
	bool changed = false;
#pragma unroll
	for (uint32_t k = 0; k < kPer; ++k) {
		const uint32_t q = threadIdx.x + k * kSThreads;
		nv[k] = make_uint2(kTerminal, 0);
		if (q < clen) {
			nv[k] = J[q];
			const uint32_t t = nv[k].x - start;  // inside the chunk iff t < clen (kTerminal and n are not)
			if (t < clen) {
				const uint2 b = J[t];
				nv[k] = make_uint2(b.x, sat_add(nv[k].y, b.y));
				changed = true;
			}
		}
	}
	__syncthreads();
#pragma unroll
	for (uint32_t k = 0; k < kPer; ++k) {
		const uint32_t q = threadIdx.x + k * kSThreads;
		if (q < clen)
			J[q] = nv[k];
	}
	return __syncthreads_or(changed) != 0;
}

// ---- 1a: exit table -------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kSThreads) exit_kernel(const uint8_t *__restrict__ in, uint32_t n, uint2 *__restrict__ exit_tab,
							 uint2 *__restrict__ entry, StreamCtl *ctl)
{
	__shared__ uint8_t sm_in[kChunk + 8];
	__shared__ uint2 J[kChunk];
	const uint32_t start = blockIdx.x * kChunk, clen = min(kChunk, n - start);
	if (blockIdx.x == 0 && threadIdx.x < 40)
		ctl->flags[threadIdx.x] = 0;
	if (blockIdx.x == 0 && threadIdx.x == 0)
		ctl->err_key = ~0ull;
	if (threadIdx.x == 0)
		entry[blockIdx.x] = make_uint2(kNone, 0);
	stage_and_parse(in, n, start, clen, sm_in, J);
	while (double_round(J, start, clen)) {
	}
	for (uint32_t q = threadIdx.x; q < clen; q += kSThreads)
		exit_tab[start + q] = J[q];
}

// ---- 1b: the real chain, chunk to chunk -------------------------------------------------------------------
__global__ void chain_kernel(const uint2 *__restrict__ exit_tab, uint32_t n, uint2 *__restrict__ entry, StreamCtl *ctl)
{
	if (threadIdx.x != 0 || blockIdx.x != 0)
		return;
	uint32_t cur = 0, out = 0;
	while (cur < n) {
		entry[cur / kChunk] = make_uint2(cur, out);
		const uint2 e = exit_tab[cur];
		out = sat_add(out, e.y);
		cur = e.x;
	}
	ctl->end_pos = cur;
	ctl->total = out;
}

__device__ __forceinline__ void report(StreamCtl *ctl, uint32_t pos, int code)
{
	atomicMin(&ctl->err_key, (unsigned long long)pos * 4ull + (code == S_DATA_MALFORMED ? 0ull : 1ull));
}

// ---- 2: tags of a chunk, literals, source indices ----------------------------------------------------------
__global__ void __launch_bounds__(kSThreads) expand_kernel(const uint8_t *__restrict__ in, uint32_t n, uint8_t *__restrict__ out,
							   uint32_t cap, const uint2 *__restrict__ entry, uint32_t *__restrict__ S,
							   StreamCtl *ctl)
{
	extern __shared__ __align__(16) uint8_t dsm[];	// kExpandSmem bytes
	uint2 *J0 = reinterpret_cast<uint2 *>(dsm);
	uint2 *J64 = J0 + kChunk;
	uint2 *tags = J64 + kChunk;
	uint2 *spine = tags + kTagSlots;
	uint8_t *sm_in = reinterpret_cast<uint8_t *>(spine + kSpineSlots);
	__shared__ uint32_t n_spine, n_tags;
	const uint2 ent = entry[blockIdx.x];
	if (ent.x == kNone)
		return;	 // a long literal jumps over this chunk
	const uint32_t start = blockIdx.x * kChunk, clen = min(kChunk, n - start);
	stage_and_parse(in, n, start, clen, sm_in, J0);
	for (uint32_t q = threadIdx.x; q < clen; q += kSThreads)
		J64[q] = J0[q];
	__syncthreads();
#pragma unroll 1
	for (int r = 0; r < 6; ++r)
		double_round(J64, start, clen);
	if (threadIdx.x == 0) {
		uint32_t cur = ent.x, o = ent.y, k = 0;
		while (cur - start < clen) {
			spine[k++] = make_uint2(cur, o);
			const uint2 j = J64[cur - start];
			o = sat_add(o, j.y);
			cur = j.x;
		}
		n_spine = k;
	}
	__syncthreads();
	if (threadIdx.x < n_spine) {
		uint32_t cur = spine[threadIdx.x].x, o = spine[threadIdx.x].y, k = 0;
		while (k < 64 && cur - start < clen) {
			tags[threadIdx.x * 64 + k++] = make_uint2(cur, o);
			const uint2 j = J0[cur - start];
			o = sat_add(o, j.y);
			cur = j.x;
		}
		if (threadIdx.x == n_spine - 1)
			n_tags = threadIdx.x * 64 + k;
	}
	__syncthreads();

	// ---- run the tags: one warp per tag ----
	const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
	for (uint32_t t = warp; t < n_tags; t += kSThreads / 32) {
		const uint32_t p = tags[t].x, o = tags[t].y, q = p - start;
		const uint32_t tag = sm_in[q], kind = tag & 3u, lf = tag >> 2, avail = n - p;
		const uint32_t room = o <= cap ? cap - o : 0u;
		if (kind == 0) {
			uint32_t len = lf + 1, hdr = 1;
			if (lf >= 60) {
				const uint32_t nb = lf - 59;
				if (avail - 1 < nb) {  // length bytes cut off (reference: UB)
					if (lane == 0)
						report(ctl, p, S_DATA_MALFORMED);
					continue;
				}
				uint32_t v = 0;
				for (uint32_t b = 0; b < nb; ++b)
					v |= (uint32_t)sm_in[q + 1 + b] << (8 * b);
				len = v + 1;
				hdr = 1 + nb;
			}
			// input shortage (a length of 2^31 or more passes the reference's signed test and fails on space, :374)
			const bool bad = (int32_t)len >= 0 ? (avail - hdr < len) : (room >= len);
			if (bad || room < len) {
				if (lane == 0)
					report(ctl, p, bad ? S_DATA_MALFORMED : S_OUTPUT_OVERRUN);
				continue;
			}
			const uint8_t *src = in + p + hdr;
			for (uint32_t i = lane; i < len; i += 32) {
				out[o + i] = src[i];
				S[o + i] = o + i;
			}
		} else {
			const uint32_t hdr = kind == 1 ? 2u : (kind == 2 ? 3u : 5u);
			if (avail < hdr) {  // offset bytes cut off (reference: UB)
				if (lane == 0)
					report(ctl, p, S_DATA_MALFORMED);
				continue;
			}
			uint32_t off = sm_in[q + 1], len = lf + 1;
			if (kind == 1) {
				len = (lf & 7u) + 4;
				off |= (tag >> 5) << 8;
			} else {
				off |= (uint32_t)sm_in[q + 2] << 8;
				if (kind == 3)
					off |= ((uint32_t)sm_in[q + 3] << 16) | ((uint32_t)sm_in[q + 4] << 24);
			}
			if (off - 1u >= o || room < len) {  // off == 0 or off > produced (:302), then space
				if (lane == 0)
					report(ctl, p, off - 1u >= o ? S_DATA_MALFORMED : S_OUTPUT_OVERRUN);
				continue;
			}
			for (uint32_t i = lane; i < len; i += 32)
				S[o + i] = o + i - off;
		}
	}
}

// ---- 3: resolve the back-references, gather, result --------------------------------------------------------
__global__ void __launch_bounds__(256) resolve_kernel(uint8_t *__restrict__ out, uint32_t cap, uint32_t *__restrict__ S, StreamCtl *ctl,
						      uint32_t *__restrict__ out_len, int32_t *__restrict__ status)
{
	cg::grid_group grid = cg::this_grid();
	const unsigned long long key = ctl->err_key;
	if (key != ~0ull) {  // uniform over the grid: no barrier has been passed yet
		if (blockIdx.x == 0 && threadIdx.x == 0) {
			*status = (key & 3ull) == 0 ? S_DATA_MALFORMED : S_OUTPUT_OVERRUN;
			*out_len = 0;
		}
		return;
	}
	const uint32_t total = ctl->total;  // <= cap: every tag passed its space check
	const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nthreads = gridDim.x * blockDim.x;
	// Each round at least doubles every unresolved jump, so a chain of depth d resolves in ceil(log2 d) rounds and
	// one more finds nothing to change.  The depth is below the output length <= cap < 2^32: at most 33 rounds, and
	// 40 is enough (an offset-1 run over 2^31 bytes takes 31).
	for (int round = 0; round < 40; ++round) {
		bool changed = false;
		for (uint32_t o = tid; o < total; o += nthreads) {
			const uint32_t s = S[o];
			if (s != o) {
				const uint32_t t = S[s];
				if (t != s) {
					S[o] = t;  // (a concurrent update of S[s] only makes the jump longer)
					changed = true;
				}
			}
		}
		if (__syncthreads_or(changed) && threadIdx.x == 0)
			atomicOr(&ctl->flags[round], 1u);
		grid.sync();
		if (*reinterpret_cast<volatile uint32_t *>(&ctl->flags[round]) == 0)
			break;
	}
	for (uint32_t o = tid; o < total; o += nthreads) {
		const uint32_t s = S[o];
		if (s != o)
			out[o] = out[s];  // S[s] == s: a literal byte, written by expand_kernel and never rewritten
	}
	if (tid == 0) {
		*status = S_OK;
		*out_len = total;
	}
	(void)cap;
}

}  // namespace csb

using namespace csb;

static size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

extern "C" size_t csb_stream_aux_bytes(uint32_t src_len, uint32_t cap, int which)
{
	if (which == 0) {
		const size_t chunks = ((size_t)src_len + kChunk - 1) / kChunk;
		return al256(sizeof(StreamCtl)) + al256((size_t)src_len * 8) + al256(chunks * 8) + 256;
	}
	return al256((size_t)cap * 4) + 256;
}

extern "C" int csb_launch_decompress_stream(const uint8_t *d_in, uint32_t src_len, uint8_t *d_out, uint32_t cap, uint32_t *d_out_len,
					    int32_t *d_status, void *d_aux_in, void *d_aux_out, csb_stream_t s)
{
	if (src_len == 0)
		return 1;  // nothing to parallelise: the caller's ordinary path returns (0, 0)
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e > 1 ? e : (int)cudaErrorUnknown;
	static int coop_ok[64], coop_ctas[64];
	int dev = 0;
	if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64)
		return 1;
	if (!coop_ok[dev]) {
		int coop = 0, per_sm = 0;
		cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
		if (!coop || cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, resolve_kernel, 256, 0) != cudaSuccess || per_sm < 1) {
			cudaGetLastError();
			coop_ok[dev] = -1;
		} else {
			coop_ctas[dev] = per_sm * di.sm_count;
			coop_ok[dev] = 1;
		}
	}
	if (coop_ok[dev] < 0)
		return 1;
	uint8_t *a = (uint8_t *)d_aux_in;
	StreamCtl *ctl = (StreamCtl *)a;
	uint2 *exit_tab = (uint2 *)(a + al256(sizeof(StreamCtl)));
	uint2 *entry = (uint2 *)(a + al256(sizeof(StreamCtl)) + al256((size_t)src_len * 8));
	uint32_t *S = (uint32_t *)d_aux_out;
	const uint32_t chunks = (src_len + kChunk - 1) / kChunk;

	exit_kernel<<<chunks, kSThreads, 0, s>>>(d_in, src_len, exit_tab, entry, ctl);
	count_launch();
	chain_kernel<<<1, 32, 0, s>>>(exit_tab, src_len, entry, ctl);
	count_launch();
	static bool attr_set[64];
	if (!attr_set[dev]) {
		if ((e = (int)cudaFuncSetAttribute(expand_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kExpandSmem)))
			return e > 1 ? e : (int)cudaErrorUnknown;
		attr_set[dev] = true;
	}
	expand_kernel<<<chunks, kSThreads, kExpandSmem, s>>>(d_in, src_len, d_out, cap, entry, S, ctl);
	count_launch();
	if ((e = (int)cudaGetLastError()))
		return e > 1 ? e : (int)cudaErrorUnknown;
	// grid of the cooperative kernel: enough threads for ~8 output bytes each, at most what is co-resident
	long want = ((long)cap / 8 + 255) / 256;
	if (want < 1)
		want = 1;
	if (want > coop_ctas[dev])
		want = coop_ctas[dev];
	void *args[] = {(void *)&d_out, (void *)&cap, (void *)&S, (void *)&ctl, (void *)&d_out_len, (void *)&d_status};
	e = (int)cudaLaunchCooperativeKernel((const void *)resolve_kernel, dim3((unsigned)want), dim3(256), args, 0, s);
	count_launch();
	if (e)
		return e > 1 ? e : (int)cudaErrorUnknown;
	return 0;
}
