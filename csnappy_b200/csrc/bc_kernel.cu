// bc_kernel.cu -- the block_compressor page container on device buffers (include/csnappy_batch.h csnappy_bc_compress,
// csnappy_bc_index, csnappy_bc_decompress_pages, csnappy_bc_decompress): the grid-wide index scan, the header writer,
// the gather of page requests and the kernels that reduce a read to its result.  Compression, the stored-page rule,
// the payload gather and decoding are the existing kernels (compress_kernel.cu, pack_kernel.cu, decompress_*.cu).
#include "device_common.cuh"
#include "kernels.h"

namespace csb {

constexpr int kBcThreads = 256;
constexpr int kBcItems = 16;
constexpr uint32_t kBcTile = kBcThreads * kBcItems;  // index entries per CTA of the scan
constexpr int kBcMidThreads = 1024;
// Payload sums saturate here.  An entry above max_clen counts as kSat, so "the payload runs past the container" is
// true from the first malformed entry on, whatever follows it: the end of the decodable prefix is one monotone test
// on the running sum, and saturating addition stays associative, so the sum can be scanned in any grouping.
constexpr uint64_t kSat = 1ull << 62;

__device__ __forceinline__ uint64_t sat_add(uint64_t a, uint64_t b)
{
	const uint64_t s = a + b;  // both <= 2^62: no wrap
	return s > kSat ? kSat : s;
}

// a little-endian u32 at any byte alignment: the aligned words that hold its bytes, funnel-shifted
__device__ __forceinline__ uint32_t ld_u32_any(const uint8_t *p)
{
	const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 3u);
	const uint32_t *w = reinterpret_cast<const uint32_t *>(p - sh);
	return sh ? __funnelshift_r(w[0], w[1], sh * 8) : w[0];
}

__device__ __forceinline__ uint64_t shfl_up_u64(uint64_t v, int d)
{
	return __shfl_up_sync(0xffffffffu, v, d);
}

// saturating inclusive scan over the warp
__device__ __forceinline__ uint64_t warp_scan_sat(uint64_t v, uint32_t lane)
{
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) {
		const uint64_t u = shfl_up_u64(v, d);
		if (lane >= (uint32_t)d)
			v = sat_add(v, u);
	}
	return v;
}

// Pass 1: the saturated payload sum of each tile, kept in index[tile * kBcTile] (the tile's own first output word,
// which only the same tile's pass 3 overwrites) so that the call needs no scratch memory.
__global__ void __launch_bounds__(kBcThreads) bc_index_reduce_kernel(const uint8_t *__restrict__ ent, uint32_t n,
								     uint32_t max_clen, uint64_t *__restrict__ index)
{
	__shared__ uint64_t wsum[kBcThreads / 32];
	const uint64_t base = (uint64_t)blockIdx.x * kBcTile;
	uint64_t s = 0;
#pragma unroll 4
	for (int k = 0; k < kBcItems; ++k) {
		const uint64_t i = base + (uint32_t)k * kBcThreads + threadIdx.x;
		if (i < n) {
			const uint32_t cl = ld_u32_any(ent + 4 * i);
			s = sat_add(s, cl > max_clen ? kSat : cl);
		}
	}
	const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
	s = warp_scan_sat(s, lane);
	if (lane == 31)
		wsum[w] = s;
	__syncthreads();
	if (threadIdx.x == 0) {
		uint64_t t = 0;
		for (int j = 0; j < kBcThreads / 32; ++j)
			t = sat_add(t, wsum[j]);
		index[base] = t;
	}
}

// Pass 2 (one CTA): exclusive saturating scan of the tile sums, in place.  One u64 per 4096 entries.
__global__ void __launch_bounds__(kBcMidThreads) bc_index_tiles_kernel(uint32_t n_tiles, uint64_t *__restrict__ index)
{
	__shared__ uint64_t part[kBcMidThreads];
	const uint32_t t = threadIdx.x;
	const uint32_t per = (n_tiles + kBcMidThreads - 1) / kBcMidThreads;
	const uint32_t lo = t * per < n_tiles ? t * per : n_tiles;
	const uint32_t hi = lo + per < n_tiles ? lo + per : n_tiles;
	uint64_t sum = 0;
	for (uint32_t i = lo; i < hi; ++i)
		sum = sat_add(sum, index[(uint64_t)i * kBcTile]);
	part[t] = sum;
	__syncthreads();
	for (uint32_t d = 1; d < kBcMidThreads; d <<= 1) {  // Hillis-Steele inclusive scan
		const uint64_t v = t >= d ? part[t - d] : 0;
		__syncthreads();
		part[t] = sat_add(part[t], v);
		__syncthreads();
	}
	uint64_t run = t ? part[t - 1] : 0;
	for (uint32_t i = lo; i < hi; ++i) {
		const uint64_t v = index[(uint64_t)i * kBcTile];
		index[(uint64_t)i * kBcTile] = run;
		run = sat_add(run, v);
	}
}

// Pass 3: per entry i, excl = saturated sum of the entries before it.  Entry i is in the decodable prefix when
// excl + value(i) <= room (room = container_length - first_off): index[i] = first_off + excl, else bad_off.
// len (optional) gets the entry for prefix pages and 0 behind; prefix (optional) gets the first page outside it.
__global__ void __launch_bounds__(kBcThreads) bc_index_kernel(const uint8_t *__restrict__ ent, uint32_t n, uint32_t max_clen,
							      uint64_t first_off, uint64_t room, uint64_t bad_off,
							      uint64_t *__restrict__ index, uint32_t *__restrict__ len,
							      uint32_t *__restrict__ prefix)
{
	__shared__ uint64_t wsum[kBcThreads / 32];
	const uint64_t base = (uint64_t)blockIdx.x * kBcTile;
	const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
	uint64_t carry = index[base];  // this tile's exclusive offset from pass 2
	__syncthreads();	       // read by every thread before the k = 0 step overwrites it
	for (int k = 0; k < kBcItems; ++k) {
		const uint64_t i = base + (uint32_t)k * kBcThreads + threadIdx.x;
		const uint32_t cl = i < n ? ld_u32_any(ent + 4 * i) : 0u;
		const uint64_t v = cl > max_clen ? kSat : cl;
		const uint64_t incl_w = warp_scan_sat(v, lane);
		uint64_t excl_w = shfl_up_u64(incl_w, 1);
		if (lane == 0)
			excl_w = 0;
		if (lane == 31)
			wsum[w] = incl_w;
		__syncthreads();
		uint64_t before = carry, total = carry;
		for (uint32_t j = 0; j < kBcThreads / 32; ++j) {
			if (j == w)
				before = total;
			total = sat_add(total, wsum[j]);
		}
		if (i < n) {
			const uint64_t excl = sat_add(before, excl_w), incl = sat_add(excl, v);
			const bool bad = incl > room;
			index[i] = bad ? bad_off : first_off + excl;
			if (len)
				len[i] = bad ? 0u : cl;
			if (prefix && bad && excl <= room)  // excl is the previous entry's incl: the one transition
				*prefix = (uint32_t)i;
		}
		carry = total;
		__syncthreads();  // wsum is rewritten by the next step
	}
}

// [u32 nr][u32 clen[nr]] at any alignment, and the container length (payload end of the last page)
__global__ void __launch_bounds__(256) bc_header_kernel(const uint32_t *__restrict__ clen, uint32_t n,
							const uint64_t *__restrict__ index, uint8_t *__restrict__ cont,
							uint64_t *__restrict__ cont_length)
{
	const bool aligned = (reinterpret_cast<uintptr_t>(cont) & 3u) == 0;
	for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += (uint64_t)gridDim.x * blockDim.x) {
		const uint32_t v = i ? clen[i - 1] : n;
		uint8_t *p = cont + 4 * i;
		if (aligned) {
			*reinterpret_cast<uint32_t *>(p) = v;
		} else {
			p[0] = (uint8_t)v;
			p[1] = (uint8_t)(v >> 8);
			p[2] = (uint8_t)(v >> 16);
			p[3] = (uint8_t)(v >> 24);
		}
	}
	if (blockIdx.x == 0 && threadIdx.x == 0)
		*cont_length = n ? index[n - 1] + clen[n - 1] : 4u;
}

// Request k -> decoder input (in_off[k], in_len[k]) and tag[k]: 0, or the status the request ends with without a
// decode (a page number >= nr, a page outside the decodable prefix, an index that does not fit this container).
// Tagged requests decode an empty block at the container start, which writes no output.
__global__ void __launch_bounds__(256) bc_request_kernel(const uint8_t *__restrict__ cont, uint64_t cont_length,
							 uint32_t max_clen, const uint64_t *__restrict__ index, uint32_t nr,
							 const uint32_t *__restrict__ pages, uint32_t n,
							 uint64_t *__restrict__ in_off, uint32_t *__restrict__ in_len,
							 int32_t *__restrict__ tag)
{
	for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
		const uint32_t p = pages[k];
		int32_t t = 0;
		uint64_t o = 0;
		uint32_t l = 0;
		if (p >= nr) {
			t = -101;  // CSNAPPY_E_BAD_ARG
		} else {
			o = index[p];
			if (o != ~0ull)
				l = ld_u32_any(cont + 4 + 4 * (uint64_t)p);
			if (o == ~0ull || l > max_clen || o > cont_length || l > cont_length - o)
				t = -5;	 // CSNAPPY_E_DATA_MALFORMED
		}
		in_off[k] = t ? 0 : o;
		in_len[k] = t ? 0u : l;
		tag[k] = t;
	}
}

__global__ void __launch_bounds__(256) bc_request_status_kernel(const int32_t *__restrict__ tag, uint32_t n,
								uint32_t *__restrict__ out_len, int32_t *__restrict__ status)
{
	for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
		const int32_t t = tag[k];
		if (t) {
			status[k] = t;
			out_len[k] = 0;
		}
	}
}

// Whole-container result, step 1: over the prefix pages, the sum of out_len and the smallest (page, status) key of a
// failed page.  Pages behind a failing page are decoded and counted, as in the host reader.
__global__ void __launch_bounds__(256) bc_finish_reduce_kernel(const uint32_t *__restrict__ out_len,
							       const int32_t *__restrict__ status, uint32_t nr,
							       struct csb_bc_result *r)
{
	const uint32_t n = r->prefix < nr ? r->prefix : nr;
	unsigned long long sum = 0, key = ~0ull;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const int32_t st = status[i];
		if (st == 0)
			sum += out_len[i];
		else if (key == ~0ull)  // i only grows within a thread: its first failure is its smallest
			key = ((unsigned long long)i << 32) | (uint32_t)st;
	}
#pragma unroll
	for (int d = 16; d; d >>= 1) {
		sum += __shfl_down_sync(0xffffffffu, sum, d);
		const unsigned long long o = __shfl_down_sync(0xffffffffu, key, d);
		key = o < key ? o : key;
	}
	if ((threadIdx.x & 31u) == 0) {
		if (sum)
			atomicAdd(reinterpret_cast<unsigned long long *>(&r->sum), sum);
		if (key != ~0ull)
			atomicMin(reinterpret_cast<unsigned long long *>(&r->key), key);
	}
}

// step 2, one thread: the index error at the prefix end competes with the decode failures; the smallest page wins
__global__ void bc_finish_kernel(uint32_t nr, int32_t hdr_rc, const struct csb_bc_result *__restrict__ r,
				 uint64_t *__restrict__ out_length, int32_t *__restrict__ status, uint32_t *__restrict__ failed_page)
{
	if (hdr_rc || nr == 0) {
		*status = hdr_rc;
		*out_length = 0;
		return;
	}
	unsigned long long key = r->key;
	if (r->prefix < nr) {
		const unsigned long long k = ((unsigned long long)r->prefix << 32) | (uint32_t)-5;
		key = k < key ? k : key;
	}
	*out_length = r->sum;
	if (key == ~0ull) {
		*status = 0;
	} else {
		*status = (int32_t)(uint32_t)key;
		if (failed_page)
			*failed_page = (uint32_t)(key >> 32);
	}
}

static long grid_for(uint64_t units, long per_cta, long cap)
{
	long ctas = (long)((units + per_cta - 1) / per_cta);
	if (ctas < 1)
		ctas = 1;
	return ctas > cap ? cap : ctas;
}

}  // namespace csb

using namespace csb;

extern "C" int csb_launch_bc_index(const uint8_t *ent, uint32_t n, uint32_t max_clen, uint64_t first_off, uint64_t room,
				   uint64_t bad_off, uint64_t *index, uint32_t *len, uint32_t *prefix, csb_stream_t s)
{
	if (n == 0)
		return 0;
	const uint32_t tiles = (uint32_t)(((uint64_t)n + kBcTile - 1) / kBcTile);
	if (room > kSat - 1)
		room = kSat - 1;
	bc_index_reduce_kernel<<<tiles, kBcThreads, 0, s>>>(ent, n, max_clen, index);
	count_launch();
	int e = (int)cudaGetLastError();
	if (e)
		return e;
	bc_index_tiles_kernel<<<1, kBcMidThreads, 0, s>>>(tiles, index);
	count_launch();
	if ((e = (int)cudaGetLastError()))
		return e;
	bc_index_kernel<<<tiles, kBcThreads, 0, s>>>(ent, n, max_clen, first_off, room, bad_off, index, len, prefix);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_bc_header(const uint32_t *clen, uint32_t n, const uint64_t *index, uint8_t *cont,
				    uint64_t *cont_length, csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	bc_header_kernel<<<(int)grid_for((uint64_t)n + 1, 256, (long)di.sm_count * 8), 256, 0, s>>>(clen, n, index, cont,
													    cont_length);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_bc_requests(const uint8_t *cont, uint64_t cont_length, uint32_t max_clen, const uint64_t *index,
				      uint32_t nr, const uint32_t *pages, uint32_t n, uint64_t *in_off, uint32_t *in_len,
				      int32_t *tag, csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	bc_request_kernel<<<(int)grid_for(n, 256, (long)di.sm_count * 8), 256, 0, s>>>(cont, cont_length, max_clen, index, nr,
											    pages, n, in_off, in_len, tag);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_bc_request_status(const int32_t *tag, uint32_t n, uint32_t *out_len, int32_t *status,
					    csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	bc_request_status_kernel<<<(int)grid_for(n, 256, (long)di.sm_count * 8), 256, 0, s>>>(tag, n, out_len, status);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_bc_finish(const uint32_t *out_len, const int32_t *status_pages, uint32_t nr, int32_t hdr_rc,
				    struct csb_bc_result *r, uint64_t *out_length, int32_t *status, uint32_t *failed_page,
				    csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	if (!hdr_rc && nr) {
		bc_finish_reduce_kernel<<<(int)grid_for(nr, 256 * 4, (long)di.sm_count * 8), 256, 0, s>>>(out_len, status_pages, nr,
													  r);
		count_launch();
		if ((e = (int)cudaGetLastError()))
			return e;
	}
	bc_finish_kernel<<<1, 1, 0, s>>>(nr, hdr_rc, r, out_length, status, failed_page);
	count_launch();
	return (int)cudaGetLastError();
}
