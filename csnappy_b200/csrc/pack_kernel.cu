// pack_kernel.cu -- exclusive scan of per-block compressed sizes and gather of the strided
// output slots into one contiguous payload.  Device-side equivalent of the running
// `written += p - compressed` of csnappy_compress (/root/reference/csnappy_compress.c:647-653)
// and of block_compressor's size index (block_compressor.c:298-335).  Also hosts the small
// per-device bookkeeping shared by all launchers.
#include <atomic>
#include <mutex>

#include "device_common.cuh"
#include "kernels.h"

namespace csb {

static std::atomic<uint64_t> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int device_info(DeviceInfo *out)
{
	static std::mutex mu;
	static DeviceInfo cache[64];
	static bool have[64];
	int dev = 0;
	cudaError_t e = cudaGetDevice(&dev);
	if (e != cudaSuccess)
		return (int)e;
	std::lock_guard<std::mutex> lk(mu);
	if (dev < 0 || dev >= 64)
		return (int)cudaErrorInvalidDevice;
	if (!have[dev]) {
		DeviceInfo di;
		if ((e = cudaDeviceGetAttribute(&di.sm_count, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess)
			return (int)e;
		if ((e = cudaDeviceGetAttribute(&di.smem_per_block_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess)
			return (int)e;
		if ((e = cudaDeviceGetAttribute(&di.smem_per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev)) != cudaSuccess)
			return (int)e;
		cache[dev] = di;
		have[dev] = true;
	}
	*out = cache[dev];
	return 0;
}

// Block-claim counters: a per-device ring of device words handed out round-robin, so a launch never
// allocates (a stream-ordered allocation per launch showed up as milliseconds of launch jitter).
// A slot is reused after kCounterSlots further launches on this device.  LIMIT: a kernel still running when
// 65536 later launches (on other streams of the same device) have been issued would share its counter with a
// new launch; the host-side launch rate (~5 us per launch) makes that a kernel running for > 0.3 s next to a
// stream issuing launches back to back -- the batched callers in csnappy_shim.c pass their own counters instead.
constexpr unsigned kCounterSlots = 65536;
uint32_t *next_counter()
{
	static std::mutex mu;
	static uint32_t *ring[64];
	static std::atomic<unsigned> cursor[64];
	int dev = 0;
	if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64)
		return nullptr;
	if (!ring[dev]) {
		std::lock_guard<std::mutex> lk(mu);
		if (!ring[dev]) {
			uint32_t *p = nullptr;
			if (cudaMalloc((void **)&p, kCounterSlots * sizeof(uint32_t)) != cudaSuccess)
				return nullptr;
			ring[dev] = p;
		}
	}
	return ring[dev] + (cursor[dev].fetch_add(1, std::memory_order_relaxed) % kCounterSlots);
}

constexpr int kScanThreads = 1024;

// Stored-block rule of block_compressor.c:316-318: a block whose compressed size is not smaller than
// its input is kept raw, and its recorded size is the input size.  page_len == 0 disables the rule.
__device__ __forceinline__ uint32_t block_in_len(uint32_t i, uint32_t page_len, uint64_t total_in)
{
	const uint64_t at = (uint64_t)i * page_len;
	const uint64_t left = total_in > at ? total_in - at : 0;
	return left < page_len ? (uint32_t)left : page_len;
}

__global__ void __launch_bounds__(256) clamp_kernel(const uint32_t *__restrict__ len, uint32_t n, uint32_t page_len,
						    uint64_t total_in, uint32_t *__restrict__ clen)
{
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const uint32_t ilen = block_in_len(i, page_len, total_in);
		clen[i] = len[i] >= ilen ? ilen : len[i];
	}
}

// single-CTA exclusive scan: off[i] = sum(len[0..i)), off[n] = total
__global__ void __launch_bounds__(kScanThreads) scan_kernel(const uint32_t *__restrict__ len, uint32_t n,
							    uint64_t *__restrict__ off)
{
	__shared__ uint64_t part[kScanThreads];
	const uint32_t t = threadIdx.x;
	const uint32_t per = (n + kScanThreads - 1) / kScanThreads;
	const uint32_t lo = t * per < n ? t * per : n;
	const uint32_t hi = lo + per < n ? lo + per : n;
	uint64_t sum = 0;
	for (uint32_t i = lo; i < hi; ++i)
		sum += len[i];
	part[t] = sum;
	__syncthreads();
	for (uint32_t d = 1; d < kScanThreads; d <<= 1) {  // Hillis-Steele inclusive scan
		const uint64_t v = t >= d ? part[t - d] : 0;
		__syncthreads();
		part[t] += v;
		__syncthreads();
	}
	uint64_t run = part[t] - sum;
	for (uint32_t i = lo; i < hi; ++i) {
		off[i] = run;
		run += len[i];
	}
	if (t == kScanThreads - 1)
		off[n] = part[t];
}

// one warp per block: packed[off[i] .. off[i]+len[i]) = slots[i*stride ..).  Destination words are
// written 4-byte aligned; the (arbitrarily aligned) source is realigned with a funnel shift.
// With `raw` set, block i comes from raw + i * page_len instead of its slot when its compressed
// size (slot_len[i]) is not smaller than its input (the stored-block rule above).
__global__ void __launch_bounds__(256) gather_kernel(const uint8_t *__restrict__ slots, uint64_t stride,
						     const uint32_t *__restrict__ len, uint32_t n,
						     uint8_t *__restrict__ packed, const uint64_t *__restrict__ off,
						     const uint8_t *__restrict__ raw, uint32_t page_len,
						     uint64_t total_in, const uint32_t *__restrict__ slot_len)
{
	const uint32_t lane = threadIdx.x & 31u;
	const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
	for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += warps) {
		const uint32_t m = len[i];
		const uint8_t *src = slots + (uint64_t)i * stride;
		if (raw && slot_len[i] >= block_in_len(i, page_len, total_in))
			src = raw + (uint64_t)i * page_len;
		uint8_t *dst = packed + off[i];
		uint32_t head = (uint32_t)((4u - (reinterpret_cast<uintptr_t>(dst) & 3u)) & 3u);
		if (head > m)
			head = m;
		if (lane < head)
			dst[lane] = src[lane];
		const uint32_t words = (m - head) >> 2;
		const uint8_t *s = src + head;
		const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(s) & 3u);
		const uint32_t *sw = reinterpret_cast<const uint32_t *>(s - sh);
		uint32_t *dw = reinterpret_cast<uint32_t *>(dst + head);
		if (sh == 0) {
			for (uint32_t w = lane; w < words; w += 32)
				dw[w] = sw[w];
		} else {
			// reads sw[w+1] only when it still overlaps [src, src+m): true because sh != 0
			for (uint32_t w = lane; w < words; w += 32)
				dw[w] = __funnelshift_r(sw[w], sw[w + 1], sh * 8);
		}
		const uint32_t tail = head + (words << 2);
		if (tail + lane < m)
			dst[tail + lane] = src[tail + lane];
	}
}

// Framing of csnappy_compress (/root/reference/csnappy_compress.c:621-656) for a BATCH of buffers: fragment f of
// buffer b = fbuf[f] lands behind that buffer's varint32 header and its earlier fragments.  One warp per fragment
// moves the bytes; the first fragment's warp (or, for an empty buffer, the buffer's own pseudo-fragment) also
// writes the header and the buffer's total length.
//   off[f]      exclusive scan of the fragment sizes over the whole batch
//   bfirst[b]   index of buffer b's first fragment (bfirst[n_buffers] = n_frag); an empty buffer owns none
__global__ void __launch_bounds__(256) frame_kernel(const uint8_t *__restrict__ slots, uint64_t stride,
						    const uint32_t *__restrict__ len, const uint64_t *__restrict__ off,
						    const uint32_t *__restrict__ fbuf, const uint32_t *__restrict__ bfirst,
						    const uint32_t *__restrict__ blen, uint32_t n_frag, uint32_t n_buffers,
						    uint8_t *__restrict__ out, uint64_t out_stride, uint32_t *__restrict__ out_len)
{
	const uint32_t lane = threadIdx.x & 31u;
	const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
	const uint32_t w0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	// headers and totals: one lane per buffer
	for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < n_buffers; b += gridDim.x * blockDim.x) {
		uint8_t *o = out + (uint64_t)b * out_stride;
		uint32_t v = blen[b], k = 0;
		while (v >= 128) {  // encode_varint32, csnappy_compress.c:46-73
			o[k++] = (uint8_t)(v | 0x80u);
			v >>= 7;
		}
		o[k++] = (uint8_t)v;
		out_len[b] = k + (uint32_t)(off[bfirst[b + 1]] - off[bfirst[b]]);
	}
	for (uint32_t f = w0; f < n_frag; f += warps) {
		const uint32_t b = fbuf[f], m = len[f];
		const uint32_t n = blen[b];
		const uint32_t hdr = n < (1u << 7) ? 1u : (n < (1u << 14) ? 2u : (n < (1u << 21) ? 3u : (n < (1u << 28) ? 4u : 5u)));
		const uint8_t *src = slots + (uint64_t)f * stride;
		uint8_t *dst = out + (uint64_t)b * out_stride + hdr + (off[f] - off[bfirst[b]]);
		uint32_t head = (uint32_t)((4u - (reinterpret_cast<uintptr_t>(dst) & 3u)) & 3u);
		if (head > m)
			head = m;
		if (lane < head)
			dst[lane] = src[lane];
		const uint32_t words = (m - head) >> 2;
		const uint8_t *s = src + head;
		const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(s) & 3u);
		const uint32_t *sw = reinterpret_cast<const uint32_t *>(s - sh);
		uint32_t *dw = reinterpret_cast<uint32_t *>(dst + head);
		if (sh == 0) {
			for (uint32_t w = lane; w < words; w += 32)
				dw[w] = sw[w];
		} else {
			for (uint32_t w = lane; w < words; w += 32)
				dw[w] = __funnelshift_r(sw[w], sw[w + 1], sh * 8);
		}
		const uint32_t tail = head + (words << 2);
		if (tail + lane < m)
			dst[tail + lane] = src[tail + lane];
	}
}

}  // namespace csb

using namespace csb;

extern "C" int csb_launch_frame(const uint8_t *slots, uint64_t slot_stride, const uint32_t *len, const uint64_t *off,
				const uint32_t *fbuf, const uint32_t *bfirst, const uint32_t *blen, uint32_t n_frag,
				uint32_t n_buffers, uint8_t *out, uint64_t out_stride, uint32_t *out_len, csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	if (n_buffers == 0)
		return 0;
	long units = n_frag > n_buffers / 32 ? (long)n_frag : (long)n_buffers / 32 + 1;
	long ctas = (units + 7) / 8;
	if (ctas > (long)di.sm_count * 8)
		ctas = (long)di.sm_count * 8;
	frame_kernel<<<(int)ctas, 256, 0, s>>>(slots, slot_stride, len, off, fbuf, bfirst, blen, n_frag, n_buffers, out, out_stride,
					       out_len);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" uint64_t csb_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

extern "C" int csb_launch_pack(const uint8_t *slots, uint64_t slot_stride, const uint32_t *len, uint32_t n_blocks,
			       uint8_t *packed, uint64_t *off, csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	scan_kernel<<<1, kScanThreads, 0, s>>>(len, n_blocks, off);
	count_launch();
	if ((e = (int)cudaGetLastError()))
		return e;
	if (packed && n_blocks) {
		long ctas = ((long)n_blocks + 7) / 8;
		if (ctas > (long)di.sm_count * 8)
			ctas = (long)di.sm_count * 8;
		gather_kernel<<<(int)ctas, 256, 0, s>>>(slots, slot_stride, len, n_blocks, packed, off, nullptr, 0, 0, nullptr);
		count_launch();
		e = (int)cudaGetLastError();
	}
	return e;
}

// Pack with the stored-block rule: clen[i] = min(len[i], input length of block i); off = exclusive
// scan of clen; packed gets the slot bytes, or the raw input block where compression did not help.
extern "C" int csb_launch_pack_stored(const uint8_t *slots, uint64_t slot_stride, const uint32_t *len, uint32_t n_blocks,
				      const uint8_t *in, uint32_t page_len, uint64_t total_in, uint32_t *clen,
				      uint8_t *packed, uint64_t *off, csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	if (n_blocks == 0) {
		scan_kernel<<<1, kScanThreads, 0, s>>>(len, 0, off);
		count_launch();
		return (int)cudaGetLastError();
	}
	long ctas = ((long)n_blocks + 255) / 256;
	if (ctas > (long)di.sm_count * 4)
		ctas = (long)di.sm_count * 4;
	clamp_kernel<<<(int)ctas, 256, 0, s>>>(len, n_blocks, page_len, total_in, clen);
	count_launch();
	if ((e = (int)cudaGetLastError()))
		return e;
	scan_kernel<<<1, kScanThreads, 0, s>>>(clen, n_blocks, off);
	count_launch();
	if ((e = (int)cudaGetLastError()))
		return e;
	ctas = ((long)n_blocks + 7) / 8;
	if (ctas > (long)di.sm_count * 8)
		ctas = (long)di.sm_count * 8;
	gather_kernel<<<(int)ctas, 256, 0, s>>>(slots, slot_stride, clen, n_blocks, packed, off, in, page_len, total_in, len);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_clamp(const uint32_t *len, uint32_t n_blocks, uint32_t page_len, uint64_t total_in, uint32_t *clen,
				csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	if (n_blocks == 0)
		return 0;
	long ctas = ((long)n_blocks + 255) / 256;
	if (ctas > (long)di.sm_count * 4)
		ctas = (long)di.sm_count * 4;
	clamp_kernel<<<(int)ctas, 256, 0, s>>>(len, n_blocks, page_len, total_in, clen);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_gather(const uint8_t *slots, uint64_t slot_stride, const uint32_t *len, uint32_t n_blocks,
				 uint8_t *packed, const uint64_t *off, const uint8_t *raw, uint32_t page_len, uint64_t total_in,
				 const uint32_t *slot_len, csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	if (n_blocks == 0)
		return 0;
	long ctas = ((long)n_blocks + 7) / 8;
	if (ctas > (long)di.sm_count * 8)
		ctas = (long)di.sm_count * 8;
	gather_kernel<<<(int)ctas, 256, 0, s>>>(slots, slot_stride, len, n_blocks, packed, off, raw, page_len, total_in, slot_len);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_scan(const uint32_t *len, uint32_t n_blocks, uint64_t *off, csb_stream_t s)
{
	scan_kernel<<<1, kScanThreads, 0, s>>>(len, n_blocks, off);
	count_launch();
	return (int)cudaGetLastError();
}
