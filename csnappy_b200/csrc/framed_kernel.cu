// framed_kernel.cu -- the Snappy framing format (include/csnappy_batch.h, csnappy_framed_*): masked CRC-32C of
// 64 KiB chunks, the chunk writer, the serial chunk walk of the reader and its verify step.
//
// Stream = [ff 06 00 00 "sNaPpY"] then chunks [u8 type][u24 LE length][body].  A data chunk's body is
// [u32 LE masked crc32c(uncompressed bytes)] followed by csnappy_compress(chunk) (type 0x00) or the bytes
// themselves (type 0x01).
//
// CRC-32C (Castagnoli, reflected 0x82F63B78, init ~0, final ~0), one warp per chunk of up to 65536 bytes:
//   * the chunk is cut into 32 slices of 2048 bytes aligned to its END: lane l covers [n - 2048 (32 - l),
//     n - 2048 (31 - l)) clipped to [0, n), so only the first active lane's slice is short;
//   * each lane runs slicing-by-8 (8 x 256-entry tables in shared memory) over its slice from register 0 --
//     the lane holding byte 0 starts from ~0 instead, which folds the init of the whole chunk in;
//   * lane l's register is advanced over the 31 - l slices behind it by ONE multiplication with x^(8*2048*(31-l))
//     mod P (a 32-entry table), and the lanes' registers are XOR-reduced.  CRC registers are linear in their
//     start value, so that XOR is the register after the whole chunk.
#include "device_common.cuh"
#include "kernels.h"

namespace csb {

constexpr uint32_t kCrcPoly = 0x82F63B78u;
constexpr uint32_t kSlice = 2048;  // bytes per lane: 32 * 2048 = the 65536-byte chunk of the format
constexpr uint64_t kNone = ~0ull;  // no failure key

// a * b mod P, reflected bit order (bit 31 = x^0): zlib's multmodp
__host__ __device__ constexpr uint32_t gf_mul(uint32_t a, uint32_t b)
{
	uint32_t p = 0;
	for (int i = 0; i < 32; ++i) {
		p ^= (a & 0x80000000u) ? b : 0u;
		a <<= 1;
		b = (b & 1u) ? (b >> 1) ^ kCrcPoly : b >> 1;
	}
	return p;
}

struct CrcTables {
	uint32_t t[8][256];  // t[k][i]: register after byte i followed by k zero bytes, from register 0
	uint32_t adv[32];    // adv[j] = x^(8 * 2048 * j) mod P: advance a register over j whole slices
};

__host__ __device__ constexpr CrcTables make_crc_tables()
{
	CrcTables c{};
	for (uint32_t i = 0; i < 256; ++i) {
		uint32_t r = i;
		for (int k = 0; k < 8; ++k)
			r = (r & 1u) ? (r >> 1) ^ kCrcPoly : r >> 1;
		c.t[0][i] = r;
	}
	for (int k = 1; k < 8; ++k)
		for (uint32_t i = 0; i < 256; ++i)
			c.t[k][i] = (c.t[k - 1][i] >> 8) ^ c.t[0][c.t[k - 1][i] & 0xffu];
	// x^(8*2048) by squaring x^1 (0x40000000) 14 times: x^(2^14) = x^16384 = x^(8*2048)
	uint32_t step = 0x40000000u;
	for (int i = 0; i < 14; ++i)
		step = gf_mul(step, step);
	uint32_t p = 0x80000000u;  // x^0
	for (int j = 0; j < 32; ++j) {
		c.adv[j] = p;
		p = gf_mul(p, step);
	}
	return c;
}

__device__ const CrcTables kCrcTables = make_crc_tables();

// the tables into shared memory; every thread of the CTA takes part, ends with a barrier
__device__ __forceinline__ void load_crc_tables(CrcTables &s)
{
	const uint32_t *g = &kCrcTables.t[0][0];
	uint32_t *d = &s.t[0][0];
	for (uint32_t i = threadIdx.x; i < sizeof(CrcTables) / 4; i += blockDim.x)
		d[i] = g[i];
	__syncthreads();
}

__device__ __forceinline__ uint32_t crc_mask(uint32_t crc) { return ((crc >> 15) | (crc << 17)) + 0xa282ead8u; }

// Masked CRC-32C of p[0, n), n <= 65536, any alignment; every lane of the warp calls it and gets the result.
__device__ __noinline__ uint32_t warp_crc32c(const CrcTables &T, const uint8_t *__restrict__ p, uint32_t n)
{
	const uint32_t lane = threadIdx.x & 31u;
	const int hi_i = (int)n - (int)(kSlice * (31u - lane));
	const uint32_t hi = hi_i > 0 ? (uint32_t)hi_i : 0u;
	const uint32_t lo = hi > kSlice ? hi - kSlice : 0u;
	const uint32_t first = n ? 31u - (n - 1) / kSlice : 31u;  // the lane holding byte 0 (lane 31 for n == 0)
	uint32_t r = lane == first ? 0xffffffffu : 0u;
	const uint8_t *q = p + lo;
	uint32_t m = hi - lo;
	uint32_t head = (uint32_t)((8u - (reinterpret_cast<uintptr_t>(q) & 7u)) & 7u);
	if (head > m)
		head = m;
	for (uint32_t i = 0; i < head; ++i)
		r = T.t[0][(r ^ q[i]) & 0xffu] ^ (r >> 8);
	q += head;
	m -= head;
	const uint2 *w = reinterpret_cast<const uint2 *>(q);
	const uint32_t words = m >> 3;
#pragma unroll 4
	for (uint32_t k = 0; k < words; ++k) {
		const uint2 v = __ldg(w + k);
		const uint32_t a = v.x ^ r, b = v.y;
		r = T.t[7][a & 0xffu] ^ T.t[6][(a >> 8) & 0xffu] ^ T.t[5][(a >> 16) & 0xffu] ^ T.t[4][a >> 24] ^
		    T.t[3][b & 0xffu] ^ T.t[2][(b >> 8) & 0xffu] ^ T.t[1][(b >> 16) & 0xffu] ^ T.t[0][b >> 24];
	}
	q += (size_t)words << 3;
	for (uint32_t i = 0; i < (m & 7u); ++i)
		r = T.t[0][(r ^ q[i]) & 0xffu] ^ (r >> 8);
	r = gf_mul(T.adv[31u - lane], r);
#pragma unroll
	for (int o = 16; o; o >>= 1)
		r ^= __shfl_xor_sync(0xffffffffu, r, o);
	return crc_mask(~r);
}

// dst[0, m) = src[0, m) with the whole warp: destination words 4-byte aligned, the source realigned with a funnel
// shift (gather_kernel, pack_kernel.cu).  Reads no aligned word that holds none of src[0, m).
__device__ __forceinline__ void warp_copy(uint8_t *__restrict__ dst, const uint8_t *__restrict__ src, uint32_t m)
{
	const uint32_t lane = threadIdx.x & 31u;
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

__device__ __forceinline__ uint32_t varint_len(uint32_t n)
{
	return n < (1u << 7) ? 1u : (n < (1u << 14) ? 2u : (n < (1u << 21) ? 3u : (n < (1u << 28) ? 4u : 5u)));
}

__device__ __forceinline__ uint32_t chunk_len(uint64_t n, uint32_t k)
{
	const uint64_t left = n - (uint64_t)k * CSB_FRAMED_CHUNK;
	return left < CSB_FRAMED_CHUNK ? (uint32_t)left : CSB_FRAMED_CHUNK;
}

// ---- writer --------------------------------------------------------------------------------------------------
// One warp per chunk: masked CRC of chunk k -> crc[k].  With flen (the compressed sizes of the input's 32 KiB
// fragments) also the record size of the chunk: 8 + the compressed payload (varint + fragments 2k, 2k+1) when that is
// smaller than n - n/8, else 8 + n.
__global__ void __launch_bounds__(256) framed_crc_kernel(const uint8_t *__restrict__ in, uint64_t n, uint32_t n_chunks,
							 uint32_t *__restrict__ crc, const uint32_t *__restrict__ flen,
							 uint32_t n_frag, uint32_t *__restrict__ rec)
{
	__shared__ CrcTables T;
	load_crc_tables(T);
	const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
	for (uint32_t k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < n_chunks; k += warps) {
		const uint32_t m = chunk_len(n, k);
		const uint32_t c = warp_crc32c(T, in + (uint64_t)k * CSB_FRAMED_CHUNK, m);
		if ((threadIdx.x & 31u) == 0) {
			crc[k] = c;
			if (flen) {
				const uint32_t f1 = 2 * k + 1 < n_frag ? flen[2 * k + 1] : 0u;
				const uint32_t clen = varint_len(m) + flen[2 * k] + f1;
				rec[k] = 8u + (clen < m - m / 8 ? clen : m);
			}
		}
	}
}

// One warp per chunk: header, CRC and payload of chunk k at out + 10 + off[k].  Block 0 also writes the stream
// identifier and *out_length.
__global__ void __launch_bounds__(256) framed_write_kernel(const uint8_t *__restrict__ in, uint64_t n, uint32_t n_chunks,
							   const uint8_t *__restrict__ slots, uint64_t slot_stride,
							   const uint32_t *__restrict__ flen, uint32_t n_frag,
							   const uint32_t *__restrict__ crc, const uint32_t *__restrict__ rec,
							   const uint64_t *__restrict__ off, uint8_t *__restrict__ out,
							   uint64_t *__restrict__ out_length)
{
	const uint32_t lane = threadIdx.x & 31u;
	if (blockIdx.x == 0 && threadIdx.x < 10) {
		// ff 06 00 00 73 4e 61 50 70 59: type 0xff, length 6, "sNaPpY"
		const uint32_t t = threadIdx.x;
		out[t] = (uint8_t)(t < 8 ? 0x50614e73000006ffull >> (8 * t) : 0x5970u >> (8 * (t - 8)));
		if (threadIdx.x == 0)
			*out_length = 10u + off[n_chunks];
	}
	const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
	for (uint32_t k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < n_chunks; k += warps) {
		const uint32_t m = chunk_len(n, k);
		const uint32_t body = rec[k] - 4u;
		const bool comp = rec[k] != 8u + m;  // a stored record is 8 + m bytes, a compressed one fewer
		uint8_t *dst = out + 10u + off[k];
		const uint32_t c = crc[k];
		if (lane < 8) {
			const uint32_t hdr = lane < 4 ? ((comp ? 0x00u : 0x01u) | (body << 8)) : c;
			dst[lane] = (uint8_t)(hdr >> (8 * (lane & 3u)));
		}
		if (!comp) {
			warp_copy(dst + 8, in + (uint64_t)k * CSB_FRAMED_CHUNK, m);
			continue;
		}
		const uint32_t hv = varint_len(m);
		if (lane < hv)
			dst[8 + lane] = (uint8_t)(((m >> (7 * lane)) & 0x7fu) | (lane + 1 < hv ? 0x80u : 0u));
		const uint32_t f0 = flen[2 * k];
		warp_copy(dst + 8 + hv, slots + (uint64_t)(2 * k) * slot_stride, f0);
		if (2 * k + 1 < n_frag)
			warp_copy(dst + 8 + hv + f0, slots + (uint64_t)(2 * k + 1) * slot_stride, flen[2 * k + 1]);
	}
}

// ---- reader ----------------------------------------------------------------------------------------------------
enum : uint32_t { kClassMalformed = 0, kClassOutput = 1, kClassChecksum = 2 };

__device__ __forceinline__ uint32_t get_u24(const uint8_t *p) { return p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16; }
__device__ __forceinline__ uint32_t get_u32(const uint8_t *p) { return get_u24(p) | (uint32_t)p[3] << 24; }

// The reader's rules for the chain of chunk headers of ONE stream src[0, len) with output capacity cap, shared by the
// single and the batched walk.  Calls rec(pos, out, olen, crc, plen, compressed) for every data chunk before the first
// failure the walk can detect itself (framing, identifier, varint, data length, capacity) and returns that failure's
// key position * 4 + class (kNone if there is none); *out_total = the output bytes of the recorded chunks.
template <class Rec>
__device__ __forceinline__ uint64_t walk_chunks(const uint8_t *__restrict__ src, uint64_t len, uint64_t cap,
						uint64_t *out_total, Rec &&rec)
{
	uint64_t pos = 0, out = 0, key = kNone;
	while (pos < len) {
		if (len - pos < 4) {
			key = pos * 4 + kClassMalformed;
			break;
		}
		const uint8_t *h = src + pos;
		const uint32_t type = h[0], blen = get_u24(h + 1);
		const uint64_t body = pos + 4;
		if (len - body < blen || (pos == 0 && type != 0xffu)) {
			key = pos * 4 + kClassMalformed;
			break;
		}
		if (type == 0xffu) {
			const uint8_t *b = h + 4;
			if (blen != 6 || b[0] != 's' || b[1] != 'N' || b[2] != 'a' || b[3] != 'P' || b[4] != 'p' || b[5] != 'Y') {
				key = pos * 4 + kClassMalformed;
				break;
			}
		} else if (type <= 0x01u) {
			if (blen < 4u + (type == 0u ? 1u : 0u)) {
				key = pos * 4 + kClassMalformed;
				break;
			}
			const uint32_t plen = blen - 4;
			uint32_t olen = plen;
			if (type == 0u) {  // varint32 of csnappy_get_uncompressed_length, then the format's 65536 limit
				const uint8_t *v = h + 8;
				uint32_t shift = 0, used = 0, value = 0;
				bool bad = false;
				for (;;) {
					if (shift >= 32 || used == plen) {
						bad = true;
						break;
					}
					const uint32_t c = v[used++];
					value |= (c & 0x7fu) << shift;
					if (c < 128)
						break;
					shift += 7;
				}
				if (bad || value > CSB_FRAMED_CHUNK) {
					key = pos * 4 + kClassMalformed;
					break;
				}
				olen = value;
			} else if (plen > CSB_FRAMED_CHUNK) {
				key = pos * 4 + kClassMalformed;
				break;
			}
			if (olen > cap - out) {
				key = pos * 4 + kClassOutput;
				break;
			}
			rec(pos, out, olen, get_u32(h + 4), plen, type == 0u);
			out += olen;
		} else if (type <= 0x7fu) {  // reserved unskippable
			key = pos * 4 + kClassMalformed;
			break;
		}
		// 0x80..0xfe: skippable / padding
		pos = body + blen;
	}
	*out_total = out;
	return key;
}

// The chain of chunk headers, one thread: the chunk table of csb_framed_table and the result words.
__global__ void framed_walk_kernel(const uint8_t *__restrict__ src, uint64_t len, uint64_t cap, struct csb_framed_table t)
{
	uint64_t out;
	uint32_t nd = 0, nc = 0;
	const uint64_t key = walk_chunks(src, len, cap, &out,
					 [&](uint64_t pos, uint64_t o, uint32_t olen, uint32_t crc, uint32_t plen, bool comp) {
						 t.pos[nd] = pos;
						 t.out_off[nd] = o;
						 t.out_len[nd] = olen;
						 t.crc[nd] = crc;
						 if (comp) {
							 t.cidx[nd] = nc;
							 t.c_pos[nc] = pos;
							 t.c_len[nc] = plen;
							 t.c_out_off[nc] = o;
							 ++nc;
						 } else {
							 t.cidx[nd] = 0xffffffffu;
						 }
						 ++nd;
					 });
	t.res->n_data = nd;
	t.res->n_comp = nc;
	t.res->walk_key = key;
	t.res->walk_out = out;
	t.res->verify_key = kNone;
}

// One warp per data chunk: a stored chunk is copied src -> dst; a compressed one must have decoded (status 0) to
// exactly its varint's length.  Then the masked CRC of the chunk's bytes is compared with the stored one.  The
// smallest failing key wins.
__global__ void __launch_bounds__(256) framed_verify_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
							    struct csb_framed_table t)
{
	__shared__ CrcTables T;
	load_crc_tables(T);
	const uint32_t nd = t.res->n_data;
	const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
	for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < nd; i += warps) {
		const uint64_t pos = t.pos[i];
		const uint32_t olen = t.out_len[i], j = t.cidx[i];
		uint8_t *o = dst + t.out_off[i];
		uint64_t key = kNone;
		uint32_t c;
		if (j != 0xffffffffu) {
			if (t.c_status[j] != 0 || t.c_produced[j] != olen) {
				key = pos * 4 + kClassMalformed;
				c = 0;
			} else {
				c = warp_crc32c(T, o, olen);
			}
		} else {
			const uint8_t *s = src + pos + 8;
			warp_copy(o, s, olen);
			c = warp_crc32c(T, s, olen);
		}
		if (key == kNone && c != t.crc[i])
			key = pos * 4 + kClassChecksum;
		if ((threadIdx.x & 31u) == 0 && key != kNone)
			atomicMin(reinterpret_cast<unsigned long long *>(&t.res->verify_key), (unsigned long long)key);
	}
}

// One thread: the call's result from the smallest failure key.
__global__ void framed_finish_kernel(struct csb_framed_table t, uint64_t *__restrict__ out_length,
				     int32_t *__restrict__ status, uint64_t *__restrict__ failed_offset)
{
	const csb_framed_result r = *t.res;
	const uint64_t key = r.walk_key < r.verify_key ? r.walk_key : r.verify_key;
	if (key == kNone) {
		*status = 0;
		*out_length = r.walk_out;
		return;
	}
	const uint64_t pos = key >> 2;
	const uint32_t cls = (uint32_t)(key & 3u);
	uint64_t produced = r.walk_out;  // a walk failure: every data chunk recorded lies before it
	if (key != r.walk_key) {
		uint32_t lo = 0, hi = r.n_data;  // the data chunk at `pos` (positions ascend)
		while (hi - lo > 1) {
			const uint32_t mid = (lo + hi) / 2;
			if (t.pos[mid] <= pos)
				lo = mid;
			else
				hi = mid;
		}
		produced = t.out_off[lo];
	}
	*status = cls == kClassMalformed ? -5 : (cls == kClassOutput ? -2 : -102);
	*out_length = produced;
	if (failed_offset)
		*failed_offset = pos;
}

// ---- many streams in one call (csnappy_framed_batch_*) --------------------------------------------------------------
// Writer.  One warp per chunk of every stream: masked CRC and record size, as framed_crc_kernel, with the chunk's input
// and fragments taken from the host-built chunk table.
__global__ void __launch_bounds__(256) framed_batch_crc_kernel(const uint8_t *__restrict__ in, uint32_t n_chunks,
							       struct csb_framed_batch_wtable t)
{
	__shared__ CrcTables T;
	load_crc_tables(T);
	const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
	for (uint32_t k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < n_chunks; k += warps) {
		const uint32_t m = t.c_len[k];
		const uint32_t c = warp_crc32c(T, in + t.c_in[k], m);
		if ((threadIdx.x & 31u) == 0) {
			const uint32_t f = t.c_frag[k];
			const uint32_t f1 = m > CSB_FRAGMENT_MAX ? t.flen[f + 1] : 0u;
			const uint32_t clen = varint_len(m) + t.flen[f] + f1;
			t.crc[k] = c;
			t.rec[k] = 8u + (clen < m - m / 8 ? clen : m);
		}
	}
}

// One warp per chunk: header, CRC and payload of chunk k at its stream's slot + 10 + (off[k] - off[the stream's first
// chunk]).  Then one thread per stream writes its identifier (empty streams too) and out_length.
__global__ void __launch_bounds__(256) framed_batch_write_kernel(const uint8_t *__restrict__ in, uint32_t n_chunks,
								 uint32_t n_streams, const uint8_t *__restrict__ slots,
								 uint64_t slot_stride, struct csb_framed_batch_wtable t,
								 uint8_t *__restrict__ out, uint64_t *__restrict__ out_length)
{
	const uint32_t lane = threadIdx.x & 31u;
	const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
	for (uint32_t k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < n_chunks; k += warps) {
		const uint32_t m = t.c_len[k], st = t.c_stream[k], rec = t.rec[k];
		const uint32_t body = rec - 4u;
		const bool comp = rec != 8u + m;  // a stored record is 8 + m bytes, a compressed one fewer
		uint8_t *dst = out + t.s_out[st] + 10u + (t.off[k] - t.off[t.s_first[st]]);
		const uint32_t c = t.crc[k];
		if (lane < 8) {
			const uint32_t hdr = lane < 4 ? ((comp ? 0x00u : 0x01u) | (body << 8)) : c;
			dst[lane] = (uint8_t)(hdr >> (8 * (lane & 3u)));
		}
		if (!comp) {
			warp_copy(dst + 8, in + t.c_in[k], m);
			continue;
		}
		const uint32_t hv = varint_len(m);
		if (lane < hv)
			dst[8 + lane] = (uint8_t)(((m >> (7 * lane)) & 0x7fu) | (lane + 1 < hv ? 0x80u : 0u));
		const uint32_t f = t.c_frag[k], f0 = t.flen[f];
		warp_copy(dst + 8 + hv, slots + (uint64_t)f * slot_stride, f0);
		if (m > CSB_FRAGMENT_MAX)
			warp_copy(dst + 8 + hv + f0, slots + (uint64_t)(f + 1) * slot_stride, t.flen[f + 1]);
	}
	const uint32_t threads = gridDim.x * blockDim.x;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_streams; i += threads) {
		uint8_t *o = out + t.s_out[i];
		// ff 06 00 00 73 4e 61 50 70 59: type 0xff, length 6, "sNaPpY"
		for (uint32_t b = 0; b < 10; ++b)
			o[b] = (uint8_t)(b < 8 ? 0x50614e73000006ffull >> (8 * b) : 0x5970u >> (8 * (b - 8)));
		out_length[i] = 10u + (t.off[t.s_first[i + 1]] - t.off[t.s_first[i]]);
	}
}

// Reader.  One thread per stream walks its chunk headers (walk_chunks) into its own region of the r_* tables.  With
// `length` set it is the decompressed_length walk instead: unbounded capacity, no table writes, the declared data
// length and 0 / -5 per stream.
__global__ void __launch_bounds__(128) framed_batch_walk_kernel(const uint8_t *__restrict__ src, uint32_t n_streams,
								struct csb_framed_batch_rtable t, uint64_t *__restrict__ length,
								int32_t *__restrict__ status)
{
	const uint32_t threads = gridDim.x * blockDim.x;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_streams; i += threads) {
		const uint8_t *s = src + t.s_src[i];
		uint64_t out;
		if (length) {
			const uint64_t key = walk_chunks(s, t.s_len[i], kNone, &out,
							 [](uint64_t, uint64_t, uint32_t, uint32_t, uint32_t, bool) {});
			length[i] = out;
			status[i] = key == kNone ? 0 : -5;
			continue;
		}
		const uint64_t reg = t.s_reg[i];
		uint32_t nd = 0, nc = 0;
		const uint64_t key = walk_chunks(s, t.s_len[i], t.s_cap[i], &out,
						 [&](uint64_t pos, uint64_t o, uint32_t olen, uint32_t crc, uint32_t plen, bool comp) {
							 const uint64_t r = reg + nd;
							 t.r_pos[r] = pos;
							 t.r_out[r] = o;
							 t.r_len[r] = olen;
							 t.r_crc[r] = crc;
							 t.r_plen[r] = plen;
							 t.r_cidx[r] = comp ? nc++ : 0xffffffffu;
							 ++nd;
						 });
		t.nd[i] = nd;
		t.nc[i] = nc;
		t.walk_key[i] = key;
		t.walk_out[i] = out;
		t.verify_key[i] = kNone;
	}
}

// One warp per stream: its region's records into the contiguous tables at the scanned bases, with the stream index and
// absolute source / destination offsets.  Thread 0 also stores the batch totals next to each other for the read-back.
__global__ void __launch_bounds__(256) framed_batch_compact_kernel(uint32_t n_streams, struct csb_framed_batch_rtable t)
{
	const uint32_t lane = threadIdx.x & 31u;
	if (blockIdx.x == 0 && threadIdx.x == 0) {
		t.totals[0] = t.d_base[n_streams];
		t.totals[1] = t.c_base[n_streams];
	}
	const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
	for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n_streams; i += warps) {
		const uint32_t nd = t.nd[i];
		const uint64_t reg = t.s_reg[i], db = t.d_base[i], cb = t.c_base[i], so = t.s_src[i], doff = t.s_dst[i];
		for (uint32_t j = lane; j < nd; j += 32) {
			const uint64_t r = reg + j, k = db + j;
			const uint64_t pos = so + t.r_pos[r], o = doff + t.r_out[r];
			const uint32_t ci = t.r_cidx[r];
			t.pos[k] = pos;
			t.out_off[k] = o;
			t.out_len[k] = t.r_len[r];
			t.crc[k] = t.r_crc[r];
			t.stream[k] = i;
			if (ci != 0xffffffffu) {
				const uint64_t c = cb + ci;
				t.cidx[k] = (uint32_t)c;
				t.c_pos[c] = pos;
				t.c_len[c] = t.r_plen[r];
				t.c_out_off[c] = o;
			} else {
				t.cidx[k] = 0xffffffffu;
			}
		}
	}
}

// One warp per data chunk of the batch: framed_verify_kernel's checks; the failure key, relative to the chunk's
// stream, goes to that stream's verify_key only.
__global__ void __launch_bounds__(256) framed_batch_verify_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
								  struct csb_framed_batch_rtable t)
{
	__shared__ CrcTables T;
	load_crc_tables(T);
	const uint64_t nd = t.totals[0];
	const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
	for (uint64_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < nd; i += warps) {
		const uint64_t pos = t.pos[i];
		const uint32_t olen = t.out_len[i], j = t.cidx[i], st = t.stream[i];
		uint8_t *o = dst + t.out_off[i];
		const uint64_t rel = pos - t.s_src[st];
		uint64_t key = kNone;
		uint32_t c;
		if (j != 0xffffffffu) {
			if (t.c_status[j] != 0 || t.c_produced[j] != olen) {
				key = rel * 4 + kClassMalformed;
				c = 0;
			} else {
				c = warp_crc32c(T, o, olen);
			}
		} else {
			const uint8_t *s = src + pos + 8;
			warp_copy(o, s, olen);
			c = warp_crc32c(T, s, olen);
		}
		if (key == kNone && c != t.crc[i])
			key = rel * 4 + kClassChecksum;
		if ((threadIdx.x & 31u) == 0 && key != kNone)
			atomicMin(reinterpret_cast<unsigned long long *>(&t.verify_key[st]), (unsigned long long)key);
	}
}

// One thread per stream: its result from the smaller of its walk and verify keys, as framed_finish_kernel, with the
// binary search confined to the stream's own range of the compacted table.
__global__ void __launch_bounds__(128) framed_batch_finish_kernel(uint32_t n_streams, struct csb_framed_batch_rtable t,
								  uint64_t *__restrict__ out_length,
								  int32_t *__restrict__ status,
								  uint64_t *__restrict__ failed_offset)
{
	const uint32_t threads = gridDim.x * blockDim.x;
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_streams; i += threads) {
		const uint64_t wk = t.walk_key[i], vk = t.verify_key[i];
		const uint64_t key = wk < vk ? wk : vk;
		if (key == kNone) {
			status[i] = 0;
			out_length[i] = t.walk_out[i];
			continue;
		}
		const uint64_t pos = key >> 2;
		const uint32_t cls = (uint32_t)(key & 3u);
		uint64_t produced = t.walk_out[i];  // a walk failure: every data chunk recorded lies before it
		if (key != wk) {
			const uint64_t at = t.s_src[i] + pos;
			uint64_t lo = t.d_base[i], hi = lo + t.nd[i];  // the data chunk at `pos` (positions ascend)
			while (hi - lo > 1) {
				const uint64_t mid = (lo + hi) / 2;
				if (t.pos[mid] <= at)
					lo = mid;
				else
					hi = mid;
			}
			produced = t.out_off[lo] - t.s_dst[i];
		}
		status[i] = cls == kClassMalformed ? -5 : (cls == kClassOutput ? -2 : -102);
		out_length[i] = produced;
		if (failed_offset)
			failed_offset[i] = pos;
	}
}

static int grid_for(uint32_t units, int per_cta, int sm_count)
{
	long ctas = ((long)units + per_cta - 1) / per_cta;
	if (ctas > (long)sm_count * 8)
		ctas = (long)sm_count * 8;
	return ctas < 1 ? 1 : (int)ctas;
}

}  // namespace csb

using namespace csb;

extern "C" int csb_launch_framed_crc(const uint8_t *in, uint64_t n, uint32_t *crc, const uint32_t *flen, uint32_t n_frag,
				     uint32_t *rec, csb_stream_t s)
{
	const uint64_t chunks = (n + CSB_FRAMED_CHUNK - 1) / CSB_FRAMED_CHUNK;
	if (chunks == 0)
		return 0;
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	framed_crc_kernel<<<grid_for((uint32_t)chunks, 8, di.sm_count), 256, 0, s>>>(in, n, (uint32_t)chunks, crc, flen, n_frag, rec);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_framed_write(const uint8_t *in, uint64_t n, const uint8_t *slots, uint64_t slot_stride,
				       const uint32_t *flen, uint32_t n_frag, const uint32_t *crc, const uint32_t *rec,
				       const uint64_t *off, uint8_t *out, uint64_t *out_length, csb_stream_t s)
{
	const uint32_t chunks = (uint32_t)((n + CSB_FRAMED_CHUNK - 1) / CSB_FRAMED_CHUNK);
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	framed_write_kernel<<<grid_for(chunks, 8, di.sm_count), 256, 0, s>>>(in, n, chunks, slots, slot_stride, flen, n_frag, crc,
									     rec, off, out, out_length);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_framed_walk(const uint8_t *src, uint64_t len, uint64_t cap, const struct csb_framed_table *t,
				      csb_stream_t s)
{
	framed_walk_kernel<<<1, 1, 0, s>>>(src, len, cap, *t);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_framed_verify(const uint8_t *src, uint8_t *dst, uint32_t n_data, const struct csb_framed_table *t,
					uint64_t *out_length, int32_t *status, uint64_t *failed_offset, csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	if (n_data) {
		framed_verify_kernel<<<grid_for(n_data, 8, di.sm_count), 256, 0, s>>>(src, dst, *t);
		count_launch();
		if ((e = (int)cudaGetLastError()))
			return e;
	}
	framed_finish_kernel<<<1, 1, 0, s>>>(*t, out_length, status, failed_offset);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_framed_batch_crc(const uint8_t *in, uint32_t n_chunks, const struct csb_framed_batch_wtable *t,
					   csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	framed_batch_crc_kernel<<<grid_for(n_chunks, 8, di.sm_count), 256, 0, s>>>(in, n_chunks, *t);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_framed_batch_write(const uint8_t *in, uint32_t n_chunks, uint32_t n_streams, const uint8_t *slots,
					     uint64_t slot_stride, const struct csb_framed_batch_wtable *t, uint8_t *out,
					     uint64_t *out_length, csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	const uint32_t units = n_chunks > n_streams / 32 ? n_chunks : n_streams / 32;
	framed_batch_write_kernel<<<grid_for(units, 8, di.sm_count), 256, 0, s>>>(in, n_chunks, n_streams, slots, slot_stride,
										    *t, out, out_length);
	count_launch();
	return (int)cudaGetLastError();
}

// one thread per stream: small CTAs, so that few streams still spread over the SMs
static int grid_per_stream(uint32_t n_streams, int sm_count)
{
	long ctas = ((long)n_streams + 127) / 128;
	if (ctas > (long)sm_count * 16)
		ctas = (long)sm_count * 16;
	return ctas < 1 ? 1 : (int)ctas;
}

extern "C" int csb_launch_framed_batch_walk(const uint8_t *src, uint32_t n_streams, const struct csb_framed_batch_rtable *t,
					    uint64_t *length, int32_t *status, csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	framed_batch_walk_kernel<<<grid_per_stream(n_streams, di.sm_count), 128, 0, s>>>(src, n_streams, *t, length, status);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_framed_batch_compact(uint32_t n_streams, const struct csb_framed_batch_rtable *t, csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	framed_batch_compact_kernel<<<grid_for(n_streams, 8, di.sm_count), 256, 0, s>>>(n_streams, *t);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_framed_batch_verify(const uint8_t *src, uint8_t *dst, uint32_t n_data, uint32_t n_streams,
					      const struct csb_framed_batch_rtable *t, uint64_t *out_length, int32_t *status,
					      uint64_t *failed_offset, csb_stream_t s)
{
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;
	if (n_data) {
		framed_batch_verify_kernel<<<grid_for(n_data, 8, di.sm_count), 256, 0, s>>>(src, dst, *t);
		count_launch();
		if ((e = (int)cudaGetLastError()))
			return e;
	}
	framed_batch_finish_kernel<<<grid_per_stream(n_streams, di.sm_count), 128, 0, s>>>(n_streams, *t, out_length, status,
											     failed_offset);
	count_launch();
	return (int)cudaGetLastError();
}
