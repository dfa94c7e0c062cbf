// decompress_kernel.cu -- batched Snappy raw-stream decoder for sm_100a.
//
// Per block: the semantics of csnappy_decompress_noheader
// (/root/reference/csnappy_decompress.c:319-387) -- first failing tag in stream order
// decides the code; literal: input shortage (-5) before space (-3); copy: offset validity
// (-5) before space (-3); end of input at a tag boundary is success -- or, with
// CSNAPPY_BATCH_WITH_HEADER, of csnappy_decompress (csnappy_decompress.c:394-411).
//
// A GROUP of G lanes (8, 16 or 32) owns one block; a persistent CTA per SM holds as many groups
// as shared memory allows (compressed block + output block: 24 x 4 KiB pages per SM).  Two paths:
//
//   staged     compressed block and output both fit the group's shared memory (4 KiB pages,
//              32 KiB fragments).  The block arrives with one bulk async copy (UBLKCP, mbarrier
//              completion).  The tag stream is decoded in BATCHES of G tags:
//                walk     the only inherently serial part -- tag k+1 starts where tag k ends -- is
//                         reduced to one byte load + one 256-entry table lookup per tag (the
//                         reference's char_table idea, csnappy_decompress.c:139-185), executed
//                         uniformly by the group; it also produces the output offset of every
//                         tag (the prefix sum of lengths) and the length-type errors;
//                decode   lane k decodes tag k completely (offset bytes, source, validity) --
//                         G tags in parallel;
//                execute  tags run in stream order, every lane moving bytes: literals and disjoint
//                         copies G bytes per step, overlapping copies (offset < length) as a
//                         pattern fill or in offset-sized rounds, all against shared memory.
//              The finished block leaves with one bulk async store (shared -> global).
//   global     blocks that do not fit shared memory (whole multi-chunk streams through the drop-in API), or
//              of which fewer than 8 would fit per SM (32 KiB fragments): same three phases, but the input is
//              read through L1 and the output lives in global memory, back-references through L2; no staging
//              area, so every warp of the CTA runs its own block and the L2 latency is hidden by their number.
#include <mutex>

#include "device_common.cuh"
#include "kernels.h"

namespace csb {

constexpr int E_OK = 0, E_HEADER_BAD = -1, E_OUTPUT_INSUF = -2, E_OUTPUT_OVERRUN = -3, E_DATA_MALFORMED = -5;
constexpr int kMaxThreadsD = 832;
constexpr int kMinStagedGroups = 8;  // fewer staged blocks per SM than this: use the global path instead


struct DecompressParams {
	csb_decompress_args a;
	uint32_t *counter;
	uint32_t in_area;   // staged input capacity (multiple of 16), 0 => streaming only
	uint32_t out_area;  // staged output capacity (multiple of 16)
	uint32_t group_smem;
	uint32_t groups;  // groups per CTA that own shared memory
};

// ---- global path: blocks that do not fit shared memory -----------------------------------------
// Same three phases as the staged path (walk / lane-per-tag decode / steps of G/8 tags), but the
// compressed block is read through L1 (ld.global.nc) and the output lives in global memory:
// back-references are read through L2 (ld.global.cg) after the __syncwarp that follows every step, which
// orders them behind the stores of earlier steps.  Needs no staging area, so a CTA runs as many groups
// as it has warps; the latency of L2 is hidden by the number of groups, not inside one.
// Batches are G/2 tags so that the G walk words + 8-byte descriptors of the staged layout (12 G bytes)
// hold 2 walk words + a 16-byte descriptor per tag.
template <int G>
__device__ __forceinline__ int decode_global(const Group<G> &g, const uint8_t *src, uint32_t ilen, uint8_t *dst,
					     uint32_t cap, uint32_t lut_a, uint32_t meta_a, uint32_t *produced_out)
{
	constexpr uint32_t GB = G / 2, Q = G / 8;
	const uint32_t pos_a = meta_a, out_a = meta_a + 4 * GB, desc_a = meta_a + 8 * GB;
	const uint32_t sub = g.lane & 7u, tq = g.lane >> 3;
	uint32_t pos = 0, produced = 0;
	for (;;) {
		// ---- walk ----
		uint32_t k = 0, e = 0;
		for (; k < GB; ++k) {
			if (pos >= ilen)
				break;
			e = lds_u32(lut_a + 4 * (uint32_t)__ldg(src + pos));
			sts_u32(pos_a + 4 * k, pos);
			sts_u32(out_a + 4 * k, produced);
			const uint32_t adv = e & 0xffffu, len = e >> 16;
			if (adv == 0xffffu || ilen - pos < adv || cap - produced < len)
				break;
			pos += adv;
			produced += len;
		}
		const uint32_t ntags = k;
		int werr = E_OK;
		bool stop = false, longlit = false;
		if (k < GB) {
			if (pos >= ilen)
				stop = true;  // end of input at a tag boundary
			else if ((e & 0xffffu) == 0xffffu)
				longlit = true;
			else if (ilen - pos < (e & 0xffffu))
				werr = E_DATA_MALFORMED;  // literal payload or copy offset bytes cut off by end of input
			else
				werr = E_OUTPUT_OVERRUN;  // (a copy still has its offset validated first)
		}
		g.sync();

		// ---- decode: lane k owns tag k ----
		// descriptor: x = source (output offset, or input position for a literal), y = destination output offset,
		//             z = len | literal << 8 | overlap << 9 | serial step << 10 | period << 16 | rounds << 24
		uint32_t dx = 0, dy = 0, dz = 0, mylen = 0, myo = 0, src_end = 0;
		bool bad = false, dep = false, cp = false;
		if (g.lane < ntags + (werr == E_OUTPUT_OVERRUN ? 1u : 0u)) {
			const uint32_t p = lds_u32(pos_a + 4 * g.lane), o = lds_u32(out_a + 4 * g.lane);
			const uint32_t tag = __ldg(src + p);
			const uint32_t kind = tag & 3u;
			uint32_t len = (tag >> 2) + 1;
			dy = o;
			if (kind == 0) {
				dx = p + 1;
				dz = len | (1u << 8);
			} else {
				uint32_t off = __ldg(src + p + 1);
				if (kind == 1) {
					len = ((tag >> 2) & 7u) + 4;
					off |= (tag >> 5) << 8;
				} else {
					off |= (uint32_t)__ldg(src + p + 2) << 8;
					if (kind == 3)
						off |= ((uint32_t)__ldg(src + p + 3) << 16) | ((uint32_t)__ldg(src + p + 4) << 24);
				}
				bad = off - 1u >= o;  // off == 0 or off > produced, csnappy_decompress.c:302
				dx = o - off;
				dz = len;
				cp = true;
				src_end = o - off + len;
				if (off < len) {
					dz |= (1u << 9) | (off << 16);
					dep = true;
				}
			}
			mylen = g.lane < ntags ? len : 0u;
			myo = o;
		}
		const unsigned badmask = g.ballot(bad);
		if (badmask || werr != E_OK)
			return badmask ? E_DATA_MALFORMED : werr;  // an invalid offset at or before the failing tag wins
		{
			const uint32_t first = g.lane & ~(Q - 1);
			const uint32_t o_first = g.bcast(myo, (int)first);
			dep = dep || (cp && g.lane < ntags && src_end > o_first);
			const unsigned dm = g.ballot(dep);
			uint32_t smax = mylen;
#pragma unroll
			for (uint32_t x = 1; x < Q; x <<= 1)
				smax = max(smax, __shfl_xor_sync(g.mask, smax, x, G));
			if (Q == 1 || ((dm >> first) & ((1u << Q) - 1u)))
				dz |= 1u << 10;
			dz |= ((smax + 7) >> 3) << 24;
		}
		if (g.lane < GB)
			sts_v4(desc_a + 16 * g.lane, dx, dy, dz, 0);
		g.sync();

		// ---- execute in stream order ----
		for (uint32_t t = 0; t < ntags; t += Q) {
			const uint4 d = lds_v4(desc_a + 16 * min(t + tq, GB - 1));
			if (!(d.z & (1u << 10))) {
				// independent step: 8 lanes per tag, all Q tags at once
				const uint32_t len = t + tq < ntags ? (d.z & 0xffu) : 0u, rounds = (d.z >> 24) & 0xfu;
				for (uint32_t j = 0; j < rounds; ++j) {
					const uint32_t i = sub + 8 * j;
					if (i < len)
						dst[d.y + i] = (d.z & (1u << 8)) ? __ldg(src + d.x + i) : __ldcg(dst + d.x + i);
				}
				g.sync();
				continue;
			}
			const uint32_t t_end = min(t + Q, ntags);
			for (uint32_t u = t; u < t_end; ++u) {
				const uint4 c = lds_v4(desc_a + 16 * u);
				const uint32_t len = c.z & 0xffu;
				uint8_t *to = dst + c.y;
				if (c.z & (1u << 8)) {
					for (uint32_t i = g.lane; i < len; i += G)
						to[i] = __ldg(src + c.x + i);
				} else {
					const uint8_t *from = dst + c.x;
					const uint32_t off = (c.z >> 16) & 0xffu;
					if (!(c.z & (1u << 9))) {
						for (uint32_t i = g.lane; i < len; i += G)
							to[i] = __ldcg(from + i);
					} else if (off >= (uint32_t)G) {
						for (uint32_t q = 0; q < len; q += G) {
							const uint32_t i = q + g.lane;
							if (i < len)
								to[i] = __ldcg(from + i);
							g.sync();
						}
					} else {
						for (uint32_t i = g.lane; i < len; i += G)
							to[i] = __ldcg(from + (i % off));
					}
				}
				g.sync();
			}
		}

		// ---- a long literal ends the batch and is copied by all lanes ----
		if (longlit) {
			const uint32_t tag = __ldg(src + pos++);
			const uint32_t nb = (tag >> 2) + 1 - 60;
			if (ilen - pos < nb)
				return E_DATA_MALFORMED;
			uint32_t v = 0;
			for (uint32_t b = 0; b < nb; ++b)
				v |= (uint32_t)__ldg(src + pos + b) << (8 * b);
			pos += nb;
			const uint32_t len = v + 1;  // 0xffffffff wraps to a zero-length literal (csnappy_decompress.c:370)
			if ((int32_t)len >= 0) {
				if (ilen - pos < len)
					return E_DATA_MALFORMED;
			} else if (cap - produced >= len) {
				return E_DATA_MALFORMED;
			}
			if (cap - produced < len)
				return E_OUTPUT_OVERRUN;
			uint32_t i = g.lane;
			for (; i + 3 * G < len; i += 4 * G) {
				const uint8_t b0 = __ldg(src + pos + i), b1 = __ldg(src + pos + i + G), b2 = __ldg(src + pos + i + 2 * G),
					      b3 = __ldg(src + pos + i + 3 * G);
				dst[produced + i] = b0;
				dst[produced + i + G] = b1;
				dst[produced + i + 2 * G] = b2;
				dst[produced + i + 3 * G] = b3;
			}
			for (; i < len; i += G)
				dst[produced + i] = __ldg(src + pos + i);
			pos += len;
			produced += len;
			g.sync();
		}
		if (stop)
			break;
	}
	*produced_out = produced;
	return E_OK;
}

// ---- staged path: one batch of up to G tags ---------------------------------------------------
// Returns 1 when the stream is finished (rc says how), 0 to continue with the next batch.
// gs = the group's shared memory; sin_off / sout_off = offsets of the staged input / output in it;
// lut_a / meta_a = shared addresses of the walk table and of the group's G walk words + G descriptors.
//
// GIN = true: the compressed block is NOT staged; tag bytes, offsets and literal payloads are read
// straight from global memory through L1 (ld.global.nc).  That halves the shared memory per block, so
// almost twice as many blocks are in flight per SM -- the decoder is bound by the latency of its
// serial chain, and more independent chains is what hides it.
template <bool GIN>
struct InBytes {
	uint32_t sin_a;	     // shared address of the staged block (GIN = false)
	const uint8_t *src;  // global address of the block (GIN = true)
	__device__ __forceinline__ uint32_t u8(uint32_t pos) const
	{
		return GIN ? (uint32_t)__ldg(src + pos) : lds_u8(sin_a + pos);
	}
};

// copy len input bytes at pos to shared address to_a with all lanes (long literals, stored blocks)
template <int G, bool GIN>
__device__ __forceinline__ void copy_in_to_shared(const Group<G> &g, const InBytes<GIN> &in, uint32_t pos, uint32_t to_a,
						  uint32_t len)
{
	if (GIN) {
		uint32_t i = g.lane;
		for (; i + 3 * G < len; i += 4 * G) {
			const uint32_t b0 = in.u8(pos + i), b1 = in.u8(pos + i + G), b2 = in.u8(pos + i + 2 * G),
				       b3 = in.u8(pos + i + 3 * G);
			sts_u8(to_a + i, b0);
			sts_u8(to_a + i + G, b1);
			sts_u8(to_a + i + 2 * G, b2);
			sts_u8(to_a + i + 3 * G, b3);
		}
		for (; i < len; i += G)
			sts_u8(to_a + i, in.u8(pos + i));
	} else {
		const uint32_t head = min((0u - to_a) & 3u, len);
		if (g.lane < head)
			sts_u8(to_a + g.lane, lds_u8(in.sin_a + pos + g.lane));
		const uint32_t words = (len - head) >> 2;
		for (uint32_t w = g.lane; w < words; w += G)
			sts_u32(to_a + head + 4 * w, lds32u_a(in.sin_a + pos + head + 4 * w));
		const uint32_t tail = head + (words << 2);
		if (tail + g.lane < len)
			sts_u8(to_a + tail + g.lane, lds_u8(in.sin_a + pos + tail + g.lane));
	}
}

template <int G, bool GIN>
__device__ __forceinline__ int decode_batch(const Group<G> &g, const InBytes<GIN> &in, uint32_t sout_a, uint32_t lut_a,
					    uint32_t meta_a, uint32_t &st_pos, uint32_t &st_produced, int &st_irem,
					    int &st_orem, int &rc)
{
	int irem = st_irem, orem = st_orem;
	if (irem == 0) {  // end of input at a tag boundary
		rc = E_OK;
		return 1;
	}
	const uint32_t last = st_pos + (uint32_t)irem - 1;  // GIN: never read past the block
	// ---- walk: positions and output offsets of up to G tags; ONE exit test per tag ----
	// lut[tag] = input bytes of the whole tag | output bytes << 16; a long literal has 0xffff input
	// bytes, so "input exhausted", "long literal", "payload cut off" and "no space" all show up as a
	// negative remainder and are told apart once, after the loop.  pos | produced << 16 advances with
	// one packed add.
	const uint32_t state0 = st_pos | (st_produced << 16);
	const int irem0 = irem;
	uint32_t state = state0, ra = st_pos;
	uint32_t k = 0, e = 0;
	// fast walk: per tag only the input remainder is tested; output space is tested for the batch as a whole
#pragma unroll 8
	for (; k < (uint32_t)G; ++k) {
		e = lds_u32(lut_a + 4 * in.u8(GIN ? min(ra, last) : ra));
		sts_u32(meta_a + 4 * k, state);
		const uint32_t adv = e & 0xffffu;
		const int x = irem - (int)adv;
		if (x < 0)
			break;
		state += e;
		ra += adv;
		irem = x;
	}
	if ((state >> 16) - st_produced <= (uint32_t)orem) {
		orem -= (int)((state >> 16) - st_produced);
	} else {
		// the batch does not fit the output: walk it again with the per-tag space test to find the tag that fails
		state = state0;
		ra = st_pos;
		irem = irem0;
		for (k = 0; k < (uint32_t)G; ++k) {
			e = lds_u32(lut_a + 4 * in.u8(GIN ? min(ra, last) : ra));
			sts_u32(meta_a + 4 * k, state);
			const uint32_t adv = e & 0xffffu;
			const int x = irem - (int)adv, y = orem - (int)(e >> 16);
			if ((x | y) < 0)
				break;
			state += e;
			ra += adv;
			irem = x;
			orem = y;
		}
	}
	uint32_t pos = state & 0xffffu, produced = state >> 16;
	const uint32_t ntags = k;  // complete tags of this batch
	int werr = E_OK;
	bool stop = false, longlit = false;
	if (k < (uint32_t)G) {
		if (irem == 0)
			stop = true;  // end of input at a tag boundary
		else if ((e & 0xffffu) == 0xffffu)
			longlit = true;
		else if (irem < (int)(e & 0xffffu))
			werr = E_DATA_MALFORMED;  // literal payload or copy offset bytes cut off by end of input
		else
			werr = E_OUTPUT_OVERRUN;  // (a copy still has its offset validated first, below)
	}
	g.sync();

	// ---- decode: lane k owns tag k (plus the tag that ran out of space: offset check only) ----
	// descriptor: x = source shared address | len << 20 | overlap << 28 | global literal << 29 | serial step << 30,
	//             y = destination shared address | period << 20 | copy rounds of the step << 26
	// Tags execute in STEPS of Q = G/8 consecutive tags, 8 lanes per tag, when no tag of the step reads
	// what the step writes; such dependent steps (and overlapping copies) run one tag at a time.
	constexpr uint32_t Q = G / 8;
	uint32_t d0 = 0, d1 = 0, mylen = 0, myo = 0;
	bool bad = false, dep = false, cp = false;
	uint32_t src_end = 0;
	if (g.lane < ntags + (werr == E_OUTPUT_OVERRUN ? 1u : 0u)) {
		const uint32_t mp = lds_u32(meta_a + 4 * g.lane);
		const uint32_t p = mp & 0xffffu, o = mp >> 16;
		const uint32_t tag = in.u8(p);
		const uint32_t kind = tag & 3u;
		uint32_t len = (tag >> 2) + 1;
		d1 = sout_a + o;
		if (kind == 0) {
			// literal: source is the input (a shared address, or -- bit 29 -- a position in the global block)
			d0 = (GIN ? (p + 1) | (1u << 29) : in.sin_a + p + 1) | (len << 20);
		} else {
			uint32_t off = in.u8(p + 1);
			if (kind == 1) {
				len = ((tag >> 2) & 7u) + 4;
				off |= (tag >> 5) << 8;
			} else {
				off |= in.u8(p + 2) << 8;
				if (kind == 3)
					off |= (in.u8(p + 3) << 16) | (in.u8(p + 4) << 24);
			}
			bad = off - 1u >= o;  // off == 0 or off > produced, csnappy_decompress.c:302
			d0 = ((d1 - off) & 0xfffffu) | (len << 20);
			cp = true;
			src_end = o - off + len;
			if (off < len) {  // overlapping: mode bit + the period
				d0 |= 1u << 28;
				d1 |= off << 20;
				dep = true;
			}
		}
		mylen = g.lane < ntags ? len : 0u;
		myo = o;
	}
	const unsigned badmask = g.ballot(bad);
	if (badmask || werr != E_OK) {
		// first failing tag in stream order: an invalid offset at or before the walk's failing tag wins
		rc = badmask ? E_DATA_MALFORMED : werr;
		return 1;
	}
	if (Q > 1) {
		// a copy whose source reaches into the output of its own step makes the step serial
		const uint32_t first = g.lane & ~(Q - 1);
		const uint32_t o_first = g.bcast(myo, (int)first);
		dep = dep || (cp && g.lane < ntags && src_end > o_first);
		const unsigned dm = g.ballot(dep);
		uint32_t smax = mylen;
#pragma unroll
		for (uint32_t x = 1; x < Q; x <<= 1)
			smax = max(smax, __shfl_xor_sync(g.mask, smax, x, G));
		if ((dm >> first) & ((1u << Q) - 1u))
			d0 |= 1u << 30;
		d1 |= ((smax + 7) >> 3) << 26;
	}
	const uint32_t desc_a = meta_a + 4 * G;
	sts_v2(desc_a + 8 * g.lane, d0, d1);
	g.sync();

	// ---- execute in stream order ----
	const uint32_t sub = g.lane & 7u, tq = g.lane >> 3;
	for (uint32_t t = 0; t < ntags; t += Q) {
		if (Q > 1) {
			const uint2 d = lds_v2(desc_a + 8 * (t + tq));
			if (!(d.x & (1u << 30))) {
				// independent step: 8 lanes per tag, all Q tags at once
				const uint32_t from = (d.x & 0xfffffu) + sub, to = (d.y & 0xfffffu) + sub;
				const uint32_t len = (d.x >> 20) & 0xffu, rounds = (d.y >> 26) & 0xfu;
				for (uint32_t j = 0; j < rounds; ++j)
					if (sub + 8 * j < len)
						sts_u8(to + 8 * j, (GIN && (d.x & (1u << 29))) ? in.u8(from + 8 * j) : lds_u8(from + 8 * j));
				g.sync();
				continue;
			}
		}
		const uint32_t t_end = min(t + Q, ntags);
		for (uint32_t u = t; u < t_end; ++u) {
			const uint2 d = lds_v2(desc_a + 8 * u);
			const uint32_t from = (d.x & 0xfffffu) + g.lane, to = (d.y & 0xfffffu) + g.lane;
			const uint32_t len = (d.x >> 20) & 0xffu;
			if (!(d.x & (3u << 28))) {
				// literal or disjoint copy (len <= 64): at most 64 / G predicated rounds, no loop
#pragma unroll
				for (uint32_t j = 0; j < 64u / G; ++j)
					if (g.lane + j * G < len)
						sts_u8(to + j * G, lds_u8(from + j * G));
			} else if (GIN && (d.x & (1u << 29))) {
				// literal from the global block
#pragma unroll
				for (uint32_t j = 0; j < 64u / G; ++j)
					if (g.lane + j * G < len)
						sts_u8(to + j * G, in.u8(from + j * G));
			} else {
				const uint32_t off = (d.y >> 20) & 0x3fu;
				if (off == 1) {
					const uint32_t v = lds_u8(from - g.lane);
					for (uint32_t i = g.lane; i < len; i += G)
						sts_u8(to + i - g.lane, v);
				} else if (off >= (uint32_t)G) {
					// a round of G bytes only reads what earlier rounds wrote
					for (uint32_t c = 0; c < len; c += G) {
						if (c + g.lane < len)
							sts_u8(to + c, lds_u8(from + c));
						g.sync();
					}
				} else {
					// short period: byte i repeats the pattern [o - off, o)
					for (uint32_t i = g.lane; i < len; i += G)
						sts_u8(to + i - g.lane, lds_u8(from - g.lane + i % off));
				}
			}
			g.sync();
		}
	}

	// ---- a long literal (61+ bytes, 1-4 length bytes) ends the batch and is copied by all lanes ----
	if (longlit) {
		const uint32_t ilen = pos + (uint32_t)irem;
		const uint32_t tag = in.u8(pos++);
		const uint32_t nb = (tag >> 2) + 1 - 60;
		if (ilen - pos < nb) {
			rc = E_DATA_MALFORMED;
			return 1;
		}
		uint32_t v = 0;
		for (uint32_t b = 0; b < nb; ++b)
			v |= in.u8(pos + b) << (8 * b);
		pos += nb;
		const uint32_t len = v + 1;  // 0xffffffff wraps to a zero-length literal (csnappy_decompress.c:370)
		// (a length of 2^31 or more passes the reference's signed input check and fails on space, :374)
		if ((int32_t)len >= 0 && ilen - pos < len) {
			rc = E_DATA_MALFORMED;
			return 1;
		}
		if ((uint32_t)orem < len) {
			rc = E_OUTPUT_OVERRUN;
			return 1;
		}
		copy_in_to_shared<G, GIN>(g, in, pos, sout_a + produced, len);
		pos += len;
		produced += len;
		irem = (int)(ilen - pos);
		orem -= (int)len;
		g.sync();
	}
	st_pos = pos;
	st_produced = produced;
	st_irem = irem;
	st_orem = orem;
	if (stop) {
		rc = E_OK;
		return 1;
	}
	return 0;
}

enum : int { DS_NEED = 0, DS_LOADING = 1, DS_RUN = 2 };

template <int G, bool GIN>
__global__ void __launch_bounds__(kMaxThreadsD, 1) decompress_kernel(const DecompressParams p)
{
	extern __shared__ __align__(128) uint8_t smem[];
	__shared__ uint32_t lut[256];
	// walk table (csnappy_decompress.c:139-185 restated): input bytes of the whole tag | output bytes << 16
	for (uint32_t t = threadIdx.x; t < 256; t += blockDim.x) {
		const uint32_t kind = t & 3u, l = (t >> 2) + 1;
		uint32_t e;
		if (kind == 0)
			e = l > 60 ? 0xffffu : ((1 + l) | (l << 16));
		else if (kind == 1)
			e = 2u | ((((t >> 2) & 7u) + 4) << 16);
		else
			e = (kind == 2 ? 3u : 5u) | (l << 16);
		lut[t] = e;
	}
	__syncthreads();

	const Group<G> g;
	const uint32_t gid = threadIdx.x / G;
	if (gid >= p.groups)
		return;	 // padding lanes of the last warp (no block-wide barriers below)
	const csb_decompress_args &a = p.a;
	uint8_t *gs = smem + (size_t)gid * p.group_smem;
	uint8_t *sout = gs + p.in_area;
	uint32_t *meta = reinterpret_cast<uint32_t *>(sout + p.out_area);  // G walk words + G descriptors
	const uint32_t bar = smem_u32(meta + 3 * G), meta_a = smem_u32(meta), lut_a = smem_u32(lut);
	const unsigned full = (G == 32) ? 0xffffffffu : ((1u << G) - 1u);

	if (g.lane == 0) {
		mbar_init(bar, 1);
		fence_mbar_init();
	}
	g.sync();

	int state = DS_NEED;
	uint32_t parity = 0, blk = 0;
	uint32_t st_pos = 0, st_produced = 0;  // input / output cursor of the staged block
	int st_irem = 0, st_orem = 0;	       // input bytes left, output capacity left
	InBytes<GIN> in;
	in.sin_a = smem_u32(gs);
	in.src = nullptr;
	const uint32_t sout_a = smem_u32(sout);
	bool raw = false;
	uint8_t *dst = nullptr;

	for (;;) {
		if (state == DS_NEED) {
			if (g.lane == 0)
				blk = atomicAdd(p.counter, 1u);
			blk = g.bcast(blk, 0);
			if (blk >= a.n_blocks)
				break;
			const uint8_t *src = a.in + (a.in_off ? a.in_off[blk] : (uint64_t)blk * a.in_stride);
			uint32_t ilen = a.in_len[blk];
			uint32_t cap = a.out_cap ? a.out_cap[blk] : a.uniform_cap;
			dst = a.out + (a.out_off ? a.out_off[blk] : (uint64_t)blk * a.out_stride);
			int rc = E_OK;
			if (a.flags & 2u) {  // varint32 length prefix, csnappy_decompress.c:45-71, 404-409
				uint32_t shift = 0, used = 0, value = 0;
				for (;;) {
					if (shift >= 32 || used == ilen) {
						rc = E_HEADER_BAD;
						break;
					}
					const uint32_t c = src[used++];
					value |= (c & 0x7fu) << shift;
					if (c < 128)
						break;
					shift += 7;
				}
				if (rc == E_OK) {
					if (value > cap)
						rc = E_OUTPUT_INSUF;
					cap = value;
					src += used;
					ilen -= used;
				}
			}
			if (rc == E_OK && !((GIN || ilen + 32 <= p.in_area) && cap <= p.out_area && ilen < 65535u)) {  // 0xffff is the walk's long-literal marker: a staged block is shorter
				uint32_t produced = 0;
				if ((a.flags & 4u) && ilen == cap) {  // stored block too large to stage: plain copy
					for (uint32_t i = g.lane; i < ilen; i += G)
						dst[i] = src[i];
					produced = ilen;
				} else {
					rc = decode_global<G>(g, src, ilen, dst, cap, lut_a, meta_a, &produced);
				}
				if (g.lane == 0) {
					a.status[blk] = rc;
					a.out_len[blk] = rc == E_OK ? produced : 0u;
				}
				continue;
			}
			if (rc != E_OK) {
				if (g.lane == 0) {
					a.status[blk] = rc;
					a.out_len[blk] = 0u;
				}
				continue;
			}
			// staged: the previous block's output store must have finished reading shared memory
			if (g.lane == 0)
				bulk_wait_read0();
			g.sync();
			st_pos = 0;
			st_produced = 0;
			st_irem = (int)ilen;
			st_orem = (int)cap;
			raw = (a.flags & 4u) && ilen == cap;  // stored block (block_compressor.c:378)
			if (GIN) {
				in.src = src;
				state = DS_RUN;
			} else {
				bool bulk;
				in.sin_a = smem_u32(gs) + stage_block<G>(g, gs, src, ilen, bar, &bulk);
				state = bulk ? DS_LOADING : DS_RUN;
			}
			g.sync();
		}
		if (state == DS_LOADING) {
			if (g.ballot(mbar_test(bar, parity)) != full)
				continue;
			parity ^= 1u;
			state = DS_RUN;
		}

		int rc = E_OK;
		if (raw) {
			// stored block: plain copy into the output area
			copy_in_to_shared<G, GIN>(g, in, 0, sout_a, (uint32_t)st_irem);
			st_produced = (uint32_t)st_irem;
			g.sync();
		} else if (!decode_batch<G, GIN>(g, in, sout_a, lut_a, meta_a, st_pos, st_produced, st_irem, st_orem, rc)) {
			continue;
		}

		// ---- block finished ----
		const uint32_t produced = st_produced;
		if (rc == E_OK) {
			if ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
				const uint32_t n16 = produced & ~15u;
				if (n16) {
					fence_proxy_async();  // this lane's generic writes to sout -> async proxy
					g.sync();
					if (g.lane == 0) {
						bulk_s2g(dst, smem_u32(sout), n16);
						bulk_commit();
					}
				}
				for (uint32_t i = n16 + g.lane; i < produced; i += G)
					dst[i] = sout[i];
			} else {
				for (uint32_t i = g.lane; i < produced; i += G)
					dst[i] = sout[i];
			}
		}
		if (g.lane == 0) {
			a.status[blk] = rc;
			a.out_len[blk] = rc == E_OK ? produced : 0u;
		}
		state = DS_NEED;
	}
	// outstanding bulk stores read shared memory: they must finish before the CTA's memory is released
	if (g.lane == 0)
		bulk_wait_read0();
}

}  // namespace csb

using namespace csb;

template <int G, bool GIN>
static int launch_decompress_gi(const DecompressParams &p, int threads, int ctas, size_t smem, cudaStream_t s)
{
	// set the kernel's attributes and launch as one step (see launch_compress_g)
	static std::mutex mu;
	std::lock_guard<std::mutex> lk(mu);
	cudaError_t e = cudaFuncSetAttribute(decompress_kernel<G, GIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	if (e != cudaSuccess)
		return (int)e;
	// leave the rest of the unified array to L1: the unstaged input is read through it
	e = cudaFuncSetAttribute(decompress_kernel<G, GIN>, cudaFuncAttributePreferredSharedMemoryCarveout,
				 (int)((smem + 2048) * 100 / (228 * 1024) + 1));
	if (e != cudaSuccess)
		return (int)e;
	decompress_kernel<G, GIN><<<ctas, threads, smem, s>>>(p);
	count_launch();
	return (int)cudaGetLastError();
}

template <int G>
static int launch_decompress_g(const DecompressParams &p, bool gin, int threads, int ctas, size_t smem, cudaStream_t s)
{
	return gin ? launch_decompress_gi<G, true>(p, threads, ctas, smem, s)
		   : launch_decompress_gi<G, false>(p, threads, ctas, smem, s);
}

extern "C" int csb_launch_decompress(const struct csb_decompress_args *a, csb_stream_t s)
{
	if (a->n_blocks == 0)
		return 0;
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;

	DecompressParams p;
	p.a = *a;
	const int G = a->lanes ? a->lanes : 32;
	// staging capacities: output from the (uniform) capacity or the stride, input from the hint,
	// the stride, or the format's worst case for that output size; both capped at fragment scale
	uint64_t out_cap = a->out_cap ? a->out_stride : a->uniform_cap;
	if (out_cap > CSB_FRAGMENT_MAX)
		out_cap = CSB_FRAGMENT_MAX;
	uint64_t in_cap = a->max_in_len;
	if (!in_cap) {
		in_cap = 32 + out_cap + out_cap / 6;
		if (!a->in_off && a->in_stride && a->in_stride < in_cap)
			in_cap = a->in_stride;
	}
	if (in_cap > 32 + CSB_FRAGMENT_MAX + CSB_FRAGMENT_MAX / 6)
		in_cap = 32 + CSB_FRAGMENT_MAX + CSB_FRAGMENT_MAX / 6;
	const bool gin = a->stage_input == 2;  // 2: read the compressed block through L1 instead of staging it (measured slower)
	p.in_area = gin ? 0u : (uint32_t)((in_cap + 15) & ~15ull) + 32;  // + staging shift (< 16) + slack for over-reads
	p.out_area = (uint32_t)((out_cap + 15) & ~15ull);
	const uint32_t meta_bytes = 12u * (uint32_t)G + 16u;  // walk words, descriptors, mbarrier
	p.group_smem = p.in_area + p.out_area + meta_bytes;

	const int ctas_per_sm = a->ctas_per_sm > 0 ? a->ctas_per_sm : 1;
	long budget = (long)di.smem_per_sm / ctas_per_sm - 1024 - 1024;  // 1024: the static walk table
	if (gin) {
		// keep part of the unified L1/shared array as L1 for the input stream
		const long cap_kb = a->smem_kb > 0 ? a->smem_kb : 164;
		if (budget > cap_kb * 1024 / ctas_per_sm)
			budget = cap_kb * 1024 / ctas_per_sm;
	}
	if (budget > di.smem_per_block_optin - 1024)
		budget = di.smem_per_block_optin - 1024;
	int groups = (int)(budget / p.group_smem);
	const int max_groups = kMaxThreadsD / G;
	if (groups > max_groups)
		groups = max_groups;
	const bool unstaged = (groups < kMinStagedGroups && a->stage_input != 1) || a->stage_input == 3 || groups < 1;
	// One lane per block (decompress_lane_kernel.cu) when there are enough blocks to fill the machine with lanes
	// (1280 per SM): measured crossovers on a B200 are ~24 Ki blocks against the warp-per-block global path
	// (32 KiB fragments: 116 vs 77 GB/s at 32 Ki, 300 vs 77 at 128 Ki) and ~150 Ki blocks against the staged path
	// (mixed 4 KiB pages: 408 vs 417 GB/s at 128 Ki, 538 vs 430 at 256 Ki).  Needs 16-byte aligned output slots.
	const bool lane_ok = !a->out_off && ((reinterpret_cast<uintptr_t>(a->out) | a->out_stride) & 15u) == 0;
	// stage_input 4 asks for it; slots it cannot write (the container reader's pages of any size, a caller's odd
	// stride) take the routing below instead of failing the call
	const uint32_t lane_min = (uint32_t)di.sm_count * (unstaged ? 160u : 1100u);
	if (lane_ok && (a->stage_input == 4 || (a->stage_input == 0 && a->n_blocks >= lane_min)))
		return csb_launch_decompress_lane(a, s);
	if (unstaged) {
		// too few blocks fit shared memory for their chains to hide each other: global path, one group per warp slot
		p.in_area = p.out_area = 0;
		p.group_smem = meta_bytes;
		groups = kMaxThreadsD / G;
	}
	long want = ((long)a->n_blocks + groups - 1) / groups;
	long ctas = (long)di.sm_count * ctas_per_sm;
	if (ctas > want) {
		ctas = want;
		if (a->n_blocks < (uint32_t)(di.sm_count * groups)) {
			ctas = a->n_blocks < (uint32_t)di.sm_count ? (long)a->n_blocks : (long)di.sm_count;
			groups = (int)(((long)a->n_blocks + ctas - 1) / ctas);
		}
	}
	p.groups = (uint32_t)groups;
	const int threads = (groups * G + 31) / 32 * 32;  // whole warps; surplus lanes exit at once
	const size_t smem = (size_t)groups * p.group_smem;

	uint32_t *counter = a->counter ? a->counter : next_counter();
	if (!counter)
		return (int)cudaErrorMemoryAllocation;
	cudaError_t ce = cudaMemsetAsync(counter, 0, sizeof(uint32_t), s);
	if (ce != cudaSuccess)
		return (int)ce;
	p.counter = counter;
	switch (G) {
	case 32: e = launch_decompress_g<32>(p, gin, threads, (int)ctas, smem, s); break;
	case 16: e = launch_decompress_g<16>(p, gin, threads, (int)ctas, smem, s); break;
	case 8: e = launch_decompress_g<8>(p, gin, threads, (int)ctas, smem, s); break;
	default: e = (int)cudaErrorInvalidValue; break;
	}
	return e;
}
