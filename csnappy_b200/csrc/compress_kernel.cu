// compress_kernel.cu -- batched Snappy fragment compressor for sm_100a.
//
// Produces, for every block, exactly the bytes csnappy_compress_fragment produces
// (/root/reference/csnappy_compress.c:469-606) for the same input and table size.
//
// The reference's greedy parse is a serial dependency chain (every probe reads and
// overwrites a hash slot), so the kernel is bound by the latency of one dependent chain per
// block times the blocks that fit on chip, not by HBM (profiles/, DESIGN.md 4.1).  The design
// therefore minimises the dependent instructions per block and keeps every resident block busy:
//
//   * one GROUP of G lanes (8, 16 or 32: a slice of one warp) per block; a persistent CTA per
//     SM holds as many groups as shared memory allows (u16 hash table of 1<<wm bytes + the
//     staged input: 18 x 4 KiB pages per SM at wm 13); groups claim blocks from a global counter;
//   * the block is staged with ONE bulk async copy (cp.async.bulk -> UBLKCP, completion on an
//     mbarrier) issued by one lane while the group clears its hash table;
//   * the parse is a loop of "probe steps".  A probe step evaluates G consecutive probe positions of the
//     reference's scan at once -- they depend only on the skip counter (csnappy_compress.c:535-542) -- finds the
//     first hit with ballot/ffs and commits exactly the table writes the serial code would have made.  The
//     post-copy bookkeeping of the reference (insert ip-1, re-probe ip, csnappy_compress.c:587-593) is folded
//     into the same step: lane 0 inserts ip-1, lane 1 probes ip, lanes 2.. already run the next scan from ip+1,
//     because that is exactly the order in which the serial code touches the table.  Two forms of the step:
//     a FAST PATH for 32 consecutive positions without shared hash slots (slot pairs are told apart by a second
//     insert + readback and the window is cut in front of the first conflicting lane; the parse continues
//     inside the window after a copy), and a GENERAL path (strided windows, three lanes on one slot -> match.any,
//     16- and 8-lane groups);
//   * match extension compares 4*G bytes per step and reduces with redux.min; emission is DEFERRED: the chain
//     stores an 8-byte token per match and every 32 tokens the group writes them out together, each lane its own
//     literal + copy tag, with byte stores straight into the block's HBM slot (L2 merges them);
//   * the per-group control flow is a flat state machine (claim / wait for the bulk copy / step), so the groups
//     sharing a warp never wait for each other at block boundaries; 32-lane groups stay in an inner window loop;
//   * fragments too large to stage in useful numbers (32 KiB + a 32 KiB table: 3 per SM) are read from global
//     memory instead (Input<false>): only the table stays in shared memory, 7 chains per SM.
#include <stdlib.h>

#include <mutex>
#include <type_traits>

#include "device_common.cuh"
#include "kernels.h"

namespace csb {

constexpr uint32_t kInPad = 48;	     // staging shift (< 16) + slack after the input for over-reads of the match extension
constexpr uint32_t kTailMargin = 15; // kInputMarginBytes, csnappy_compress.c:468
constexpr int kMaxThreads = 640;

struct CompressParams {
	csb_compress_args a;
	uint32_t *counter;     // dynamic block claim
	uint32_t table_bytes;  // 1 << wm
	uint32_t in_cap;       // longest block the staging area holds (<= 32768)
	uint32_t in_area;      // bytes reserved for the staged input incl. pad (multiple of 16)
	uint32_t group_smem;   // table_bytes + in_area + 16 (mbarrier)
	uint32_t groups;       // groups per CTA that own shared memory
};

// ---- where a block's bytes are read from ---------------------------------------------------------
// STAGED: the copy in shared memory (4 KiB pages: table + page = 12.6 KB, 18 pages per SM).  Not STAGED: global
// memory through L1 / L2 (ld.global.nc) -- for fragments of which the staged form fits only 2-3 times per SM
// (32 KiB + a 32 KiB table): with only the table in shared memory 7 chains run per SM, each a little slower
// (the candidate load is an L2 round trip).  Both forms tolerate positions at or past the end of the block:
// staged reads land in the staging pad, unstaged reads are clamped to the last word / byte of the block; either
// way bytes at or past n are unspecified and every caller masks them (min(..., room)).
template <bool STAGED>
struct Input;
template <>
struct Input<true> {
	uint32_t a;  // shared address of byte 0
	__device__ __forceinline__ uint32_t u32(uint32_t pos) const { return lds32u_a(a + pos); }
	__device__ __forceinline__ uint32_t u8(uint32_t pos) const { return lds_u8(a + pos); }
};
template <>
struct Input<false> {
	const uint8_t *base;   // byte 0
	const uint8_t *base4;  // base rounded down to a 4-byte boundary
	uint32_t boff, wlast, blast;  // base - base4; offset from base4 of the last word holding a block byte; n - 1
	__device__ __forceinline__ void set(const uint8_t *src, uint32_t n)
	{
		base = src;
		boff = (uint32_t)(reinterpret_cast<uintptr_t>(src) & 3u);
		base4 = src - boff;
		blast = n ? n - 1 : 0;
		wlast = (boff + blast) & ~3u;
	}
	static __device__ __forceinline__ uint32_t ldg32(const uint8_t *p)
	{
		uint32_t v;
		asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
		return v;
	}
	__device__ __forceinline__ uint32_t u32(uint32_t pos) const
	{
		const uint32_t o = boff + pos, w0 = min(o & ~3u, wlast), w1 = min(w0 + 4u, wlast);
		return __funnelshift_r(ldg32(base4 + w0), ldg32(base4 + w1), (o & 3u) * 8u);
	}
	__device__ __forceinline__ uint32_t u8(uint32_t pos) const
	{
		uint32_t v;
		asm volatile("ld.global.nc.u8 %0, [%1];" : "=r"(v) : "l"(base + min(pos, blast)) : "memory");
		return v;
	}
};

// ---- output: lane-parallel byte stores into the block's HBM slot ----------------------------

// literal tag + payload, csnappy_compress.c:332-371.  Returns bytes written.
template <int G, bool ST>
__device__ __forceinline__ uint32_t emit_literal(const Group<G> &g, uint8_t *dst, const Input<ST> &in, uint32_t src,
						 uint32_t len)
{
	const uint32_t v = len - 1;
	uint32_t hb, hdr;
	if (v < 60) {
		hb = 1;
		hdr = v << 2;
	} else if (v < 256) {
		hb = 2;
		hdr = (60u << 2) | (v << 8);
	} else {
		hb = 3;
		hdr = (61u << 2) | (v << 8);
	}
	const uint32_t total = hb + len;
	if (total <= (uint32_t)G) {
		// common case: header and payload in one store
		if (g.lane < total)
			dst[g.lane] = g.lane < hb ? (uint8_t)(hdr >> (8 * g.lane)) : (uint8_t)in.u8(src + g.lane - hb);
		return total;
	}
	if (g.lane < hb)
		dst[g.lane] = (uint8_t)(hdr >> (8 * g.lane));
	dst += hb;
	if (len <= 4u * G) {
		for (uint32_t i = g.lane; i < len; i += G)
			dst[i] = (uint8_t)in.u8(src + i);
	} else {
		// word stores: head bytes up to a 4-byte aligned destination, realigned source words, tail
		const uint32_t head = (uint32_t)(-(intptr_t)dst) & 3u;
		if (g.lane < head)
			dst[g.lane] = (uint8_t)in.u8(src + g.lane);
		const uint32_t words = (len - head) >> 2;
		uint32_t *dw = reinterpret_cast<uint32_t *>(dst + head);
		for (uint32_t w = g.lane; w < words; w += G)
			dw[w] = in.u32(src + head + 4 * w);
		const uint32_t tail = head + (words << 2);
		if (tail + g.lane < len)
			dst[tail + g.lane] = (uint8_t)in.u8(src + tail + g.lane);
	}
	return total;
}

// one copy element as a little-endian word + its size (2 or 3), csnappy_compress.c:373-393
__device__ __forceinline__ uint32_t copy_piece(uint32_t offset, uint32_t len, uint32_t *nb)
{
	if (len < 12 && offset < 2048) {
		*nb = 2;
		return 1u | ((len - 4) << 2) | ((offset >> 8) << 5) | ((offset & 0xff) << 8);
	}
	*nb = 3;
	return 2u | ((len - 1) << 2) | (offset << 8);
}

// split rule of csnappy_compress.c:395-415: 64s while len >= 68, one 60 if len > 64, the rest
template <int G>
__device__ __forceinline__ uint32_t emit_copy(const Group<G> &g, uint8_t *dst, uint32_t offset, uint32_t len)
{
	uint32_t done = 0;
	if (len > 64) {
		const uint32_t q = len >= 68 ? (len - 68) / 64 + 1 : 0;
		uint32_t rem = len - 64 * q;  // 4..67
		const uint32_t n60 = rem > 64 ? 1 : 0;
		rem -= 60 * n60;
		const uint32_t lead = q + n60;	// all 3-byte copy-2 elements
		for (uint32_t t = g.lane; t < lead; t += G) {
			const uint32_t w = 2u | (((t < q ? 64u : 60u) - 1) << 2) | (offset << 8);
			uint8_t *d = dst + 3 * t;
			d[0] = (uint8_t)w;
			d[1] = (uint8_t)(w >> 8);
			d[2] = (uint8_t)(w >> 16);
		}
		done = 3 * lead;
		len = rem;
	}
	uint32_t nb;
	const uint32_t w = copy_piece(offset, len, &nb);
	if (g.lane < nb)
		dst[done + g.lane] = (uint8_t)(w >> (8 * g.lane));
	return done + nb;
}

// ---- deferred emission ------------------------------------------------------------------------
// The parse only records a token per match -- (next_emit | ip << 16, candidate | length << 16), token k of
// a batch in the registers of lane k -- and every G matches the group emits them together: sizes in parallel,
// output offsets by a shuffle scan, then every lane writes ITS token (literal header + payload + copy tag).
// That replaces ~30 warp instructions per match in the serial chain by ~6 amortised ones.  Tokens
// with a literal over 32 bytes or a copy over 64 bytes are written by the whole group instead.
template <int G, bool ST>
__device__ __forceinline__ uint32_t flush_tokens(const Group<G> &g, uint8_t *dst, uint32_t op, const Input<ST> &in,
						 uint32_t count, uint32_t tx, uint32_t ty)
{
	g.sync();
	{
		const uint32_t k = g.lane;
		const bool have = k < count;
		uint32_t ne = 0, litlen = 0, off = 1, m = 4;
		if (have) {
			const uint2 t = make_uint2(tx, ty);  // token k lives in lane k (one batch = G tokens)
			ne = t.x & 0xffffu;
			litlen = (t.x >> 16) - ne;
			off = (t.x >> 16) - (t.y & 0xffffu);
			m = t.y >> 16;
		}
		const uint32_t hb = litlen == 0 ? 0u : (litlen <= 60 ? 1u : (litlen <= 256 ? 2u : 3u));
		const uint32_t q = m >= 68 ? (m - 68) / 64 + 1 : 0;  // split rule, csnappy_compress.c:395-415
		uint32_t rem = m - 64 * q;
		const uint32_t n60 = rem > 64 ? 1u : 0u;
		rem -= 60 * n60;
		const uint32_t nbc = 3 * (q + n60) + ((rem < 12 && off < 2048) ? 2u : 3u);
		const uint32_t size = have ? hb + litlen + nbc : 0u;
		uint32_t incl = size;
#pragma unroll
		for (uint32_t d = 1; d < (uint32_t)G; d <<= 1) {
			const uint32_t v = g.up(incl, d);
			if (g.lane >= d)
				incl += v;
		}
		const uint32_t at = op + incl - size;
		const bool small = have && litlen <= 32 && m <= 64;
		if (small) {
			uint8_t *d = dst + at;
			if (litlen) {
				*d++ = (uint8_t)((litlen - 1) << 2);
				for (uint32_t i = 0; i < litlen; ++i)
					d[i] = (uint8_t)in.u8(ne + i);
				d += litlen;
			}
			uint32_t nb;
			const uint32_t w = copy_piece(off, m, &nb);
			d[0] = (uint8_t)w;
			d[1] = (uint8_t)(w >> 8);
			if (nb == 3)
				d[2] = (uint8_t)(w >> 16);
		}
		unsigned big = g.ballot(have && !small);
		while (big) {
			const int kk = __ffs(big) - 1;
			big &= big - 1;
			const uint32_t bne = g.bcast(ne, kk), blit = g.bcast(litlen, kk), boff = g.bcast(off, kk);
			const uint32_t bm = g.bcast(m, kk);
			uint32_t o2 = g.bcast(at, kk);
			if (blit)
				o2 += emit_literal<G, ST>(g, dst + o2, in, bne, blit);
			emit_copy<G>(g, dst + o2, boff, bm);
		}
		op += g.bcast(incl, G - 1);
	}
	g.sync();
	return op;
}

// match extension, bounded by n (csnappy_compress.c:252-295): the first G bytes one byte per lane (most
// copies end there), then 4*G bytes per step.  ip / cd: the two 4-byte-equal positions, room = n - ip.
template <int G, bool ST>
__device__ __forceinline__ uint32_t extend_match(const Group<G> &g, const Input<ST> &in, uint32_t ip, uint32_t cd,
						 uint32_t room)
{
#ifndef CSB_EXT_BALLOT  // redux.min on the first mismatching lane: measured +1.7 % over ballot + ffs
	const uint32_t first = g.min((in.u8(cd + 4 + g.lane) != in.u8(ip + 4 + g.lane) || 4 + g.lane >= room) ? g.lane : (uint32_t)G);
	if (first < (uint32_t)G)
		return 4 + first;
#else
	const unsigned ne = g.ballot(in.u8(cd + 4 + g.lane) != in.u8(ip + 4 + g.lane) || 4 + g.lane >= room);
	if (ne)
		return 3 + __ffs(ne);
#endif
	uint32_t m = 4 + G;
	for (;;) {
		const uint32_t d = min(m + 4 * g.lane, room);
		const uint32_t x = in.u32(cd + d) ^ in.u32(ip + d);
		uint32_t mk = x ? d + ((uint32_t)(__ffs(x) - 1) >> 3) : 0x7fffffffu;
		mk = g.min(min(mk, room));
		if (mk < m + 4 * G)
			return mk;
		m += 4 * G;
	}
}

// ---- the kernel ------------------------------------------------------------------------------

enum : int { ST_NEED = 0, ST_LOADING = 1, ST_RUN = 2 };

template <int G, bool ST>
__global__ void __launch_bounds__(kMaxThreads, 1) compress_kernel(const CompressParams p)
{
	extern __shared__ __align__(128) uint8_t smem[];
	const Group<G> g;
	const uint32_t gid = threadIdx.x / G;
	if (gid >= p.groups)
		return;	 // padding lanes of the last warp (no block-wide barriers in this kernel)
	const csb_compress_args &a = p.a;
	uint8_t *gs = smem + (size_t)gid * p.group_smem;
	uint16_t *tab = reinterpret_cast<uint16_t *>(gs);
	uint8_t *sarea = gs + p.table_bytes;  // staged input, 16-byte aligned
	const uint32_t sarea_a = smem_u32(sarea), tab_a = smem_u32(tab);
	Input<ST> in;  // staged: sarea_a + (src & 15), the shared address where the block's first byte lands
	const uint32_t bar = smem_u32(sarea + p.in_area);
	const unsigned full = (G == 32) ? 0xffffffffu : ((1u << G) - 1u);

	if (g.lane == 0) {
		mbar_init(bar, 1);
		fence_mbar_init();
	}
	g.sync();

	int state = ST_NEED;
	uint32_t parity = 0;
	// per-block state
	uint32_t blk = 0, n = 0, ip_limit = 0, op = 0, next_emit = 0, wbase = 1, t = 0, ntok = 0;
	uint32_t tx = 0, ty = 0;  // this lane's token of the current batch (token k of a batch lives in lane k)
	int shift = 0, j0 = 0;
	uint8_t *dst = nullptr;

	for (;;) {
		if (state == ST_NEED) {
			if (g.lane == 0)
				blk = atomicAdd(p.counter, 1u);
			blk = g.bcast(blk, 0);
			if (blk >= a.n_blocks)
				break;
			const uint64_t in_at = a.in_off ? a.in_off[blk] : (uint64_t)blk * a.in_stride;
			n = a.in_len ? a.in_len[blk] : a.uniform_len;
			if (a.total_len) {
				const uint64_t left = a.total_len > in_at ? a.total_len - in_at : 0;
				if (left < n)
					n = (uint32_t)left;
			}
			if (n > p.in_cap) {
				// REQUIRES of the reference (csnappy.h:38): at most 32768 bytes -- and never more than the staging
				// area holds.  The reference has no error channel here; the batch has one: the size entry.
				if (g.lane == 0)
					a.out_len[blk] = CSB_LEN_REFUSED;
				continue;
			}
			const uint8_t *src = a.in + in_at;
			dst = a.out + (uint64_t)blk * a.out_stride;
			// table size for this block (csnappy_compress.c:638-646 when SHRINK_TABLE is set)
			int ws = a.wm;
			if ((a.flags & 1u) && n < CSB_FRAGMENT_MAX) {
				for (ws = 9; ws < a.wm; ++ws)
					if ((1u << (ws - 1)) >= n)
						break;
			}
			shift = 33 - ws;
			ip_limit = n >= kTailMargin ? n - kTailMargin : 0;
			op = 0;
			next_emit = 0;
			wbase = 1;
			j0 = 0;
			t = 0;

			g.sync();  // every lane is done with the previous block's input and table
			if (n >= kTailMargin) {	 // zero the table, csnappy_compress.c:501
				uint4 *t4 = reinterpret_cast<uint4 *>(tab);
				const uint32_t nv = (1u << ws) >> 4;
				const uint4 z = make_uint4(0, 0, 0, 0);
				for (uint32_t i = g.lane; i < nv; i += G)
					t4[i] = z;
			}
			if constexpr (ST) {
				bool bulk;
				in.a = sarea_a + stage_block<G>(g, sarea, src, n, bar, &bulk);
				state = bulk ? ST_LOADING : ST_RUN;
			} else {
				in.set(src, n);
				state = ST_RUN;
			}
			g.sync();
		}
		if (state == ST_LOADING) {
			if (g.ballot(mbar_test(bar, parity)) != full)
				continue;
			parity ^= 1u;
			state = ST_RUN;
		}

		bool fin;
		do {
			fin = false;
			if (n < kTailMargin) {  // csnappy_compress.c:497: too short to probe at all -- one literal, and no read past n
				fin = true;
				break;
			}
			// ---- fast path (G == 32): a window of CONSECUTIVE positions in which no two lanes share a hash slot ----
			// The common window of compressible data: lanes 0..cut-1 probe wbase + lane with stride 1 (probe indices
			// j0 + lane <= 31: page start, right behind a copy, or the stride-1 head of a later window), so
			// ip = wbase + lane needs no shuffle, "all lanes valid" is a scalar test, and with every slot private to one
			// lane the table entries read before the inserts ARE the candidates the serial code sees, however many
			// copies the window holds.  The candidate bytes are loaded before the readback is evaluated (both depend
			// only on `old`).  Two lanes on one slot (a third of the windows on URL text: repeated 4-byte groups) are
			// told apart by a second insert + readback -- after it each lane of a pair knows its partner's position --
			// and the window is CUT in front of the first lane that has a lower partner: the lanes before it are
			// conflict-free, the lanes from it on take their inserts back and are probed again by the next window.
			// Three or more lanes on one slot restore the table and hand the window to the general code below.
			// A STRIDED window (UNI = false: probe indices from 32 on, strides 2, 3, ... -- the second and later
			// windows of a scan that found nothing) takes the same front end and the same cut; it holds one copy at
			// most, positions come from the lanes by shuffle, and lanes are compared through their positions.
			auto fast_window = [&](auto uni_c) -> bool {
				constexpr bool UNI = decltype(uni_c)::value;
				uint32_t cut, pp, s;
				if constexpr (UNI) {
					cut = j0 > 0 ? 32u - (uint32_t)j0 : 32u;
					pp = wbase + g.lane;
					s = 1;
				} else {
					const uint32_t s0 = (32u + j0) >> 5;
					const int jb = ((j0 >> 5) + 1) << 5;  // first probe index with stride s0 + 1
					cut = 32u;
					pp = wbase + g.lane * s0 + max(j0 + (int)g.lane - jb, 0);
					s = (32u + j0 + g.lane) >> 5;
				}
				bool valid = pp + s <= ip_limit && g.lane < cut;
				// consecutive positions: invalid lanes read on inside the staging pad (pp + 3 <= n + 19) and never store
				const uint32_t bytes = in.u32(UNI || valid ? pp : 0u);
				const uint32_t slot = tab_a + 2 * ((bytes * kHashMul) >> shift);
				const uint32_t old = lds_u16(slot);
				g.sync();
				if (valid)
					sts_u16(slot, pp);
				g.sync();
				const uint32_t rb1 = lds_u16(slot);
				const uint32_t cand = valid ? old : 0u;  // (blocks under 15 bytes never clear the table)
				const uint32_t cb = in.u32(cand);
				const bool lost = valid && rb1 != pp;
				if (g.ballot(lost)) {
					g.sync();
					if (lost)
						sts_u16(slot, pp);
					g.sync();
					const uint32_t rb2 = lds_u16(slot);
					const bool triple = g.ballot(lost && rb2 != pp) != 0;
					g.sync();  // every lane has read back before anybody rewrites
					if (triple) {
						if (valid)
							sts_u16(slot, old);
						g.sync();
						return false;
					}
					const uint32_t q = lost ? rb1 : rb2;  // the partner's position (own position: none)
					const bool hasp = valid && q != pp;
					cut = __ffs(g.ballot(hasp && q < pp)) - 1;  // first lane with a lower partner (there is one)
					const uint32_t pcut = UNI ? wbase + cut : g.bcast(pp, (int)cut);  // its position
					const bool upper = g.lane >= cut;
					// lanes from the cut on leave the table as if they had never inserted; a lane in front of the
					// cut whose partner is behind it owns the slot again
					const bool wr_old = valid && upper && (!hasp || (q >= pcut && pp < q));
					const bool wr_pp = valid && !upper && hasp;
					if (wr_old || wr_pp)
						sts_u16(slot, wr_pp ? pp : old);
					valid = valid && !upper;
					g.sync();
				}
				const unsigned H = g.ballot(valid && cb == bytes);
				bool all_valid;
				if constexpr (UNI)
					all_valid = wbase + cut - 1 < ip_limit;
				else
					all_valid = g.ballot(valid) == (cut >= 32u ? 0xffffffffu : (1u << cut) - 1u);
				uint32_t cur = t;
				for (;;) {
					const unsigned elig = H & (0xffffffffu << cur);
					if (!elig) {
						if (!all_valid) {
							fin = true;  // ran into ip_limit without a hit
						} else {
							if constexpr (UNI)
								wbase += cut;
							else  // position of the probe behind the last one of this window
								wbase = cut < 32u ? g.bcast(pp, (int)cut) : g.bcast(pp + s, 31);
							j0 += (int)cut;
							t = 0;
						}
						break;
					}
					const uint32_t f = __ffs(elig) - 1;
					const uint32_t ip = UNI ? wbase + f : g.bcast(pp, (int)f), cd = g.bcast(cand, (int)f);
					const uint32_t m = extend_match<G, ST>(g, in, ip, cd, n - ip);
					if (g.lane == ntok) {
						tx = next_emit | (ip << 16);
						ty = cd | (m << 16);
					}
					if (++ntok == (uint32_t)G) {
						op = flush_tokens<G, ST>(g, dst, op, in, ntok, tx, ty);
						ntok = 0;
					}
					next_emit = ip + m;
					if (next_emit >= ip_limit) {
						fin = true;
						break;
					}
					// lane of the re-probe position if the parse can stay inside this window
					const uint32_t nl = UNI ? next_emit - wbase : 0x7fffffffu;
					// lanes skipped by the copy never insert: undo (ip-1 = lane nl-1 stays, ip = lane nl goes on)
					if (valid && g.lane > f && g.lane + 1 < nl)
						sts_u16(slot, old);
					bool stay = false;
					if constexpr (UNI)
						stay = nl < cut;
					if (!stay) {
						wbase = next_emit - 1;
						j0 = -2;
						t = 1;
						break;
					}
					if constexpr (UNI) {
						cur = nl;
						j0 = -(int)(nl + 1);
					}
				}
				if (!fin)
					g.sync();
				return true;
			};
			bool done_fast = false;
			if (G == 32)
				done_fast = j0 < 24 ? fast_window(std::true_type{}) : fast_window(std::false_type{});
			if (!done_fast) {
				// ---- one WINDOW of G probe positions (csnappy_compress.c:535-552 and 587-593) ----
				// Lane k probes the k-th position of the window.  j0 + k is that probe's index in the
				// reference's skip schedule (stride (32 + index) >> 5); lanes whose index is negative
				// are the post-copy bookkeeping positions (t == 1: lane 0 = ip-1, insert only; lane 1 =
				// ip, the re-probe) or lie before an in-window scan restart.  While every stride in the
				// window is 1 ("uni") the window is G consecutive bytes and the parse can CONTINUE
				// inside it after a copy: the lanes behind the copy already hold their hash, table
				// entry and compare result, and those stay valid as long as no two lanes of the window
				// share a hash slot.  That is checked by inserting speculatively and reading back;
				// lanes that turn out not to insert (skipped by a copy, or behind the end) undo.
				const bool uni = j0 <= 32 - G;
				uint32_t pp, s;
				if (uni) {
					pp = wbase + g.lane;
					s = 1;
				} else {
					const uint32_t s0 = (32u + j0) >> 5;
					const int jb = ((j0 >> 5) + 1) << 5;  // first probe index with stride s0 + 1
					pp = wbase + g.lane * s0 + max(j0 + (int)g.lane - jb, 0);
					s = (32u + j0 + g.lane) >> 5;
				}
				const bool valid = pp + s <= ip_limit;
				const uint32_t bytes = in.u32(valid ? pp : 0u);
				const uint32_t slot = tab_a + 2 * ((bytes * kHashMul) >> shift);
				const uint32_t old = lds_u16(slot);
				g.sync();
				if (valid)
					sts_u16(slot, pp);
				g.sync();
				const uint32_t rb1 = lds_u16(slot);
				const bool lost = valid && rb1 != pp;
				const bool exact = g.ballot(lost) != 0;	 // two lanes share a slot
				// candidate: the table -- or, with shared slots, the latest lower lane with the same hash
				// (invalid lanes must not follow a stale entry: blocks under 15 bytes never clear the table)
				uint32_t cand = valid ? old : 0u;
				unsigned same = 0;
				if (exact) {
					// Who shares a slot with whom?  For the common case of PAIRS in a window of consecutive
					// positions a second insert + readback answers it (the loser of the first round saw the
					// winner's position; after the losers insert, the winner sees its loser); three or more
					// lanes on one slot, or a strided window, fall back to match.any (slow: ~300 cycles).
					bool paired = false;
					if (uni) {
						g.sync();
						if (lost)
							sts_u16(slot, pp);
						g.sync();
						const uint32_t rb2 = lds_u16(slot);
						if (!g.ballot(lost && rb2 != pp)) {
							paired = true;
							const uint32_t q = lost ? rb1 : rb2;  // the partner's position (own position: none)
							same = 1u << g.lane;
							if (valid && q != pp)
								same |= 1u << (q - wbase);
						}
					}
					g.sync();  // every lane has read back before anybody restores
					if (valid)
						sts_u16(slot, old);  // back to the state before this window
					if (!paired)
						same = g.match(valid ? slot : (0x80000000u | g.lane));
					const unsigned lower = same & ((1u << g.lane) - 1u);
					const uint32_t lp = g.bcast(pp, lower ? 31 - __clz(lower) : (int)g.lane);
					if (lower)
						cand = lp;
					g.sync();
				}
				const uint32_t cb = in.u32(cand);
				const unsigned H = g.ballot(valid && cb == bytes);
				const unsigned V = g.ballot(valid);
				const bool multi = uni && !exact;

				uint32_t cur = t;      // first lane that may hit
				unsigned fhit = 32;    // exact windows: the (single) hit lane
				for (;;) {
					const unsigned elig = H & (full << cur) & full;
					if (!elig) {
						if (V != full) {
							fin = true;  // ran into ip_limit without a hit
						} else if (uni) {
							wbase += G;
							j0 += G;
							t = 0;
						} else {
							const uint32_t s0 = (32u + j0) >> 5;
							const int jb = ((j0 >> 5) + 1) << 5;
							wbase += G * s0 + max(j0 + G - jb, 0);
							j0 += G;
							t = 0;
						}
						break;
					}
					const unsigned f = __ffs(elig) - 1;
					const uint32_t ip = g.bcast(pp, (int)f), cd = g.bcast(cand, (int)f);
					const uint32_t m = extend_match<G, ST>(g, in, ip, cd, n - ip);
					// record the match; emission is deferred (flush_tokens)
					if (g.lane == ntok) {
						tx = next_emit | (ip << 16);
						ty = cd | (m << 16);
					}
					if (++ntok == (uint32_t)G) {
						op = flush_tokens<G, ST>(g, dst, op, in, ntok, tx, ty);
						ntok = 0;
					}
					next_emit = ip + m;
					if (next_emit >= ip_limit) {
						fin = true;
						break;
					}
					// lane of the re-probe position if the parse can stay inside this window
					const uint32_t nl = uni ? next_emit - wbase : 0x7fffffffu;
					if (!exact) {
						// lanes skipped by the copy never insert: undo (ip-1 = lane nl-1 stays, ip = lane nl goes on)
						if (valid && g.lane > f && g.lane + 1 < nl)
							sts_u16(slot, old);
					} else {
						fhit = f;
					}
					if (!multi || nl >= (uint32_t)G) {
						wbase = next_emit - 1;
						j0 = -2;
						t = 1;
						break;
					}
					// continue inside the window: lane nl-1 inserted ip-1, lane nl re-probes, scan restarts at nl+1
					cur = nl;
					j0 = -(int)(nl + 1);
				}
				if (!fin) {
					if (exact) {
						// the table is in its pre-window state: lanes up to the hit insert, the highest lane
						// of an equal-hash run owns the slot
						const unsigned I = fhit < 32 ? ((2u << fhit) - 1u) : 0xffffffffu;
						const unsigned rivals = same & I & ~((2u << g.lane) - 1u);
						if (valid && ((I >> g.lane) & 1u) && !rivals)
							sts_u16(slot, pp);
					}
					g.sync();
				}
			}  // general window
		} while (G == 32 && !fin);  // one group per warp: stay in the window loop until the block is parsed
		if (fin) {
			if (ntok)
				op = flush_tokens<G, ST>(g, dst, op, in, ntok, tx, ty);
			ntok = 0;
			if (next_emit < n)
				op += emit_literal<G, ST>(g, dst + op, in, next_emit, n - next_emit);
			if (g.lane == 0)
				a.out_len[blk] = op;
			state = ST_NEED;
		}
	}
}

}  // namespace csb

using namespace csb;

template <int G, bool ST>
static int launch_compress_g(const CompressParams &p, int threads, int ctas, size_t smem, cudaStream_t s)
{
	// The attributes belong to the kernel, not to the launch: a concurrent caller that set a smaller shared-memory
	// limit between our set and our launch would make the launch fail.  Set and launch as one step.
	static std::mutex mu;
	std::lock_guard<std::mutex> lk(mu);
	cudaError_t e = cudaFuncSetAttribute(compress_kernel<G, ST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	if (e != cudaSuccess)
		return (int)e;
	if (!ST) {  // the input is read through L1: leave it whatever the tables do not need
		e = cudaFuncSetAttribute(compress_kernel<G, ST>, cudaFuncAttributePreferredSharedMemoryCarveout,
					 (int)((smem + 2048) * 100 / (228 * 1024) + 1));
		if (e != cudaSuccess)
			return (int)e;
	}
	compress_kernel<G, ST><<<ctas, threads, smem, s>>>(p);
	count_launch();
	return (int)cudaGetLastError();
}

extern "C" int csb_launch_compress(const struct csb_compress_args *a, csb_stream_t s)
{
	if (a->n_blocks == 0)
		return 0;
	DeviceInfo di;
	int e = device_info(&di);
	if (e)
		return e;

	CompressParams p;
	p.a = *a;
	p.table_bytes = 1u << a->wm;
	uint32_t in_cap = a->uniform_len;
	if (a->in_len)	// per-block lengths: bounded by the stride when strided, else by the format
		in_cap = (!a->in_off && a->in_stride && a->in_stride < CSB_FRAGMENT_MAX) ? (uint32_t)a->in_stride : CSB_FRAGMENT_MAX;
	if (in_cap > CSB_FRAGMENT_MAX)
		in_cap = CSB_FRAGMENT_MAX;
	p.in_cap = in_cap;
	p.in_area = ((in_cap + 15u) & ~15u) + kInPad;
	p.group_smem = p.table_bytes + p.in_area + 16;

	const int G = a->lanes ? a->lanes : 32;
	const int ctas_per_sm = a->ctas_per_sm > 0 ? a->ctas_per_sm : 1;
	// shared memory per CTA: the SM's carve-out divided among resident CTAs (1 KiB reserved each)
	long budget = (long)di.smem_per_sm / ctas_per_sm - 1024;
	if (budget > di.smem_per_block_optin)
		budget = di.smem_per_block_optin;
	int groups = (int)(budget / p.group_smem);
	const int max_groups = kMaxThreads / G;
	// Blocks of which fewer than 8 fit an SM staged are read from global memory instead when that at least doubles the
	// chains per SM (32 KiB / wm 15: 7 instead of 3, 14.7 -> 20 GB/s; an unstaged chain runs at ~57 % of a staged one, so
	// 3 instead of 2 at wm 16 or 13 instead of 7 at 16 KiB / wm 14 do not pay).  stage_input: 0 = this rule, 1 = always
	// stage, 2 = never stage.
	bool staged = true;
	if (G == 32 && a->stage_input != 1) {
		const uint32_t lean = p.table_bytes + 16;
		const int lean_groups = (int)(budget / lean) < max_groups ? (int)(budget / lean) : max_groups;
		// (a batch that fits the staged slots of the machine in one go gains nothing from more slots)
		if (a->stage_input == 2 || (groups < 8 && lean_groups >= 2 * groups && a->n_blocks > (uint32_t)(di.sm_count * (groups > 0 ? groups : 1)))) {
			staged = false;
			p.in_area = 0;
			p.group_smem = lean;
			groups = lean_groups;
		}
	}
	if (groups > max_groups)
		groups = max_groups;
	{
		static int cap_env = -1;  // experiments: CSB_COMPRESS_GROUPS caps the groups per CTA (the rest of the array stays L1)
		if (cap_env < 0) {
			const char *e = getenv("CSB_COMPRESS_GROUPS");
			cap_env = e ? atoi(e) : 0;
		}
		if (cap_env > 0 && groups > cap_env)
			groups = cap_env;
	}
	if (groups < 1)
		return (int)cudaErrorInvalidConfiguration;
	long want = ((long)a->n_blocks + groups - 1) / groups;
	long ctas = (long)di.sm_count * ctas_per_sm;
	if (ctas > want) {
		// small batch: spread the blocks over all SMs instead of filling a few CTAs
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
	case 32:
		e = staged ? launch_compress_g<32, true>(p, threads, (int)ctas, smem, s)
			   : launch_compress_g<32, false>(p, threads, (int)ctas, smem, s);
		break;
	case 16: e = launch_compress_g<16, true>(p, threads, (int)ctas, smem, s); break;
	case 8: e = launch_compress_g<8, true>(p, threads, (int)ctas, smem, s); break;
	default: e = (int)cudaErrorInvalidValue; break;
	}
	return e;
}
