/*
 * kernels.h -- C-linkage launchers of the sm_100a kernels, called by the plain-C
 * shim (csnappy_shim.c).  Internal to the library; the public ABI is in include/.
 */
#ifndef CSNAPPY_B200_KERNELS_H_
#define CSNAPPY_B200_KERNELS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st *csb_stream_t; /* == cudaStream_t */

#define CSB_FRAGMENT_MAX 32768u
#define CSB_LEN_REFUSED 0xffffffffu /* == CSNAPPY_BATCH_LEN_REFUSED */

struct csb_compress_args {
	const uint8_t *in;
	const uint64_t *in_off; /* NULL => i * in_stride */
	uint64_t in_stride;
	const uint32_t *in_len; /* NULL => uniform_len (clipped by total_len if nonzero); an entry above 32768 or above
				   the stride is refused: out_len[i] = CSB_LEN_REFUSED, nothing written */
	uint32_t uniform_len;
	uint64_t total_len;	/* nonzero: block i has min(uniform_len, total_len - i*in_stride) bytes */
	uint32_t n_blocks;
	uint8_t *out;
	uint64_t out_stride;
	uint32_t *out_len;
	int wm;			/* log2 of hash-table bytes, 9..16 */
	uint32_t flags;		/* CSNAPPY_BATCH_SHRINK_TABLE */
	int lanes;		/* lanes cooperating on one block: 8, 16, 32 (0 = default) */
	int ctas_per_sm;	/* 0 = default */
	uint32_t *counter;	/* device word for the block claim counter (NULL: a word of the per-device ring, pack_kernel.cu next_counter) */
	int stage_input;	/* 0: choose; 1: always stage the block in shared memory; 2: read it from global memory (32-lane groups) */
};

struct csb_decompress_args {
	const uint8_t *in;
	const uint64_t *in_off;
	uint64_t in_stride;
	const uint32_t *in_len;
	uint32_t n_blocks;
	uint8_t *out;
	uint64_t out_stride;
	const uint64_t *out_off; /* NULL => i * out_stride; set: block i's output at out + out_off[i] (the lane-per-block
				    decoder, which needs 16-byte aligned strided slots, is then not selected) */
	const uint32_t *out_cap; /* NULL => uniform_cap */
	uint32_t uniform_cap;
	uint32_t *out_len;
	int32_t *status;
	uint32_t flags;		/* CSNAPPY_BATCH_WITH_HEADER | CSNAPPY_BATCH_RAW_IF_FULL */
	uint32_t max_in_len;	/* staging hint: longest input block (0 = derive) */
	int lanes;
	int ctas_per_sm;
	uint32_t *counter;	/* device word for the block claim counter (NULL: a word of the per-device ring, pack_kernel.cu next_counter) */
	int stage_input;	/* 0: choose; 1: always stage in shared memory; 2: stage only the output; 3: warp per block against
				   global memory; 4: one lane per block (decompress_lane_kernel.cu) */
	int smem_kb;		/* unstaged mode: shared memory to use per SM, rest stays L1 (0 = default) */
	int lane_warps;		/* lane-per-block decoder: warps (of 32 blocks) in flight per SM (0 = default) */
};

/* all return 0 or a cudaError_t value (> 0) */
int csb_launch_compress(const struct csb_compress_args *a, csb_stream_t s);
int csb_launch_decompress(const struct csb_decompress_args *a, csb_stream_t s);
int csb_launch_decompress_lane(const struct csb_decompress_args *a, csb_stream_t s); /* one lane per block; out and out_stride 16-byte aligned */
int csb_launch_pack(const uint8_t *slots, uint64_t slot_stride, const uint32_t *len,
		    uint32_t n_blocks, uint8_t *packed, uint64_t *off, csb_stream_t s);
int csb_launch_pack_stored(const uint8_t *slots, uint64_t slot_stride, const uint32_t *len, uint32_t n_blocks,
			   const uint8_t *in, uint32_t page_len, uint64_t total_in, uint32_t *clen,
			   uint8_t *packed, uint64_t *off, csb_stream_t s);
int csb_launch_scan(const uint32_t *len, uint32_t n_blocks, uint64_t *off, csb_stream_t s);
/* the two halves of csb_launch_pack_stored around its scan: clen[i] = min(len[i], input length of block i), and the
 * gather of the slots (or, with raw, of the stored input blocks) to packed + off[i] */
int csb_launch_clamp(const uint32_t *len, uint32_t n_blocks, uint32_t page_len, uint64_t total_in, uint32_t *clen,
		     csb_stream_t s);
int csb_launch_gather(const uint8_t *slots, uint64_t slot_stride, const uint32_t *len, uint32_t n_blocks, uint8_t *packed,
		      const uint64_t *off, const uint8_t *raw, uint32_t page_len, uint64_t total_in, const uint32_t *slot_len,
		      csb_stream_t s);
/* batched csnappy_compress framing: header + fragments of every buffer into its output slot (pack_kernel.cu) */
int csb_launch_frame(const uint8_t *slots, uint64_t slot_stride, const uint32_t *len, const uint64_t *off,
		     const uint32_t *fbuf, const uint32_t *bfirst, const uint32_t *blen, uint32_t n_frag,
		     uint32_t n_buffers, uint8_t *out, uint64_t out_stride, uint32_t *out_len, csb_stream_t s);
/* Parallel decoder of ONE long raw stream (stream_kernel.cu).  aux tables: which = 0 -> per input byte, 1 -> per output
 * byte.  Returns 0, 1 ("not for this stream": caller falls back to the warp-per-stream path), or a cudaError_t (> 1). */
size_t csb_stream_aux_bytes(uint32_t src_len, uint32_t cap, int which);
int csb_launch_decompress_stream(const uint8_t *d_in, uint32_t src_len, uint8_t *d_out, uint32_t cap, uint32_t *d_out_len,
				 int32_t *d_status, void *d_aux_in, void *d_aux_out, csb_stream_t s);
uint64_t csb_launch_count(void);

/* Snappy framing format (framed_kernel.cu) */
#define CSB_FRAMED_CHUNK 65536u
struct csb_framed_result {	/* device word block of one framed read */
	uint32_t n_data, n_comp; /* data chunks / compressed chunks the walk recorded */
	uint64_t walk_key;	 /* the walk's failure: position * 4 + class (0 malformed, 1 output, 2 checksum); ~0 none */
	uint64_t walk_out;	 /* output bytes of the recorded chunks */
	uint64_t verify_key;	 /* smallest failure key of the verify step */
};
struct csb_framed_table {	/* per data chunk i / per compressed chunk j, in stream order */
	uint64_t *pos, *out_off;
	uint32_t *out_len, *crc, *cidx; /* cidx: index j of a compressed chunk, ~0 for a stored one */
	uint64_t *c_pos, *c_out_off;	/* decoder input: src + 8 + c_pos[j], c_len[j] bytes (varint included) */
	uint32_t *c_len, *c_produced;
	int32_t *c_status;
	struct csb_framed_result *res;
};
/* masked CRC-32C per 65536-byte chunk of in[0, n); with flen (sizes of the 32 KiB fragments) also the record sizes */
int csb_launch_framed_crc(const uint8_t *in, uint64_t n, uint32_t *crc, const uint32_t *flen, uint32_t n_frag, uint32_t *rec,
			  csb_stream_t s);
int csb_launch_framed_write(const uint8_t *in, uint64_t n, const uint8_t *slots, uint64_t slot_stride, const uint32_t *flen,
			    uint32_t n_frag, const uint32_t *crc, const uint32_t *rec, const uint64_t *off, uint8_t *out,
			    uint64_t *out_length, csb_stream_t s);
int csb_launch_framed_walk(const uint8_t *src, uint64_t len, uint64_t cap, const struct csb_framed_table *t, csb_stream_t s);
int csb_launch_framed_verify(const uint8_t *src, uint8_t *dst, uint32_t n_data, const struct csb_framed_table *t,
			     uint64_t *out_length, int32_t *status, uint64_t *failed_offset, csb_stream_t s);

/* Many framed streams in one call.  Writer tables, laid out by the host: per 32 KiB fragment (compress input), per
 * 65536-byte chunk and per stream; crc / rec / off are written on the device. */
struct csb_framed_batch_wtable {
	const uint32_t *flen;	  /* compressed size per fragment (compress output) */
	const uint64_t *c_in;	  /* per chunk: absolute input offset */
	const uint32_t *c_len;	  /* per chunk: bytes, 1..65536 */
	const uint32_t *c_stream; /* per chunk: its stream */
	const uint32_t *c_frag;	  /* per chunk: its first fragment (a second one follows when c_len > 32768) */
	uint32_t *crc, *rec;	  /* per chunk: masked CRC, record size */
	const uint64_t *off;	  /* per chunk: scanned record offset; off[n_chunks] = total */
	const uint64_t *s_out;	  /* per stream: absolute output slot */
	const uint32_t *s_first;  /* per stream: first chunk; s_first[n_streams] = n_chunks */
};
/* Reader tables.  The walk of stream i writes its data chunks into its own region [s_reg[i], s_reg[i] + s_len[i] / 8 + 1)
 * of the r_* tables with stream-relative positions; the compaction copies them into the contiguous d_* / c_* tables
 * (stream order, absolute offsets) at the scanned counts d_base / c_base. */
struct csb_framed_batch_rtable {
	const uint64_t *s_src, *s_len, *s_dst, *s_cap, *s_reg; /* per stream, from the host */
	uint32_t *nd, *nc;				       /* per stream: data / compressed chunks recorded */
	uint64_t *walk_key, *walk_out, *verify_key;	       /* per stream, as csb_framed_result */
	uint64_t *d_base, *c_base;			       /* scans of nd / nc, n_streams + 1 entries */
	uint64_t *totals;				       /* [0] data chunks, [1] compressed chunks of the batch */
	uint64_t *r_pos, *r_out;			       /* region tables: relative position / output offset */
	uint32_t *r_len, *r_crc, *r_cidx, *r_plen;	       /* r_cidx: stream-local compressed index, ~0 stored */
	uint64_t *pos, *out_off;			       /* compacted data chunks: absolute src / dst offsets */
	uint32_t *out_len, *crc, *cidx, *stream;
	uint64_t *c_pos, *c_out_off; /* compacted compressed chunks: decoder input src + 8 + c_pos[j], c_len[j] bytes */
	uint32_t *c_len, *c_produced;
	int32_t *c_status;
};
int csb_launch_framed_batch_crc(const uint8_t *in, uint32_t n_chunks, const struct csb_framed_batch_wtable *t, csb_stream_t s);
int csb_launch_framed_batch_write(const uint8_t *in, uint32_t n_chunks, uint32_t n_streams, const uint8_t *slots,
				  uint64_t slot_stride, const struct csb_framed_batch_wtable *t, uint8_t *out,
				  uint64_t *out_length, csb_stream_t s);
/* length != NULL: the decompressed_length walk (unbounded capacity, no table writes) into length[i] / status[i] */
int csb_launch_framed_batch_walk(const uint8_t *src, uint32_t n_streams, const struct csb_framed_batch_rtable *t,
				 uint64_t *length, int32_t *status, csb_stream_t s);
int csb_launch_framed_batch_compact(uint32_t n_streams, const struct csb_framed_batch_rtable *t, csb_stream_t s);
int csb_launch_framed_batch_verify(const uint8_t *src, uint8_t *dst, uint32_t n_data, uint32_t n_streams,
				   const struct csb_framed_batch_rtable *t, uint64_t *out_length, int32_t *status,
				   uint64_t *failed_offset, csb_stream_t s);

/* Page container on device buffers (bc_kernel.cu).
 * Index scan of n u32 entries at ent (any alignment), grid-wide: index[i] = first_off + the sum of the entries before
 * i while that sum plus entry i stays within room and no entry so far is above max_clen (the decodable prefix),
 * bad_off for every later page.  len (optional): the entry inside the prefix, 0 behind it.  prefix (optional, set to
 * 0xffffffff beforehand): the first page behind the prefix, left as it is when there is none.  index[] is the only
 * memory the scan needs: each CTA's partial sum waits in the first word of its own range. */
int csb_launch_bc_index(const uint8_t *ent, uint32_t n, uint32_t max_clen, uint64_t first_off, uint64_t room,
			uint64_t bad_off, uint64_t *index, uint32_t *len, uint32_t *prefix, csb_stream_t s);
/* [u32 n][u32 clen[n]] at cont (any alignment); *cont_length = index[n - 1] + clen[n - 1] (4 for n == 0) */
int csb_launch_bc_header(const uint32_t *clen, uint32_t n, const uint64_t *index, uint8_t *cont, uint64_t *cont_length,
			 csb_stream_t s);
/* page requests -> decoder input in_off / in_len and tag (0, or the status of a request that is not decoded) */
int csb_launch_bc_requests(const uint8_t *cont, uint64_t cont_length, uint32_t max_clen, const uint64_t *index,
			   uint32_t nr, const uint32_t *pages, uint32_t n, uint64_t *in_off, uint32_t *in_len, int32_t *tag,
			   csb_stream_t s);
int csb_launch_bc_request_status(const int32_t *tag, uint32_t n, uint32_t *out_len, int32_t *status, csb_stream_t s);
struct csb_bc_result {	/* device words of one whole-container read */
	uint64_t key;	/* smallest (page << 32 | status) of a failed prefix page; set to ~0 beforehand */
	uint32_t prefix; /* first page behind the decodable prefix; set to ~0 beforehand */
	uint32_t pad;
	uint64_t sum;	/* bytes produced by the prefix's good pages; set to 0 beforehand */
};
/* hdr_rc != 0 or nr == 0: *status = hdr_rc, *out_length = 0; else the reduction of out_len / status_pages over the
 * prefix and the index error at its end into *status, *out_length and (on failure, when given) *failed_page */
int csb_launch_bc_finish(const uint32_t *out_len, const int32_t *status_pages, uint32_t nr, int32_t hdr_rc,
			 struct csb_bc_result *r, uint64_t *out_length, int32_t *status, uint32_t *failed_page,
			 csb_stream_t s);

#ifdef __cplusplus
}
#endif
#endif
