/*
 * csnappy_batch.h -- batched entry points of the B200-native Snappy codec.
 *
 * These are the additions BASELINE.json's north_star asks for next to the
 * csnappy.h drop-in: many independent blocks (zram 4 KiB pages,
 * kernel_3_2_10.patch:1348-1372; block_compressor pages, block_compressor.c:
 * 113-134, 307-335, 365-387; the 32 KiB fragments of csnappy_compress,
 * csnappy_compress.c:636-654) handed to the GPU in ONE call.  Per block the
 * semantics are exactly those of csnappy_compress_fragment /
 * csnappy_decompress_noheader / csnappy_decompress.
 *
 * Pointers named d_* are DEVICE pointers on the current CUDA device, pointers
 * named h_* are HOST pointers.  `stream` is a cudaStream_t passed as void*
 * (NULL = the legacy default stream).  Device-pointer calls are asynchronous
 * with respect to the host: they enqueue work on `stream` and return.
 *
 * Block i of a batch lives at
 *     base + (off ? off[i] : i * stride)
 * Strided outputs need  out_stride >= csnappy_max_compressed_length(len)  for
 * compression (the compressor never bounds-checks its output, exactly like the
 * reference, cl_tester.c:120-165) and >= capacity for decompression.
 * Fast paths engage when base, stride and offsets are multiples of 16.
 *
 * Every function returns 0, CSNAPPY_E_DEVICE or CSNAPPY_E_BAD_ARG (the framed and host container readers also a
 * stream's decode result, csnappy_bc_index CSNAPPY_E_DATA_MALFORMED for a short index; the device container readers
 * put theirs in device words); per-block
 * decoder results go to d_status[] / h_status[].
 */
#ifndef CSNAPPY_B200_CSNAPPY_BATCH_H_
#define CSNAPPY_B200_CSNAPPY_BATCH_H_

#include <stddef.h>
#include <stdint.h>

#include "csnappy.h"

#ifdef __cplusplus
extern "C" {
#endif

/* flags */
#define CSNAPPY_BATCH_SHRINK_TABLE 0x1u /* compress: per block, apply csnappy_compress()'s
					   short-chunk table rule (csnappy_compress.c:638-646) */
#define CSNAPPY_BATCH_WITH_HEADER 0x2u  /* decompress: blocks start with a varint32 length;
					   csnappy_decompress() semantics incl. -1 / -2
					   (csnappy_decompress.c:394-411) */
#define CSNAPPY_BATCH_RAW_IF_FULL 0x4u  /* decompress: a block whose input length equals its
					   output capacity is a stored block and is copied
					   (block_compressor.c:378) */

/*
 * Batched csnappy_compress_fragment (csnappy_compress.c:469-606).
 *   d_in_len == NULL  => every block is uniform_in_len bytes.
 *   d_out_len[i]      <- compressed size of block i.
 * Block lengths must be <= 32768 (and <= in_stride when strided); 9 <= wm <= 16.
 * The reference has no error channel on this side (csnappy.h:38 only REQUIRES it); here a
 * d_in_len[i] that breaks the rule is refused: d_out_len[i] = CSNAPPY_BATCH_LEN_REFUSED and
 * nothing is written to the block's slot.
 */
#define CSNAPPY_BATCH_LEN_REFUSED 0xffffffffu
int csnappy_batch_compress_fragments(const void *d_in, const uint64_t *d_in_off,
				     uint64_t in_stride, const uint32_t *d_in_len,
				     uint32_t uniform_in_len, uint32_t n_blocks,
				     void *d_out, uint64_t out_stride,
				     uint32_t *d_out_len,
				     int workmem_bytes_power_of_two, uint32_t flags,
				     void *stream);

/*
 * Batched csnappy_decompress_noheader (csnappy_decompress.c:319-387), or
 * csnappy_decompress with CSNAPPY_BATCH_WITH_HEADER.
 *   d_out_cap == NULL => every block has capacity uniform_out_cap.
 *   d_status[i]       <- 0 / -1 / -2 / -3 / -5
 *   d_out_len[i]      <- bytes produced when d_status[i] == 0, else 0.
 */
int csnappy_batch_decompress(const void *d_in, const uint64_t *d_in_off,
			     uint64_t in_stride, const uint32_t *d_in_len,
			     uint32_t n_blocks, void *d_out, uint64_t out_stride,
			     const uint32_t *d_out_cap, uint32_t uniform_out_cap,
			     uint32_t *d_out_len, int32_t *d_status, uint32_t flags,
			     void *stream);

/*
 * Batched csnappy_compress (csnappy_compress.c:621-656): n_buffers WHOLE buffers, each framed exactly like one
 * csnappy_compress() call -- varint32 length, one fragment per 32 KiB chunk, the short last chunk with the
 * reference's smaller-table rule (:638-646) -- in one call: all fragments of all buffers are compressed by one
 * launch, then headers and fragments are packed into each buffer's output slot.
 *   buffer i        d_in + (h_in_off ? h_in_off[i] : i * in_stride), h_in_len[i] bytes (NULL: uniform_in_len)
 *   output i        d_out + i * out_stride, d_out_len[i] <- its length;
 *                   out_stride >= 5 + n + n/6 + 32 * ceil(n / 32768) for the longest buffer
 * The lengths (and offsets) are HOST arrays: the fragment table is laid out on the host.  d_workspace must hold
 * csnappy_batch_compress_workspace(...) bytes (fragment slots, sizes, tables) and stay untouched until the
 * work on `stream` has finished.
 */
uint64_t csnappy_batch_compress_workspace(const uint32_t *h_in_len, uint32_t uniform_in_len, uint32_t n_buffers);
int csnappy_batch_compress(const void *d_in, const uint64_t *h_in_off, uint64_t in_stride,
			   const uint32_t *h_in_len, uint32_t uniform_in_len, uint32_t n_buffers,
			   void *d_out, uint64_t out_stride, uint32_t *d_out_len,
			   int workmem_bytes_power_of_two, void *d_workspace,
			   uint64_t workspace_bytes, void *stream);

/*
 * ONE long raw stream, device resident (csnappy_decompress_noheader semantics, csnappy_decompress.c:319-387):
 * tag starts by speculative parsing + pointer jumping, back-references by pointer jumping over the output
 * (stream_kernel.cu) instead of a serial tag walk.  This is what the host-pointer csnappy_decompress /
 * csnappy_decompress_noheader use for streams above 64 KiB.  d_workspace: csnappy_stream_decompress_workspace()
 * bytes (8 per input byte + 4 per output byte).  *d_status <- 0 / -3 / -5, *d_out_len <- bytes produced (0 on error).
 */
uint64_t csnappy_stream_decompress_workspace(uint32_t src_len, uint32_t out_cap);
int csnappy_stream_decompress(const void *d_src, uint32_t src_len, void *d_dst, uint32_t out_cap,
			      uint32_t *d_out_len, int32_t *d_status, void *d_workspace,
			      uint64_t workspace_bytes, void *stream);

/*
 * Exclusive scan of d_len[0..n) into d_off[0..n] (d_off[n] = total) and
 * gather of the strided slots into one contiguous payload:
 *     d_packed[d_off[i] .. d_off[i]+d_len[i]) = d_slots[i*slot_stride ..)
 * This is the size-gather + prefix-sum index of block_compressor.c:298-335 and
 * the fragment concatenation of csnappy_compress.c:647-653, done on the device.
 * d_packed may be NULL to compute offsets only.
 */
int csnappy_batch_pack(const void *d_slots, uint64_t slot_stride,
		       const uint32_t *d_len, uint32_t n_blocks, void *d_packed,
		       uint64_t *d_off, void *stream);

/*
 * Host-buffer variants: same semantics, HOST pointers, synchronous.  Pages are
 * streamed through the device in chunks on several CUDA streams so that H2D,
 * kernels and D2H overlap.  These are what a zram / block_compressor style
 * caller with host memory uses.
 *
 * Bytes of the caller's memory these calls touch: block i is read from
 * h_in + i * in_stride for its own length only (uniform_in_len / h_in_len[i]),
 * so h_in needs (n_blocks - 1) * in_stride + the last block's length bytes.
 * Of output slot i only the first csnappy_max_compressed_length(uniform_in_len)
 * (compress) or uniform_out_cap (decompress) bytes are written: whatever the
 * caller keeps in the rest of each slot, and after the last slot's bound,
 * stays as it was.  Inside that bound, bytes past h_out_len[i] (and all of a
 * slot whose block failed to decode) have unspecified values.
 */
int csnappy_batch_compress_fragments_host(const void *h_in, uint64_t in_stride,
					  uint32_t uniform_in_len, uint32_t n_blocks,
					  void *h_out, uint64_t out_stride,
					  uint32_t *h_out_len,
					  int workmem_bytes_power_of_two);

int csnappy_batch_decompress_host(const void *h_in, uint64_t in_stride,
				  const uint32_t *h_in_len, uint32_t n_blocks,
				  void *h_out, uint64_t out_stride,
				  uint32_t uniform_out_cap, uint32_t *h_out_len,
				  int32_t *h_status, uint32_t flags);

/*
 * block_compressor-style page container on HOST buffers (reference block_compressor.c:275-394):
 *     [u32 nr_pages][u32 clen[nr_pages]][payload_0]...[payload_{nr_pages-1}]
 * payload_i = csnappy_compress_fragment(page_i, wm), or the page itself when that is not smaller
 * (clen_i = page length, :316-318); a reader takes clen_i == page_size as "stored" (:378) -- the
 * reference's wart that a stored PARTIAL last page is not recognised is reproduced, not fixed.
 * The bytes written are identical to what block_compressor's writer loop produces with csnappy
 * and WMSIZE_ORDER = workmem_bytes_power_of_two (:99).  Chunks of pages are pipelined through the
 * device (H2D / kernels / D2H overlap); only compressed bytes cross the bus on the compressed side.
 *
 * csnappy_bc_compress_host    container_capacity >= csnappy_bc_max_container_length(); returns 0,
 *                             CSNAPPY_E_DEVICE or CSNAPPY_E_BAD_ARG.
 * csnappy_bc_decompress_host  out_capacity >= nr_pages * page_size (CSNAPPY_E_OUTPUT_INSUF else);
 *                             returns 0 or the code of the first failing page (its index goes to
 *                             *failed_page when given); *out_length = bytes produced.
 *                             The index is scanned first: the first entry above
 *                             csnappy_max_compressed_length(page_size), or whose payload runs past
 *                             container_length, fails its page with CSNAPPY_E_DATA_MALFORMED and ends
 *                             the decodable prefix.  Every page of that prefix is decoded, those after
 *                             a failing page too; *out_length sums what the prefix's successful pages
 *                             produced.  Page i goes to h_out + i * page_size; the bytes of a failed
 *                             page are unspecified, pages past the prefix are not written.
 */
uint64_t csnappy_bc_max_container_length(uint64_t input_length, uint32_t page_size);
int csnappy_bc_compress_host(const void *h_in, uint64_t input_length, uint32_t page_size,
			     void *h_container, uint64_t container_capacity,
			     uint64_t *container_length, int workmem_bytes_power_of_two);
int csnappy_bc_decompress_host(const void *h_container, uint64_t container_length,
			       uint32_t page_size, void *h_out, uint64_t out_capacity,
			       uint64_t *out_length, uint32_t *failed_page);

/*
 * The same container over SEVERAL devices from one process (SURVEY.md 8e: static sharding, per-device streams,
 * the host gathers the u32 size arrays and prefix-sums them into one container): the page range is cut into chunks,
 * chunk c is handled by devices[c mod n_devices] on that device's own worker thread and streams; there is no
 * data-path collective -- the only thing that crosses devices is the running payload position (8 bytes per chunk).
 * devices == NULL: devices 0 .. n_devices-1; n_devices == 0: every visible device.  The bytes produced are
 * identical to the single-device call.  The caller's current device is not changed.
 */
int csnappy_bc_compress_host_multi(const void *h_in, uint64_t input_length, uint32_t page_size,
				   void *h_container, uint64_t container_capacity,
				   uint64_t *container_length, int workmem_bytes_power_of_two,
				   const int *devices, int n_devices);
int csnappy_bc_decompress_host_multi(const void *h_container, uint64_t container_length,
				     uint32_t page_size, void *h_out, uint64_t out_capacity,
				     uint64_t *out_length, uint32_t *failed_page,
				     const int *devices, int n_devices);

/*
 * The same container on DEVICE buffers of the current device, asynchronous on `stream`: pages that already live in
 * device memory are written into a container there, and a container in device memory (copied there with one
 * cudaMemcpyAsync, or kept there compressed) is read there -- whole, or a batch of chosen pages.  Only the readers
 * synchronise, once, to read the 4-byte page count; the launch count grows with neither the page count nor the
 * number of requests.  Workspaces stay untouched until the work on `stream` has finished.  Every call returns 0,
 * CSNAPPY_E_DEVICE or CSNAPPY_E_BAD_ARG (csnappy_bc_index also CSNAPPY_E_DATA_MALFORMED); a refused argument (page_size
 * outside 1..32768, wm outside 9..16, more than 2^32 - 1 pages, a capacity below the bound, a short workspace, a NULL
 * buffer) returns CSNAPPY_E_BAD_ARG before any device work.  Workspace functions return UINT64_MAX beyond the limits.
 *
 * csnappy_bc_compress        d_container[0, *d_container_length) <- exactly the bytes csnappy_bc_compress_host writes
 *                            for (input, page_size, wm); d_in and d_container at any byte alignment; nothing is written
 *                            at or past *d_container_length.  container_capacity >= csnappy_bc_max_container_length().
 *                            Workspace: a fragment slot per page (csnappy_max_compressed_length(page_size) rounded up
 *                            to 16) plus 16 bytes per page.
 * csnappy_bc_index           *nr_pages <- the page count (written whenever it was read).  A container shorter than
 *                            4 + 4 * nr_pages returns CSNAPPY_E_DATA_MALFORMED; index_entries < nr_pages returns
 *                            CSNAPPY_E_BAD_ARG (index_entries 0 and d_index NULL ask for the count alone).  Else
 *                            d_index[i] <- byte offset of page i's payload from the container start, by the index scan
 *                            of csnappy_bc_decompress_host: the first entry above csnappy_max_compressed_length(
 *                            page_size), or whose payload runs past container_length, and every entry behind it get
 *                            CSNAPPY_BC_NO_PAGE.  No workspace: d_index is the scan's only memory.
 * csnappy_bc_decompress_pages  request k decodes page d_pages[k] into d_out + k * out_stride (out_stride >=
 *                            page_size), with d_index / nr_pages from csnappy_bc_index of the same container:
 *                              d_status[k] 0, d_out_len[k] = bytes produced;
 *                              or the page's decode result (what the whole-container reader reports for that page);
 *                              or CSNAPPY_E_DATA_MALFORMED for a page whose entry is CSNAPPY_BC_NO_PAGE (or does not
 *                              fit container_length);
 *                              or CSNAPPY_E_BAD_ARG for a page number >= nr_pages; d_out_len[k] = 0 on failure.
 *                            A page whose clen equals page_size is copied (a stored short last page is decoded, as in
 *                            the host reader).  Requests may repeat and come in any order; n_requests == 0 is a no-op.
 *                            Nothing outside [k * out_stride, k * out_stride + page_size) is written; bytes of a
 *                            failed request are unspecified.  Workspace: 16 bytes per request + 1 KiB.
 * csnappy_bc_decompress      *d_status, *d_out_length and *d_failed_page <- what csnappy_bc_decompress_host returns
 *                            and writes for the same bytes (*d_out_length is 0 for the header results -5 / -2;
 *                            *d_failed_page is written only on a page failure; it may be NULL).  Page i goes to
 *                            d_out + i * page_size.  Workspace: 20 bytes per page for the most pages the container
 *                            and out_capacity can hold.
 */
#define CSNAPPY_BC_NO_PAGE UINT64_MAX
uint64_t csnappy_bc_compress_workspace(uint64_t input_length, uint32_t page_size);
int csnappy_bc_compress(const void *d_in, uint64_t input_length, uint32_t page_size, void *d_container,
			uint64_t container_capacity, uint64_t *d_container_length, int workmem_bytes_power_of_two,
			void *d_workspace, uint64_t workspace_bytes, void *stream);
int csnappy_bc_index(const void *d_container, uint64_t container_length, uint32_t page_size, uint64_t *d_index,
		     uint64_t index_entries, uint32_t *nr_pages, void *stream);
uint64_t csnappy_bc_decompress_pages_workspace(uint32_t n_requests);
int csnappy_bc_decompress_pages(const void *d_container, uint64_t container_length, uint32_t page_size,
				const uint64_t *d_index, uint32_t nr_pages, const uint32_t *d_pages, uint32_t n_requests,
				void *d_out, uint64_t out_stride, uint32_t *d_out_len, int32_t *d_status,
				void *d_workspace, uint64_t workspace_bytes, void *stream);
uint64_t csnappy_bc_decompress_workspace(uint64_t container_length, uint32_t page_size, uint64_t out_capacity);
int csnappy_bc_decompress(const void *d_container, uint64_t container_length, uint32_t page_size, void *d_out,
			  uint64_t out_capacity, uint64_t *d_out_length, int32_t *d_status, uint32_t *d_failed_page,
			  void *d_workspace, uint64_t workspace_bytes, void *stream);

/*
 * Snappy FRAMING FORMAT (the format of .sz files and x-snappy-framed streams): one buffer as a stream of chunks
 *     [u8 type][u24 LE length][length bytes]
 * Every data chunk holds at most 65536 uncompressed bytes and a masked CRC-32C of them, so both directions run
 * chunk-parallel on the device and corruption is detected.
 *
 * CRC-32C: Castagnoli polynomial, reflected (0x82F63B78), init ~0, final xor ~0.
 * mask(crc) = ((crc >> 15) | (crc << 17)) + 0xa282ead8  (mod 2^32).
 *
 * Writer (csnappy_framed_compress*): the output is fully determined by (input, wm):
 *   ff 06 00 00 73 4e 61 50 70 59   stream identifier, once, also for empty input; then for chunk k of the input
 *   (65536 bytes each, the last one shorter), n_k bytes, c = csnappy_compress(chunk_k, wm) (varint included):
 *     type 0x00, body [mask(crc32c(chunk_k)) LE][c]        if len(c) < n_k - n_k / 8
 *     type 0x01, body [mask(crc32c(chunk_k)) LE][chunk_k]  otherwise.
 *   csnappy_framed_max_length(n) = 10 + 8 * ceil(n / 65536) + n is an exact bound.
 *
 * Reader (csnappy_framed_decompress*): walks the chunks from byte 0.
 *   Zero-length input is an empty stream: 0, no bytes.
 *   Fewer than 4 header bytes left, or a body running past the end: CSNAPPY_E_DATA_MALFORMED at that chunk.
 *   The first chunk must be a stream identifier; every 0xff chunk, wherever it appears, must be exactly length 6
 *   with body "sNaPpY" (concatenated streams are valid).
 *   0x00 compressed: body >= 5 bytes; the varint32 must be valid and <= 65536; the rest must decode
 *        (csnappy_decompress_noheader semantics, capacity = the varint) to exactly the varint's length.
 *   0x01 uncompressed: body >= 4 bytes and at most 65536 data bytes.
 *   0x02..0x7f (reserved, unskippable): CSNAPPY_E_DATA_MALFORMED.
 *   0x80..0xfd (reserved, skippable) and 0xfe (padding), any length: skipped.
 *   Anything else wrong with a data chunk: CSNAPPY_E_DATA_MALFORMED.
 *   A data chunk whose output would end past out_capacity: CSNAPPY_E_OUTPUT_INSUF.
 *   A data chunk whose uncompressed bytes do not match its stored masked CRC: CSNAPPY_E_CHECKSUM.
 * Of the failing chunks, the one with the smallest header position wins.  Framing, varint and capacity failures end
 * the walk (later chunk boundaries are unknown).  *out_length = the uncompressed bytes of the data chunks before the
 * winning chunk; they are in dst[0, *out_length) and correct.  Bytes in [*out_length, out_capacity) are unspecified;
 * nothing is written at or past out_capacity.  *failed_offset = the winning chunk's header position, written only on
 * a chunk failure (-2, -5, -102); the pointer may be NULL.
 * Returns 0, CSNAPPY_E_OUTPUT_INSUF, CSNAPPY_E_DATA_MALFORMED, CSNAPPY_E_CHECKSUM, CSNAPPY_E_DEVICE or
 * CSNAPPY_E_BAD_ARG; a refused argument (wm outside 9..16, a capacity below the bound, a short workspace, a NULL
 * buffer) returns CSNAPPY_E_BAD_ARG before any device work.
 */
#define CSNAPPY_E_CHECKSUM (-102)
uint64_t csnappy_framed_max_length(uint64_t input_length);

/* Device resident, asynchronous on `stream`.  *d_out_length <- stream length.  out_capacity >=
 * csnappy_framed_max_length(input_length); d_workspace: csnappy_framed_compress_workspace() bytes, untouched until
 * the work on `stream` has finished.  Returns 0, CSNAPPY_E_DEVICE or CSNAPPY_E_BAD_ARG. */
uint64_t csnappy_framed_compress_workspace(uint64_t input_length);
int csnappy_framed_compress(const void *d_in, uint64_t input_length, void *d_out, uint64_t out_capacity,
			    uint64_t *d_out_length, int workmem_bytes_power_of_two,
			    void *d_workspace, uint64_t workspace_bytes, void *stream);

/* Device resident.  *d_status <- the reader's result (0, -2, -5, -102), *d_out_length and *d_failed_offset as above.
 * The chunk walk runs first and its chunk counts are read back (the call synchronises with `stream` once); the call
 * returns with decoding and verification enqueued on `stream`.  d_workspace: csnappy_framed_decompress_workspace()
 * bytes (about 7.5 per byte of src: the chunk tables for the most chunks src_length can hold).  The return value is
 * 0, CSNAPPY_E_DEVICE or CSNAPPY_E_BAD_ARG. */
uint64_t csnappy_framed_decompress_workspace(uint64_t src_length);
int csnappy_framed_decompress(const void *d_src, uint64_t src_length, void *d_dst, uint64_t out_capacity,
			      uint64_t *d_out_length, int32_t *d_status, uint64_t *d_failed_offset,
			      void *d_workspace, uint64_t workspace_bytes, void *stream);

/* Host buffers, synchronous.  The whole input and output are staged through the device in one piece (no H2D /
 * kernel / D2H overlap), and only the valid prefix dst[0, *out_length) is copied back. */
int csnappy_framed_compress_host(const void *h_in, uint64_t input_length, void *h_out, uint64_t out_capacity,
				 uint64_t *out_length, int workmem_bytes_power_of_two);
int csnappy_framed_decompress_host(const void *h_src, uint64_t src_length, void *h_dst, uint64_t out_capacity,
				   uint64_t *out_length, uint64_t *failed_offset);

/*
 * MANY framed streams in one call, device resident, asynchronous on `stream`.  A batch call means exactly n_streams
 * independent single calls: every result below is what csnappy_framed_compress / csnappy_framed_decompress returns
 * for that stream alone, and one stream's content never affects another stream's result.  Stream i is
 * d_in + h_in_off[i] (d_src + h_src_off[i]), h_in_len[i] (h_src_len[i]) bytes, any byte offset.  The offsets, lengths
 * and capacities are HOST arrays: the host lays out the chunk tables and sizes the launches.  The launch count does
 * not grow with n_streams.
 *
 * Writer (csnappy_framed_batch_compress):
 *   output slot i is d_out + h_out_off[i]; h_out_off == NULL: slot i starts at the sum of
 *   csnappy_framed_max_length(h_in_len[j]) for j < i.  Every slot [start, start + csnappy_framed_max_length(h_in_len[i]))
 *   must end at or before out_capacity (else CSNAPPY_E_BAD_ARG); slots must not overlap (not checked).
 *   Slot i receives exactly the bytes csnappy_framed_compress(stream i, wm) writes, d_out_len[i] <- that length (an
 *   empty stream: the 10-byte identifier only).  Bytes outside [slot i, slot i + d_out_len[i]) are not written.
 * Reader (csnappy_framed_batch_decompress):
 *   d_status[i], d_out_len[i], d_failed_offset[i] and d_dst[h_dst_off[i], + d_out_len[i]) are exactly what
 *   csnappy_framed_decompress returns for stream i with out_capacity h_dst_cap[i] (0 / -2 / -5 / -102, which failing
 *   chunk wins, the valid prefix).  d_failed_offset[i] is measured from the start of stream i and written only when
 *   stream i fails; d_failed_offset may be NULL.  Nothing is written at or past h_dst_off[i] + h_dst_cap[i].  The
 *   call synchronises with `stream` once (the chunk totals of the batch size the launches), whatever n_streams is.
 * Decompressed length (csnappy_framed_batch_decompressed_length): a framed stream does not carry its total length.
 *   d_length[i] <- the sum of the data lengths its chunk headers declare (the varint of a 0x00 chunk, the body length
 *   minus 4 of a 0x01 chunk) up to the first failure the chunk walk can detect; d_status[i] <- -5 if there is such a
 *   failure, else 0.  Decoding stream i with capacity d_length[i] never returns CSNAPPY_E_OUTPUT_INSUF.  No workspace
 *   and no synchronisation: the 16 bytes per stream of offsets and lengths go to a stream-ordered allocation
 *   (cudaMallocAsync / cudaFreeAsync on `stream`, from the device's default memory pool) for the duration of the walk.
 * Limits: per stream those of the single calls (input at most (2^32 - 2) * 32768 bytes, source at most 2^35 bytes);
 *   per batch the fragments of the writer and the chunk table entries of the reader (sum of h_src_len[i] / 8 + 1) each
 *   at most 2^32 - 1.  The workspace functions return UINT64_MAX for a batch beyond them.
 * Returns 0 (n_streams == 0 included), CSNAPPY_E_DEVICE or CSNAPPY_E_BAD_ARG for the call as a whole; a refused
 * argument (wm outside 9..16, a stream or batch beyond the limits, a slot past out_capacity, a short workspace, a NULL
 * buffer) returns CSNAPPY_E_BAD_ARG before any device work.  d_workspace stays untouched until the work on `stream`
 * has finished.
 */
uint64_t csnappy_framed_batch_compress_workspace(const uint64_t *h_in_len, uint32_t n_streams);
int csnappy_framed_batch_compress(const void *d_in, const uint64_t *h_in_off, const uint64_t *h_in_len,
				  uint32_t n_streams, void *d_out, const uint64_t *h_out_off,
				  uint64_t out_capacity, uint64_t *d_out_len, int workmem_bytes_power_of_two,
				  void *d_workspace, uint64_t workspace_bytes, void *stream);
uint64_t csnappy_framed_batch_decompress_workspace(const uint64_t *h_src_len, uint32_t n_streams);
int csnappy_framed_batch_decompress(const void *d_src, const uint64_t *h_src_off, const uint64_t *h_src_len,
				    uint32_t n_streams, void *d_dst, const uint64_t *h_dst_off,
				    const uint64_t *h_dst_cap, uint64_t *d_out_len, int32_t *d_status,
				    uint64_t *d_failed_offset, void *d_workspace, uint64_t workspace_bytes,
				    void *stream);
int csnappy_framed_batch_decompressed_length(const void *d_src, const uint64_t *h_src_off,
					     const uint64_t *h_src_len, uint32_t n_streams,
					     uint64_t *d_length, int32_t *d_status, void *stream);

/* Masked CRC-32C of each 65536-byte chunk of d_in[0, length) (the last one shorter) -> d_crc[ceil(length / 65536)];
 * the framing format's checksum, on the device, asynchronous on `stream`. */
int csnappy_framed_crc32c(const void *d_in, uint64_t length, uint32_t *d_crc, void *stream);

/*
 * Library / device introspection and kernel tuning knobs (used by bench.py and
 * the tests; not needed by drop-in callers).
 */
int csnappy_b200_device_ok(void);	   /* 1 if a CUDA device is usable */
int csnappy_b200_device_count(void);	   /* visible CUDA devices (0 on error) */
const char *csnappy_b200_last_error(void); /* text of the last device error (thread local) */
uint64_t csnappy_b200_kernel_launches(void); /* kernels launched by this library so far */
/* key (value 0 restores the default; returns 0 or CSNAPPY_E_BAD_ARG):
 *   "compress_lanes" | "decompress_lanes"  lanes cooperating on one block in the warp-per-block kernels: 8 / 16 / 32
 *   "compress_stage_input"    1: always stage blocks in shared memory; 2: read them from global memory (32-lane
 *                             groups only; the default for large batches of fragments above ~14 KB)
 *   "decompress_stage_input"  1: always stage blocks in shared memory; 2: stage only the output and read the
 *                             compressed block through L1; 3: decode against global memory, a warp per block;
 *                             4: one lane per block (the default for very large batches; it needs 16-byte
 *                             aligned output slots, other layouts keep the default routing)
 *   "decompress_lane_warps"   lane-per-block decoder: warps of 32 blocks in flight per SM (default 32)
 *   "decompress_smem_kb"      shared memory per SM in mode 2
 *   "ctas_per_sm"             resident CTAs per SM of the warp-per-block kernels
 *   "stream_decode_min"       bytes from which ONE single stream takes the parallel stream decoder; -1: never
 *   "copy_threads"            helper threads that stage PAGEABLE caller memory through pinned buffers in the
 *                             host-buffer pipelines (read when the pool starts; default 7 on >= 16 cores)
 *   "chunk_mb"                MiB per chunk of the host-buffer pipelines (default 32; measured flat from 32 to 128)
 *   "no_bounce"               1: hand pageable caller memory straight to cudaMemcpyAsync (round-1 behaviour)
 *   "host_register"           1: page-lock the caller's buffers for the duration of a host-buffer call (measured
 *                             slower than the staging above unless the same buffers are registered once by the caller) */
int csnappy_b200_set_tuning(const char *key, int value);

#ifdef __cplusplus
}
#endif
#endif /* CSNAPPY_B200_CSNAPPY_BATCH_H_ */
