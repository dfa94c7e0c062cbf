/*
 * csnappy_shim.c -- plain-C host side of libcsnappy_b200.so.
 *
 * Exports (a) the six drop-in symbols of the reference's csnappy.h
 * (/root/reference/csnappy.h:30-119) on HOST pointers and (b) the batched entry
 * points of include/csnappy_batch.h.  This file contains no codec: it does
 * argument checks, the varint32 framing (csnappy_compress.c:46-73,
 * csnappy_decompress.c:45-71), buffer staging and CUDA launches.  Every byte
 * of compressed or decompressed payload is produced by the sm_100a kernels in
 * compress_kernel.cu / decompress_kernel.cu / decompress_lane_kernel.cu /
 * stream_kernel.cu.  There is no CPU fallback: without a usable device the
 * decompress calls return CSNAPPY_E_DEVICE and the compress calls (no error
 * channel in the reference ABI) abort loudly.
 *
 * Concurrency: like the reference (csnappy.h:46-72: re-entrant, callers may run
 * concurrently on disjoint buffers) every host-pointer call takes a private
 * staging CONTEXT (streams + device / pinned buffers) from a per-device pool, so
 * concurrent callers overlap on the device instead of queueing behind one lock.
 * The *_multi entry points shard one host buffer over several devices from ONE
 * process: a worker thread and a context per device, no data-path collective; the
 * only cross-device state is the running payload position of the container.
 */
#include <cuda_runtime_api.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include "../../include/csnappy.h"
#include "../../include/csnappy_batch.h"
#include "kernels.h"

#define SLOT_STRIDE_32K 38272u /* csnappy_max_compressed_length(32768) = 38261, rounded up to 16 */
#define HDR 16u		       /* device staging: [u32 out_len][i32 status][pad] then payload */
#define SMALL_CALL 65536u      /* single calls up to this size take the one-synchronisation path */
#define PIPE 4		       /* chunks in flight per device in the host-buffer pipelines */
#define MAX_DEV 64

static __thread char tls_err[256];

static int set_err(const char *what, int cuda_err)
{
	snprintf(tls_err, sizeof(tls_err), "csnappy_b200: %s: %s", what,
		 cuda_err > 0 ? cudaGetErrorString((cudaError_t)cuda_err) : "invalid argument");
	return cuda_err > 0 ? CSNAPPY_E_DEVICE : CSNAPPY_E_BAD_ARG;
}

const char *csnappy_b200_last_error(void) { return tls_err; }

int csnappy_b200_device_count(void)
{
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess) {
		set_err("cudaGetDeviceCount", (int)e);
		cudaGetLastError();
		return 0;
	}
	return n;
}

int csnappy_b200_device_ok(void) { return csnappy_b200_device_count() > 0; }

uint64_t csnappy_b200_kernel_launches(void) { return csb_launch_count(); }

/* ---- tuning knobs ------------------------------------------------------- */
static int g_compress_lanes, g_decompress_lanes, g_ctas_per_sm, g_stage_input, g_smem_kb, g_host_register, g_stream_min, g_lane_warps, g_copy_threads, g_no_bounce, g_compress_stage, g_chunk_mb;

int csnappy_b200_set_tuning(const char *key, int value)
{
	if (!key)
		return CSNAPPY_E_BAD_ARG;
	if (!strcmp(key, "compress_lanes") || !strcmp(key, "decompress_lanes")) {
		if (value != 0 && value != 8 && value != 16 && value != 32)
			return CSNAPPY_E_BAD_ARG;
		if (key[0] == 'c')
			g_compress_lanes = value;
		else
			g_decompress_lanes = value;
		return 0;
	}
	if (!strcmp(key, "compress_stage_input")) { /* 0: choose; 1: always stage blocks in shared memory; 2: never */
		if (value < 0 || value > 2)
			return CSNAPPY_E_BAD_ARG;
		g_compress_stage = value;
		return 0;
	}
	if (!strcmp(key, "decompress_stage_input")) {
		if (value < 0 || value > 4)
			return CSNAPPY_E_BAD_ARG;
		g_stage_input = value;
		return 0;
	}
	if (!strcmp(key, "decompress_smem_kb")) {
		if (value < 0 || value > 227)
			return CSNAPPY_E_BAD_ARG;
		g_smem_kb = value;
		return 0;
	}
	if (!strcmp(key, "decompress_lane_warps")) { /* blocks in flight per SM of the lane-per-block decoder, in warps of 32 */
		if (value < 0 || value > 64)
			return CSNAPPY_E_BAD_ARG;
		g_lane_warps = value;
		return 0;
	}
	if (!strcmp(key, "chunk_mb")) { /* MiB per chunk of the host-buffer pipelines (0 = default 32) */
		if (value < 0 || value > 1024)
			return CSNAPPY_E_BAD_ARG;
		g_chunk_mb = value;
		return 0;
	}
	if (!strcmp(key, "copy_threads")) { /* helper threads staging pageable caller memory (0 = default; read when the pool starts) */
		if (value < 0 || value > 64)
			return CSNAPPY_E_BAD_ARG;
		g_copy_threads = value;
		return 0;
	}
	if (!strcmp(key, "no_bounce")) { /* 1: hand pageable caller memory straight to cudaMemcpyAsync (the round-1 behaviour) */
		if (value < 0 || value > 1)
			return CSNAPPY_E_BAD_ARG;
		g_no_bounce = value;
		return 0;
	}
	if (!strcmp(key, "ctas_per_sm")) {
		if (value < 0 || value > 8)
			return CSNAPPY_E_BAD_ARG;
		g_ctas_per_sm = value;
		return 0;
	}
	if (!strcmp(key, "host_register")) { /* 1: page-lock the caller's buffers for the duration of a host-buffer call */
		if (value < 0 || value > 1)
			return CSNAPPY_E_BAD_ARG;
		g_host_register = value;
		return 0;
	}
	if (!strcmp(key, "stream_decode_min")) { /* single streams at least this long (bytes) use the parallel stream decoder; 0 = default, -1 = never */
		g_stream_min = value;
		return 0;
	}
	return CSNAPPY_E_BAD_ARG;
}

/* ---- pure host arithmetic ---------------------------------------------- */
uint32_t csnappy_max_compressed_length(uint32_t source_len) { return 32u + source_len + source_len / 6u; }

int csnappy_get_uncompressed_length(const char *start, uint32_t n, uint32_t *result)
{
	const uint8_t *p = (const uint8_t *)start;
	uint32_t used = 0, shift = 0;
	*result = 0;
	for (;;) {
		uint8_t c;
		if (shift >= 32 || used == n)
			return CSNAPPY_E_HEADER_BAD;
		c = p[used++];
		*result |= (uint32_t)(c & 0x7f) << shift;
		if (c < 128)
			return (int)used;
		shift += 7;
	}
}

static uint32_t put_varint32(uint8_t *out, uint32_t v)
{
	uint32_t k = 0;
	while (v >= 128) {
		out[k++] = (uint8_t)(v | 0x80);
		v >>= 7;
	}
	out[k++] = (uint8_t)v;
	return k;
}

static void fill_compress_args(struct csb_compress_args *a)
{
	memset(a, 0, sizeof(*a));
	a->lanes = g_compress_lanes;
	a->ctas_per_sm = g_ctas_per_sm;
	a->stage_input = g_compress_stage;
}

static void fill_decompress_args(struct csb_decompress_args *a)
{
	memset(a, 0, sizeof(*a));
	a->lanes = g_decompress_lanes;
	a->stage_input = g_stage_input;
	a->smem_kb = g_smem_kb;
	a->ctas_per_sm = g_ctas_per_sm;
	a->lane_warps = g_lane_warps;
}

/* ---- batched device-pointer entry points -------------------------------- */
int csnappy_batch_compress_fragments(const void *d_in, const uint64_t *d_in_off, uint64_t in_stride,
				     const uint32_t *d_in_len, uint32_t uniform_in_len, uint32_t n_blocks,
				     void *d_out, uint64_t out_stride, uint32_t *d_out_len,
				     int workmem_bytes_power_of_two, uint32_t flags, void *stream)
{
	struct csb_compress_args a;
	int e;
	if (workmem_bytes_power_of_two < 9 || workmem_bytes_power_of_two > 16)
		return set_err("workmem_bytes_power_of_two outside 9..16", 0);
	if (!d_in_len && uniform_in_len > CSB_FRAGMENT_MAX)
		return set_err("fragment longer than 32768 bytes", 0);
	if (n_blocks && (!d_in || !d_out || !d_out_len))
		return set_err("null buffer", 0);
	fill_compress_args(&a);
	a.in = (const uint8_t *)d_in;
	a.in_off = d_in_off;
	a.in_stride = in_stride;
	a.in_len = d_in_len;
	a.uniform_len = uniform_in_len;
	a.n_blocks = n_blocks;
	a.out = (uint8_t *)d_out;
	a.out_stride = out_stride;
	a.out_len = d_out_len;
	a.wm = workmem_bytes_power_of_two;
	a.flags = flags;
	e = csb_launch_compress(&a, (csb_stream_t)stream);
	return e ? set_err("compress launch", e) : 0;
}

int csnappy_batch_decompress(const void *d_in, const uint64_t *d_in_off, uint64_t in_stride,
			     const uint32_t *d_in_len, uint32_t n_blocks, void *d_out, uint64_t out_stride,
			     const uint32_t *d_out_cap, uint32_t uniform_out_cap, uint32_t *d_out_len,
			     int32_t *d_status, uint32_t flags, void *stream)
{
	struct csb_decompress_args a;
	int e;
	if (n_blocks && (!d_in || !d_in_len || !d_out_len || !d_status))
		return set_err("null buffer", 0);
	fill_decompress_args(&a);
	a.in = (const uint8_t *)d_in;
	a.in_off = d_in_off;
	a.in_stride = in_stride;
	a.in_len = d_in_len;
	a.n_blocks = n_blocks;
	a.out = (uint8_t *)d_out;
	a.out_stride = out_stride;
	a.out_cap = d_out_cap;
	a.uniform_cap = uniform_out_cap;
	a.out_len = d_out_len;
	a.status = d_status;
	a.flags = flags;
	e = csb_launch_decompress(&a, (csb_stream_t)stream);
	return e ? set_err("decompress launch", e) : 0;
}

int csnappy_batch_pack(const void *d_slots, uint64_t slot_stride, const uint32_t *d_len, uint32_t n_blocks,
		       void *d_packed, uint64_t *d_off, void *stream)
{
	int e;
	if (!d_off || (n_blocks && (!d_len || (d_packed && !d_slots))))
		return set_err("null buffer", 0);
	e = csb_launch_pack((const uint8_t *)d_slots, slot_stride, d_len, n_blocks, (uint8_t *)d_packed, d_off,
			    (csb_stream_t)stream);
	return e ? set_err("pack launch", e) : 0;
}

/* ---- batched csnappy_compress: many whole buffers, each framed, in one call ------------------------------
 * (csnappy_compress.c:621-656 per buffer: varint32, 32 KiB fragments, short-last-chunk table rule.)
 * The fragment table is laid out on the host from the buffer lengths, so the lengths are needed there.
 * Workspace (device): fragment slots | sizes | scan | fragment table | buffer table.                          */
static uint64_t frags_of(uint32_t len) { return ((uint64_t)len + CSB_FRAGMENT_MAX - 1) / CSB_FRAGMENT_MAX; }

static uint64_t al256(uint64_t x) { return (x + 255) & ~(uint64_t)255; }

static uint64_t batch_compress_layout(uint64_t F, uint64_t n, uint64_t *o_len, uint64_t *o_off, uint64_t *o_foff,
				      uint64_t *o_flen, uint64_t *o_fbuf, uint64_t *o_bfirst, uint64_t *o_blen)
{
	uint64_t p = al256(F * SLOT_STRIDE_32K);
	*o_len = p;
	p = al256(p + F * 4);
	*o_off = p;
	p = al256(p + (F + 1) * 8);
	*o_foff = p;
	p = al256(p + F * 8);
	*o_flen = p;
	p = al256(p + F * 4);
	*o_fbuf = p;
	p = al256(p + F * 4);
	*o_bfirst = p;
	p = al256(p + (n + 1) * 4);
	*o_blen = p;
	p = al256(p + n * 4);
	return p + 256;
}

uint64_t csnappy_batch_compress_workspace(const uint32_t *h_in_len, uint32_t uniform_in_len, uint32_t n_buffers)
{
	uint64_t F = 0, a, b, c, d, e, f, g;
	uint32_t i;
	for (i = 0; i < n_buffers; i++)
		F += frags_of(h_in_len ? h_in_len[i] : uniform_in_len);
	return batch_compress_layout(F, n_buffers, &a, &b, &c, &d, &e, &f, &g);
}

int csnappy_batch_compress(const void *d_in, const uint64_t *h_in_off, uint64_t in_stride, const uint32_t *h_in_len,
			   uint32_t uniform_in_len, uint32_t n_buffers, void *d_out, uint64_t out_stride,
			   uint32_t *d_out_len, int workmem_bytes_power_of_two, void *d_workspace,
			   uint64_t workspace_bytes, void *stream)
{
	uint64_t F = 0, o_len, o_off, o_foff, o_flen, o_fbuf, o_bfirst, o_blen, need, f = 0;
	uint32_t i, max_len = 0;
	uint8_t *ws = (uint8_t *)d_workspace, *tab = NULL;
	struct csb_compress_args a;
	cudaStream_t s = (cudaStream_t)stream;
	int e;
	if (workmem_bytes_power_of_two < 9 || workmem_bytes_power_of_two > 16)
		return set_err("workmem_bytes_power_of_two outside 9..16", 0);
	if (n_buffers == 0)
		return 0;
	if (!d_in || !d_out || !d_out_len || !d_workspace)
		return set_err("null buffer", 0);
	for (i = 0; i < n_buffers; i++) {
		uint32_t n = h_in_len ? h_in_len[i] : uniform_in_len;
		F += frags_of(n);
		if (n > max_len)
			max_len = n;
	}
	if (F > 0xffffffffull)
		return set_err("more than 2^32 fragments", 0);
	if (out_stride < 5ull + max_len + max_len / 6 + 32ull * (frags_of(max_len) ? frags_of(max_len) : 1))
		return set_err("out_stride smaller than the worst case of its buffer (5 + n + n/6 + 32 per fragment)", 0);
	need = batch_compress_layout(F, n_buffers, &o_len, &o_off, &o_foff, &o_flen, &o_fbuf, &o_bfirst, &o_blen);
	if (workspace_bytes < need)
		return set_err("workspace smaller than csnappy_batch_compress_workspace()", 0);
	/* host image of the tables [o_foff, need): fragment offsets / lengths / owners, first fragment and length per buffer */
	tab = (uint8_t *)malloc((size_t)(need - o_foff));
	if (!tab)
		return set_err("host table", (int)cudaErrorMemoryAllocation);
	{
		uint64_t *foff = (uint64_t *)tab;
		uint32_t *flen = (uint32_t *)(tab + (o_flen - o_foff)), *fbuf = (uint32_t *)(tab + (o_fbuf - o_foff));
		uint32_t *bfirst = (uint32_t *)(tab + (o_bfirst - o_foff)), *blen = (uint32_t *)(tab + (o_blen - o_foff));
		for (i = 0; i < n_buffers; i++) {
			uint32_t n = h_in_len ? h_in_len[i] : uniform_in_len, at = 0;
			uint64_t base = h_in_off ? h_in_off[i] : (uint64_t)i * in_stride;
			bfirst[i] = (uint32_t)f;
			blen[i] = n;
			while (at < n) {
				uint32_t m = n - at < CSB_FRAGMENT_MAX ? n - at : CSB_FRAGMENT_MAX;
				foff[f] = base + at;
				flen[f] = m;
				fbuf[f] = i;
				f++;
				at += m;
			}
		}
		bfirst[n_buffers] = (uint32_t)f;
	}
	/* pageable source: the copy is staged before the call returns, the table can be freed right after */
	e = (int)cudaMemcpyAsync(ws + o_foff, tab, (size_t)(need - o_foff), cudaMemcpyHostToDevice, s);
	free(tab);
	if (e)
		return set_err("H2D fragment table", e);
	if (F) {
		fill_compress_args(&a);
		a.in = (const uint8_t *)d_in;
		a.in_off = (const uint64_t *)(ws + o_foff);
		a.in_len = (const uint32_t *)(ws + o_flen);
		a.n_blocks = (uint32_t)F;
		a.out = ws;
		a.out_stride = SLOT_STRIDE_32K;
		a.out_len = (uint32_t *)(ws + o_len);
		a.wm = workmem_bytes_power_of_two;
		a.flags = CSNAPPY_BATCH_SHRINK_TABLE;
		if ((e = csb_launch_compress(&a, (csb_stream_t)s)))
			return set_err("compress launch", e);
	}
	if ((e = csb_launch_scan((const uint32_t *)(ws + o_len), (uint32_t)F, (uint64_t *)(ws + o_off), (csb_stream_t)s)))
		return set_err("scan launch", e);
	e = csb_launch_frame(ws, SLOT_STRIDE_32K, (const uint32_t *)(ws + o_len), (const uint64_t *)(ws + o_off),
			     (const uint32_t *)(ws + o_fbuf), (const uint32_t *)(ws + o_bfirst), (const uint32_t *)(ws + o_blen),
			     (uint32_t)F, n_buffers, (uint8_t *)d_out, out_stride, d_out_len, (csb_stream_t)s);
	return e ? set_err("frame launch", e) : 0;
}

/* ---- one long raw stream, device resident: the parallel stream decoder (stream_kernel.cu) ---------------- */
uint64_t csnappy_stream_decompress_workspace(uint32_t src_len, uint32_t out_cap)
{
	return (uint64_t)csb_stream_aux_bytes(src_len, out_cap, 0) + (uint64_t)csb_stream_aux_bytes(src_len, out_cap, 1);
}

int csnappy_stream_decompress(const void *d_src, uint32_t src_len, void *d_dst, uint32_t out_cap, uint32_t *d_out_len,
			      int32_t *d_status, void *d_workspace, uint64_t workspace_bytes, void *stream)
{
	const size_t t1 = csb_stream_aux_bytes(src_len, out_cap, 0);
	int e;
	if (!d_out_len || !d_status || !d_workspace || (src_len && !d_src) || (out_cap && !d_dst))
		return set_err("null buffer", 0);
	if (workspace_bytes < csnappy_stream_decompress_workspace(src_len, out_cap))
		return set_err("workspace smaller than csnappy_stream_decompress_workspace()", 0);
	e = csb_launch_decompress_stream((const uint8_t *)d_src, src_len, (uint8_t *)d_dst, out_cap, d_out_len, d_status, d_workspace,
					 (uint8_t *)d_workspace + t1, (csb_stream_t)stream);
	if (e == 1) {
		/* empty stream, or no cooperative launch on this device: the serial path of the batched decoder */
		struct csb_decompress_args a;
		uint32_t *d_len = (uint32_t *)d_workspace;
		if ((e = (int)cudaMemcpyAsync(d_len, &src_len, 4, cudaMemcpyHostToDevice, (cudaStream_t)stream)))
			return set_err("H2D len", e);
		fill_decompress_args(&a);
		a.stage_input = 3;
		a.in = (const uint8_t *)d_src;
		a.in_len = d_len;
		a.n_blocks = 1;
		a.out = (uint8_t *)d_dst;
		a.uniform_cap = out_cap;
		a.out_len = d_out_len;
		a.status = d_status;
		a.max_in_len = src_len;
		e = csb_launch_decompress(&a, (csb_stream_t)stream);
	}
	return e ? set_err("stream decoder launch", e) : 0;
}

/* ---- staging contexts for the host-pointer calls ------------------------ */
struct buf {
	void *p;
	size_t cap;
};

struct slot {
	cudaStream_t s;
	cudaEvent_t ev;
	struct buf d_in, d_slots, d_len, d_clen, d_off, d_packed, d_out, d_res, d_ctr;
	struct buf h_res; /* pinned: [u64 total] or [u32 out_len[n]][i32 status[n]] */
	struct buf h_in, h_out, h_idx; /* pinned staging of a chunk when the caller's memory is pageable */
	struct {
		const void *src; /* pinned */
		void *dst;	 /* the caller's pageable memory */
		size_t width, pitch, rows; /* `rows` runs of `width` bytes, `pitch` apart on both sides */
	} pend[3]; /* copies owed to the caller once the slot's queued device-to-host copies have landed */
	int npend;
	uint64_t first;
	uint32_t n;
};

struct ctx {
	struct ctx *next;
	int dev;
	struct slot sl[PIPE];
	struct buf h_pin;	/* pinned bounce buffer of the single small calls */
	struct buf d_aux, d_aux2; /* stream decoder tables */
};

static pthread_mutex_t pool_mu = PTHREAD_MUTEX_INITIALIZER;
static struct ctx *pool_free[MAX_DEV];

static int grow_dev(struct buf *b, size_t need)
{
	int e;
	if (need <= b->cap)
		return 0;
	if (b->p && (e = (int)cudaFree(b->p)))
		return e;
	b->p = NULL;
	b->cap = 0;
	need = (need + (1u << 20)) & ~(size_t)((1u << 20) - 1);
	if ((e = (int)cudaMalloc(&b->p, need))) {
		cudaGetLastError();
		return e;
	}
	b->cap = need;
	return 0;
}

static int grow_pin(struct buf *b, size_t need)
{
	int e;
	if (need <= b->cap)
		return 0;
	if (b->p && (e = (int)cudaFreeHost(b->p)))
		return e;
	b->p = NULL;
	b->cap = 0;
	need = (need + (1u << 16)) & ~(size_t)((1u << 16) - 1);
	if ((e = (int)cudaMallocHost(&b->p, need))) {
		cudaGetLastError();
		return e;
	}
	b->cap = need;
	return 0;
}

static void drop_dev(struct buf *b)
{
	if (b->p)
		cudaFree(b->p);
	b->p = NULL;
	b->cap = 0;
}

/* a context of the CURRENT device: from the pool, or a new one */
static int ctx_acquire(struct ctx **out)
{
	struct ctx *c = NULL;
	int dev = 0, e, i;
	if ((e = (int)cudaGetDevice(&dev)))
		return e;
	if (dev < 0 || dev >= MAX_DEV)
		return (int)cudaErrorInvalidDevice;
	pthread_mutex_lock(&pool_mu);
	c = pool_free[dev];
	if (c)
		pool_free[dev] = c->next;
	pthread_mutex_unlock(&pool_mu);
	if (!c) {
		c = (struct ctx *)calloc(1, sizeof(*c));
		if (!c)
			return (int)cudaErrorMemoryAllocation;
		c->dev = dev;
		for (i = 0; i < PIPE; i++) {
			if ((e = (int)cudaStreamCreateWithFlags(&c->sl[i].s, cudaStreamNonBlocking)) ||
			    (e = (int)cudaEventCreateWithFlags(&c->sl[i].ev, cudaEventDisableTiming))) {
				free(c); /* (streams of a failed init leak; the process is in trouble anyway) */
				return e;
			}
		}
	}
	c->next = NULL;
	*out = c;
	return 0;
}

static void ctx_release(struct ctx *c)
{
	if (!c)
		return;
	pthread_mutex_lock(&pool_mu);
	c->next = pool_free[c->dev];
	pool_free[c->dev] = c;
	pthread_mutex_unlock(&pool_mu);
}

/* free the device buffers of every idle context of the current device (after an allocation failure) */
static void pool_trim(void)
{
	struct ctx *c;
	int dev = 0, i;
	if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEV)
		return;
	pthread_mutex_lock(&pool_mu);
	for (c = pool_free[dev]; c; c = c->next) {
		for (i = 0; i < PIPE; i++) {
			struct slot *s = &c->sl[i];
			drop_dev(&s->d_in);
			drop_dev(&s->d_slots);
			drop_dev(&s->d_len);
			drop_dev(&s->d_clen);
			drop_dev(&s->d_off);
			drop_dev(&s->d_packed);
			drop_dev(&s->d_out);
			drop_dev(&s->d_res);
		}
		drop_dev(&c->d_aux);
		drop_dev(&c->d_aux2);
	}
	pthread_mutex_unlock(&pool_mu);
}

/* grow with one retry after releasing what idle contexts hold (a transient shortage must not abort a compress call) */
static int grow_dev_retry(struct buf *b, size_t need)
{
	int e = grow_dev(b, need);
	if (e == (int)cudaErrorMemoryAllocation) {
		pool_trim();
		e = grow_dev(b, need);
	}
	return e;
}

#define TRY(what, expr)                          \
	do {                                     \
		int e__ = (int)(expr);           \
		if (e__) {                       \
			rc = set_err(what, e__); \
			goto out;                \
		}                                \
	} while (0)

static void die_no_error_channel(const char *fn)
{
	fprintf(stderr, "%s: %s (this entry point has no error return in the csnappy.h ABI; aborting)\n", fn, tls_err);
	abort();
}

/* ---- pageable caller memory ---------------------------------------------------------------------------------
 * cudaMemcpyAsync on pageable memory is staged by the driver on the calling thread, and a device-to-host copy into
 * pageable memory does not return before the kernels in front of it have finished: the chunk pipeline collapses into
 * "copy, run, copy" (measured: 8 GB/s through the container calls against 46 GB/s from pinned buffers).  For
 * pageable buffers the pipelines therefore stage every chunk through PINNED slot buffers themselves: the caller's
 * bytes move between pageable and pinned memory with a small pool of copy threads, everything the device sees is
 * pinned and asynchronous. */
#define COPY_Q 256
struct ctask {
	uint8_t *d;
	const uint8_t *s;
	size_t n;
	int *pending;
};
static pthread_mutex_t cp_mu = PTHREAD_MUTEX_INITIALIZER;
static pthread_cond_t cp_work = PTHREAD_COND_INITIALIZER, cp_done = PTHREAD_COND_INITIALIZER;
static struct ctask cp_q[COPY_Q];
static unsigned cp_head, cp_tail;
static int cp_threads = -1; /* -1: not started */

static void cp_run_locked(void)
{
	/* called with cp_mu held and the queue non-empty; returns with cp_mu held */
	struct ctask t = cp_q[cp_head++ % COPY_Q];
	pthread_mutex_unlock(&cp_mu);
	memcpy(t.d, t.s, t.n);
	pthread_mutex_lock(&cp_mu);
	if (--*t.pending == 0)
		pthread_cond_broadcast(&cp_done);
}

static void *cp_worker(void *arg)
{
	(void)arg;
	pthread_mutex_lock(&cp_mu);
	for (;;) {
		while (cp_head == cp_tail)
			pthread_cond_wait(&cp_work, &cp_mu);
		cp_run_locked();
	}
	return NULL;
}

static void cp_start_locked(void)
{
	long ncpu = sysconf(_SC_NPROCESSORS_ONLN);
	int want = g_copy_threads > 0 ? g_copy_threads : (ncpu >= 16 ? 7 : (ncpu >= 4 ? (int)ncpu / 2 - 1 : 0)), i;
	cp_threads = 0;
	for (i = 0; i < want; i++) {
		pthread_t th;
		pthread_attr_t at;
		pthread_attr_init(&at);
		pthread_attr_setdetachstate(&at, PTHREAD_CREATE_DETACHED);
		if (pthread_create(&th, &at, cp_worker, NULL) == 0)
			cp_threads++;
		pthread_attr_destroy(&at);
	}
}

/* memcpy, large copies cut into slices for the copy threads; the caller works on the queue while it waits */
static void par_memcpy(void *dst, const void *src, size_t n)
{
	const size_t min_slice = 1u << 20;
	int pending = 0;
	size_t slice, off;
	if (n < 2 * min_slice) {
		memcpy(dst, src, n);
		return;
	}
	pthread_mutex_lock(&cp_mu);
	if (cp_threads < 0)
		cp_start_locked();
	slice = n / (size_t)(cp_threads + 1);
	if (slice < min_slice)
		slice = min_slice;
	slice = (slice + 4095) & ~(size_t)4095;
	for (off = 0; off < n; off += slice) {
		struct ctask *t;
		while (cp_tail - cp_head == COPY_Q) /* queue full: work it down ourselves */
			cp_run_locked();
		t = &cp_q[cp_tail++ % COPY_Q];
		t->d = (uint8_t *)dst + off;
		t->s = (const uint8_t *)src + off;
		t->n = n - off < slice ? n - off : slice;
		t->pending = &pending;
		pending++;
	}
	pthread_cond_broadcast(&cp_work);
	while (pending) {
		if (cp_head != cp_tail)
			cp_run_locked();
		else
			pthread_cond_wait(&cp_done, &cp_mu);
	}
	pthread_mutex_unlock(&cp_mu);
}

/* 1 when p is ordinary pageable host memory (not pinned / registered / managed) */
static int is_pageable(const void *p)
{
	struct cudaPointerAttributes at;
	if (!p || g_no_bounce)
		return 0;
	if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
		cudaGetLastError();
		return 1;
	}
	return at.type == cudaMemoryTypeUnregistered;
}

/* finish a slot's deferred copy-out: its device-to-host copies into the pinned staging have been queued on b->s.
 * slot_owe2: `rows` runs of `width` bytes, `pitch` apart in the staging and in the caller's memory (the bytes in
 * between belong to the caller and are not written). */
static void slot_owe2(struct slot *b, const void *pinned_src, void *dst, size_t width, size_t pitch, size_t rows)
{
	b->pend[b->npend].src = pinned_src;
	b->pend[b->npend].dst = dst;
	b->pend[b->npend].width = width;
	b->pend[b->npend].pitch = pitch;
	b->pend[b->npend].rows = rows;
	b->npend++;
}

static void slot_owe(struct slot *b, const void *pinned_src, void *dst, size_t n) { slot_owe2(b, pinned_src, dst, n, n, 1); }

static int slot_drain(struct slot *b)
{
	int e = 0, i;
	size_t r;
	if (!b->npend)
		return 0;
	e = (int)cudaStreamSynchronize(b->s);
	for (i = 0; i < b->npend && !e; i++) {
		const uint8_t *s = (const uint8_t *)b->pend[i].src;
		uint8_t *d = (uint8_t *)b->pend[i].dst;
		if (b->pend[i].width == b->pend[i].pitch)
			par_memcpy(d, s, b->pend[i].width * b->pend[i].rows);
		else
			for (r = 0; r < b->pend[i].rows; r++)
				memcpy(d + r * b->pend[i].pitch, s + r * b->pend[i].pitch, b->pend[i].width);
	}
	b->npend = 0;
	return e;
}

/* device-to-host copy of `rows` slots: the first `width` bytes of each, `pitch` apart on both sides (one flat copy
 * when width == pitch) */
static int d2h_slots(void *dst, const void *src, size_t width, size_t pitch, size_t rows, cudaStream_t s)
{
	if (!width || !rows)
		return 0;
	if (width == pitch)
		return (int)cudaMemcpyAsync(dst, src, width * rows, cudaMemcpyDeviceToHost, s);
	return (int)cudaMemcpy2DAsync(dst, pitch, src, pitch, width, rows, cudaMemcpyDeviceToHost, s);
}

/* optional page-locking of caller memory for the duration of a call ("host_register" knob) */
struct hostreg {
	void *p;
};
static void hostreg_begin(struct hostreg *r, const void *p, size_t n)
{
	/* the pages that CONTAIN the buffer (they are mapped: they hold its bytes); a copy that starts in an
	 * unregistered head of a partly registered range is refused by the driver */
	const size_t pg = (size_t)sysconf(_SC_PAGESIZE);
	uintptr_t a = (uintptr_t)p & ~(uintptr_t)(pg - 1), b = ((uintptr_t)p + n + pg - 1) & ~(uintptr_t)(pg - 1);
	r->p = NULL;
	if (!g_host_register || !p || n < (8u << 20))
		return;
	if (cudaHostRegister((void *)a, b - a, cudaHostRegisterPortable) == cudaSuccess)
		r->p = (void *)a;
	else
		cudaGetLastError(); /* already pinned by the caller, or not registrable: copy from it as it is */
}
static void hostreg_end(struct hostreg *r)
{
	if (r->p)
		cudaHostUnregister(r->p);
	r->p = NULL;
}

/* ---- single small calls: one fragment / one small stream -------------------------------------------------- */

/* one fragment (the per-page call of zram / block_compressor): pinned bounce buffers, the size travels in front of the
 * slot, ONE stream synchronisation.  Returns bytes written to out or a negative error. */
static int64_t compress_one(const uint8_t *in, uint32_t n, uint8_t *out, int wm, uint32_t kflags)
{
	int64_t rc = 0;
	struct ctx *c = NULL;
	struct slot *sl;
	struct csb_compress_args a;
	const size_t in_pad = ((size_t)n + 63) & ~(size_t)63, slot = HDR + csnappy_max_compressed_length(n);
	uint8_t *pin;
	uint32_t clen;
	TRY("context", ctx_acquire(&c));
	sl = &c->sl[0];
	TRY("cudaMallocHost", grow_pin(&c->h_pin, in_pad + slot + 64));
	TRY("cudaMalloc(in)", grow_dev_retry(&sl->d_in, (size_t)n + 64));
	TRY("cudaMalloc(slots)", grow_dev_retry(&sl->d_slots, SLOT_STRIDE_32K + HDR));
	TRY("cudaMalloc(ctr)", grow_dev_retry(&sl->d_ctr, 64));
	pin = (uint8_t *)c->h_pin.p;
	memcpy(pin, in, n);
	TRY("H2D", cudaMemcpyAsync(sl->d_in.p, pin, n, cudaMemcpyHostToDevice, sl->s));
	fill_compress_args(&a);
	a.in = (const uint8_t *)sl->d_in.p;
	a.in_stride = CSB_FRAGMENT_MAX;
	a.uniform_len = n;
	a.n_blocks = 1;
	a.out = (uint8_t *)sl->d_slots.p + HDR;
	a.out_stride = SLOT_STRIDE_32K;
	a.out_len = (uint32_t *)sl->d_slots.p;
	a.wm = wm;
	a.flags = kflags;
	a.counter = (uint32_t *)sl->d_ctr.p;
	TRY("compress launch", csb_launch_compress(&a, (csb_stream_t)sl->s));
	TRY("D2H", cudaMemcpyAsync(pin + in_pad, sl->d_slots.p, slot, cudaMemcpyDeviceToHost, sl->s));
	TRY("sync", cudaStreamSynchronize(sl->s));
	memcpy(&clen, pin + in_pad, 4);
	memcpy(out, pin + in_pad + HDR, clen);
	rc = (int64_t)clen;
out:
	ctx_release(c);
	return rc;
}

/* ---- compress pipeline: pages / fragments of ONE host buffer through one or several devices ---------------
 * Used by the block_compressor container writer (stored-block rule, size index) and by csnappy_compress on
 * large buffers (32 KiB fragments, short-last-chunk table rule, no index).  The buffer is cut into chunks;
 * chunk c goes to device c mod G.  Per chunk: H2D, compress kernel, size scan + pack on the device, then only
 * the PACKED payload travels back, straight to its final position.  That position is the sum of the packed
 * sizes of all earlier chunks: the one value that crosses devices, handed from chunk to chunk in order.     */
struct cjob {
	const uint8_t *in;
	uint64_t in_len;
	uint32_t page;
	int wm;
	uint32_t kflags;
	int stored;	      /* block_compressor.c:316-318 */
	uint8_t *index_out;   /* u32 per page, or NULL */
	uint8_t *payload_out; /* payload byte 0 */
	uint64_t nr, n_chunks;
	uint32_t chunk;
	int G;
	const int *devs; /* NULL: the current device (G == 1) */
	pthread_mutex_t mu;
	pthread_cond_t cv;
	uint64_t pos_chunk, pos; /* payload position of chunk pos_chunk */
	int in_pageable, out_pageable; /* stage the chunks through pinned slot buffers (see par_memcpy) */
	int err;
	char errtext[256];
};

struct cworker {
	struct cjob *j;
	int g;
	pthread_t th;
};

static void cjob_fail(struct cjob *j, int rc)
{
	pthread_mutex_lock(&j->mu);
	if (!j->err) {
		j->err = rc;
		memcpy(j->errtext, tls_err, sizeof(j->errtext));
	}
	pthread_cond_broadcast(&j->cv);
	pthread_mutex_unlock(&j->mu);
}

static void *compress_worker(void *arg)
{
	struct cworker *w = (struct cworker *)arg;
	struct cjob *j = w->j;
	struct ctx *c = NULL;
	const uint32_t out_stride = (csnappy_max_compressed_length(j->page) + 15u) & ~15u;
	const uint64_t n_mine = (uint64_t)w->g < j->n_chunks ? (j->n_chunks - (uint64_t)w->g + (uint64_t)j->G - 1) / (uint64_t)j->G : 0;
	uint64_t issued = 0, retired = 0;
	int rc = 0, k;
	if (j->devs)
		TRY("cudaSetDevice", cudaSetDevice(j->devs[w->g]));
	if (n_mine == 0)
		return NULL;
	TRY("context", ctx_acquire(&c));
	for (k = 0; k < PIPE && (uint64_t)k < n_mine; k++) {
		struct slot *b = &c->sl[k];
		TRY("cudaMalloc(in)", grow_dev_retry(&b->d_in, (size_t)j->chunk * j->page + 64));
		TRY("cudaMalloc(slots)", grow_dev_retry(&b->d_slots, (size_t)j->chunk * out_stride + 64));
		TRY("cudaMalloc(len)", grow_dev_retry(&b->d_len, (size_t)j->chunk * 4 + 64));
		TRY("cudaMalloc(clen)", grow_dev_retry(&b->d_clen, (size_t)j->chunk * 4 + 64));
		TRY("cudaMalloc(off)", grow_dev_retry(&b->d_off, ((size_t)j->chunk + 1) * 8 + 64));
		TRY("cudaMalloc(packed)", grow_dev_retry(&b->d_packed, (size_t)j->chunk * (j->stored ? j->page : out_stride) + 64));
		TRY("cudaMallocHost(res)", grow_pin(&b->h_res, 64));
		TRY("cudaMalloc(ctr)", grow_dev_retry(&b->d_ctr, 64));
		if (j->in_pageable)
			TRY("cudaMallocHost(in)", grow_pin(&b->h_in, (size_t)j->chunk * j->page + 64));
		if (j->out_pageable) {
			TRY("cudaMallocHost(out)", grow_pin(&b->h_out, (size_t)j->chunk * (j->stored ? j->page : out_stride) + 64));
			TRY("cudaMallocHost(idx)", grow_pin(&b->h_idx, (size_t)j->chunk * 4 + 64));
		}
		b->npend = 0;
	}
	while (retired < n_mine) {
		if (j->err)
			goto out; /* somebody else failed */
		/* retire the oldest chunk once two younger ones are queued (or nothing is left to queue) */
		if (retired < issued && (issued - retired > 2 || issued == n_mine)) {
			struct slot *b = &c->sl[retired % PIPE];
			const uint64_t gc = (uint64_t)w->g + retired * (uint64_t)j->G;
			uint64_t total, pos;
			TRY("event sync", cudaEventSynchronize(b->ev));
			total = *(uint64_t *)b->h_res.p;
			pthread_mutex_lock(&j->mu);
			while (j->pos_chunk != gc && !j->err)
				pthread_cond_wait(&j->cv, &j->mu);
			pos = j->pos;
			j->pos_chunk = gc + 1;
			j->pos += total;
			pthread_cond_broadcast(&j->cv);
			pthread_mutex_unlock(&j->mu);
			if (j->err)
				goto out;
			if (total && j->out_pageable) {
				TRY("D2H payload", cudaMemcpyAsync(b->h_out.p, b->d_packed.p, total, cudaMemcpyDeviceToHost, b->s));
				slot_owe(b, b->h_out.p, j->payload_out + pos, total); /* copied out when the slot comes round again, or at the end */
			} else if (total) {
				TRY("D2H payload", cudaMemcpyAsync(j->payload_out + pos, b->d_packed.p, total, cudaMemcpyDeviceToHost, b->s));
			}
			retired++;
			continue;
		}
		{
			struct slot *b = &c->sl[issued % PIPE];
			const uint64_t gc = (uint64_t)w->g + issued * (uint64_t)j->G;
			const uint64_t first = gc * j->chunk, left_pages = j->nr - first, in_at = first * j->page;
			const uint32_t nb = left_pages < j->chunk ? (uint32_t)left_pages : j->chunk;
			const uint64_t in_bytes = j->in_len - in_at < (uint64_t)nb * j->page ? j->in_len - in_at : (uint64_t)nb * j->page;
			struct csb_compress_args a;
			TRY("copy-out of the slot's previous chunk", slot_drain(b));
			if (j->in_pageable) {
				par_memcpy(b->h_in.p, j->in + in_at, in_bytes);
				TRY("H2D", cudaMemcpyAsync(b->d_in.p, b->h_in.p, in_bytes, cudaMemcpyHostToDevice, b->s));
			} else {
				TRY("H2D", cudaMemcpyAsync(b->d_in.p, j->in + in_at, in_bytes, cudaMemcpyHostToDevice, b->s));
			}
			fill_compress_args(&a);
			a.in = (const uint8_t *)b->d_in.p;
			a.in_stride = j->page;
			a.uniform_len = j->page;
			a.total_len = in_bytes;
			a.n_blocks = nb;
			a.out = (uint8_t *)b->d_slots.p;
			a.out_stride = out_stride;
			a.out_len = (uint32_t *)b->d_len.p;
			a.wm = j->wm;
			a.flags = j->kflags;
			a.counter = (uint32_t *)b->d_ctr.p;
			TRY("compress launch", csb_launch_compress(&a, (csb_stream_t)b->s));
			if (j->stored) {
				TRY("pack launch", csb_launch_pack_stored((const uint8_t *)b->d_slots.p, out_stride, (const uint32_t *)b->d_len.p, nb,
									  (const uint8_t *)b->d_in.p, j->page, in_bytes, (uint32_t *)b->d_clen.p,
									  (uint8_t *)b->d_packed.p, (uint64_t *)b->d_off.p, (csb_stream_t)b->s));
			} else {
				TRY("pack launch", csb_launch_pack((const uint8_t *)b->d_slots.p, out_stride, (const uint32_t *)b->d_len.p, nb,
								   (uint8_t *)b->d_packed.p, (uint64_t *)b->d_off.p, (csb_stream_t)b->s));
			}
			TRY("D2H total", cudaMemcpyAsync(b->h_res.p, (uint64_t *)b->d_off.p + nb, 8, cudaMemcpyDeviceToHost, b->s));
			if (j->index_out && j->out_pageable) {
				TRY("D2H index", cudaMemcpyAsync(b->h_idx.p, j->stored ? b->d_clen.p : b->d_len.p, (size_t)nb * 4,
								 cudaMemcpyDeviceToHost, b->s));
				slot_owe(b, b->h_idx.p, j->index_out + 4 * first, (size_t)nb * 4);
			} else if (j->index_out) {
				TRY("D2H index", cudaMemcpyAsync(j->index_out + 4 * first, j->stored ? b->d_clen.p : b->d_len.p, (size_t)nb * 4,
								 cudaMemcpyDeviceToHost, b->s));
			}
			TRY("event record", cudaEventRecord(b->ev, b->s));
			issued++;
		}
	}
out:
	if (c)
		for (k = 0; k < PIPE; k++) {
			int e = slot_drain(&c->sl[k]); /* synchronises the slot's stream */
			if (e && !rc)
				rc = set_err("copy-out", e);
			cudaStreamSynchronize(c->sl[k].s);
		}
	if (rc)
		cjob_fail(j, rc);
	ctx_release(c);
	return NULL;
}

/* run the job on G devices (devs == NULL: inline on the current device); returns 0 or a negative error */
static int run_cjob(struct cjob *j)
{
	struct cworker w[MAX_DEV];
	int g;
	pthread_mutex_init(&j->mu, NULL);
	pthread_cond_init(&j->cv, NULL);
	j->pos_chunk = 0;
	j->pos = 0;
	j->err = 0;
	if (!j->devs) {
		w[0].j = j;
		w[0].g = 0;
		compress_worker(&w[0]);
	} else {
		int started = 0;
		for (g = 0; g < j->G; g++) {
			w[g].j = j;
			w[g].g = g;
			if (pthread_create(&w[g].th, NULL, compress_worker, &w[g])) {
				set_err("pthread_create", (int)cudaErrorUnknown);
				cjob_fail(j, CSNAPPY_E_DEVICE);
				break;
			}
			started++;
		}
		for (g = 0; g < started; g++)
			pthread_join(w[g].th, NULL);
	}
	if (j->err)
		memcpy(tls_err, j->errtext, sizeof(tls_err));
	pthread_mutex_destroy(&j->mu);
	pthread_cond_destroy(&j->cv);
	return j->err;
}

static uint32_t chunk_units(uint32_t unit_bytes, uint64_t n_units, int G)
{
	/* ~32 MiB per chunk keeps PCIe busy and the kernels full; small inputs are still cut into a few chunks per device */
	uint64_t units = ((uint64_t)(g_chunk_mb > 0 ? g_chunk_mb : 32) << 20) / unit_bytes, per_dev = (n_units + (uint64_t)G - 1) / (uint64_t)G;
	if (units > (per_dev + 3) / 4)
		units = (per_dev + 3) / 4;
	if (units < 256)
		units = 256;
	if (units > n_units)
		units = n_units;
	return (uint32_t)units;
}

/* device list of a *_multi call: devices NULL -> 0..n-1; n_devices 0 -> all visible */
static int resolve_devices(const int *devices, int n_devices, int *list)
{
	int n = csnappy_b200_device_count(), i;
	if (n <= 0)
		return CSNAPPY_E_DEVICE;
	if (n_devices < 0 || n_devices > MAX_DEV)
		return set_err("n_devices", 0);
	if (n_devices == 0)
		n_devices = n;
	for (i = 0; i < n_devices; i++) {
		list[i] = devices ? devices[i] : i;
		if (list[i] < 0 || list[i] >= n)
			return set_err("device index outside the visible devices", 0);
	}
	return n_devices;
}

/*
 * Core of both compress entry points.  framed = 0: one fragment, no header.
 * framed = 1: varint32 + 32 KiB fragments with the short-chunk table rule.
 * Returns bytes written to `out` (>= 0) or a negative error.
 */
static int64_t compress_host(const uint8_t *in, uint32_t n, uint8_t *out, int wm, int framed)
{
	uint32_t hdr = framed ? put_varint32(out, n) : 0;
	uint32_t n_frag = framed ? (uint32_t)(((uint64_t)n + CSB_FRAGMENT_MAX - 1) / CSB_FRAGMENT_MAX) : (n ? 1u : 0u);
	if (wm < 9 || wm > 16)
		return set_err("workmem_bytes_power_of_two outside 9..16", 0);
	if (!framed && n > CSB_FRAGMENT_MAX)
		return set_err("csnappy_compress_fragment: input longer than 32768 bytes", 0);
	if (n_frag == 0)
		return hdr;
	if (n_frag == 1) {
		int64_t r = compress_one(in, n, out + hdr, wm, framed ? CSNAPPY_BATCH_SHRINK_TABLE : 0);
		return r < 0 ? r : (int64_t)hdr + r;
	}
	{
		/* many fragments: chunks of fragments pipelined through the device (H2D of the next chunk overlaps the
		 * kernels and the D2H of the previous ones), packed payload straight into `out` */
		struct cjob j;
		struct hostreg r1, r2;
		int rc;
		memset(&j, 0, sizeof(j));
		j.in = in;
		j.in_len = n;
		j.page = CSB_FRAGMENT_MAX;
		j.wm = wm;
		j.kflags = CSNAPPY_BATCH_SHRINK_TABLE;
		j.payload_out = out + hdr;
		j.nr = n_frag;
		j.G = 1;
		j.chunk = chunk_units(CSB_FRAGMENT_MAX, n_frag, 1);
		j.n_chunks = (j.nr + j.chunk - 1) / j.chunk;
		hostreg_begin(&r1, in, n);
		hostreg_begin(&r2, out, (size_t)n + n / 6);
		j.in_pageable = is_pageable(in);
		j.out_pageable = is_pageable(out);
		rc = run_cjob(&j);
		hostreg_end(&r1);
		hostreg_end(&r2);
		return rc ? rc : (int64_t)hdr + (int64_t)j.pos;
	}
}

char *csnappy_compress_fragment(const char *input, const uint32_t input_length, char *output,
				void *working_memory, const int workmem_bytes_power_of_two)
{
	int64_t r;
	(void)working_memory; /* the hash table lives in shared memory on the device */
	r = compress_host((const uint8_t *)input, input_length, (uint8_t *)output, workmem_bytes_power_of_two, 0);
	if (r < 0)
		die_no_error_channel("csnappy_compress_fragment");
	return output + r;
}

void csnappy_compress(const char *input, uint32_t input_length, char *compressed,
		      uint32_t *out_compressed_length, void *working_memory,
		      const int workmem_bytes_power_of_two)
{
	int64_t r;
	(void)working_memory;
	r = compress_host((const uint8_t *)input, input_length, (uint8_t *)compressed, workmem_bytes_power_of_two, 1);
	if (r < 0)
		die_no_error_channel("csnappy_compress");
	*out_compressed_length = (uint32_t)r;
}

/* raw decode of src[0..src_len) into dst with capacity cap; *produced set on success */
static int decompress_host(const uint8_t *src, uint32_t src_len, uint8_t *dst, uint32_t cap, uint32_t *produced)
{
	int rc = 0;
	struct ctx *c = NULL;
	struct slot *sl;
	struct csb_decompress_args a;
	cudaStream_t s;
	struct {
		uint32_t out_len;
		int32_t status;
	} res = {0, 0};
	uint32_t *d_res;

	TRY("context", ctx_acquire(&c));
	sl = &c->sl[0];
	s = sl->s;
	if (src_len <= SMALL_CALL && cap <= SMALL_CALL) {
		/* one small block (the per-page call of zram / block_compressor): pinned bounce buffers, the input
		 * length travels in front of the input and [out_len, status] in front of the output, ONE synchronisation */
		const size_t in_bytes = HDR + src_len, in_pad = (in_bytes + 63) & ~(size_t)63, out_bytes = HDR + cap;
		uint8_t *pin;
		uint32_t *d_ihdr, *d_ohdr;
		TRY("cudaMallocHost", grow_pin(&c->h_pin, in_pad + out_bytes + 64));
		TRY("cudaMalloc(in)", grow_dev_retry(&sl->d_in, in_bytes + 64));
		TRY("cudaMalloc(out)", grow_dev_retry(&sl->d_out, out_bytes + 64));
		TRY("cudaMalloc(ctr)", grow_dev_retry(&sl->d_ctr, 64));
		pin = (uint8_t *)c->h_pin.p;
		memset(pin, 0, HDR);
		memcpy(pin, &src_len, 4);
		memcpy(pin + HDR, src, src_len);
		TRY("H2D", cudaMemcpyAsync(sl->d_in.p, pin, in_bytes, cudaMemcpyHostToDevice, s));
		d_ihdr = (uint32_t *)sl->d_in.p;
		d_ohdr = (uint32_t *)sl->d_out.p;
		fill_decompress_args(&a);
		if (a.stage_input == 4)
			a.stage_input = 0; /* one block: never one lane */
		a.in = (const uint8_t *)sl->d_in.p + HDR;
		a.in_len = d_ihdr;
		a.n_blocks = 1;
		a.out = (uint8_t *)sl->d_out.p + HDR;
		a.uniform_cap = cap;
		a.out_len = d_ohdr;
		a.status = (int32_t *)(d_ohdr + 1);
		a.max_in_len = src_len;
		a.counter = (uint32_t *)sl->d_ctr.p;
		TRY("decompress launch", csb_launch_decompress(&a, (csb_stream_t)s));
		TRY("D2H", cudaMemcpyAsync(pin + in_pad, sl->d_out.p, out_bytes, cudaMemcpyDeviceToHost, s));
		TRY("sync", cudaStreamSynchronize(s));
		memcpy(&res, pin + in_pad, 8);
		rc = res.status;
		if (rc == 0) {
			memcpy(dst, pin + in_pad + HDR, res.out_len);
			*produced = res.out_len;
		}
		goto out;
	}
	/* one long stream */
	{
		struct hostreg r1, r2;
		const int use_stream = g_stream_min >= 0 && src_len >= (uint32_t)g_stream_min;
		TRY("cudaMalloc(in)", grow_dev_retry(&sl->d_in, (size_t)src_len + 64));
		TRY("cudaMalloc(out)", grow_dev_retry(&sl->d_out, (size_t)cap + 64));
		TRY("cudaMalloc(res)", grow_dev_retry(&sl->d_res, 64));
		TRY("cudaMalloc(ctr)", grow_dev_retry(&sl->d_ctr, 64));
		d_res = (uint32_t *)sl->d_res.p;
		hostreg_begin(&r1, src, src_len);
		hostreg_begin(&r2, dst, cap);
		rc = 0;
		do {
			int e;
			if (src_len && (e = (int)cudaMemcpyAsync(sl->d_in.p, src, src_len, cudaMemcpyHostToDevice, s))) {
				rc = set_err("H2D", e);
				break;
			}
			e = 1;
			if (use_stream) {
				/* parallel single-stream decoder (stream_kernel.cu); its tables: 8 bytes per input byte + 4 per output byte.
				 * If they cannot be had, the serial warp-per-stream path below still decodes the stream. */
				const size_t t1 = csb_stream_aux_bytes(src_len, cap, 0), t2 = csb_stream_aux_bytes(src_len, cap, 1);
				if (!grow_dev(&c->d_aux, t1) && !grow_dev(&c->d_aux2, t2))
					e = csb_launch_decompress_stream((const uint8_t *)sl->d_in.p, src_len, (uint8_t *)sl->d_out.p, cap, d_res,
									 (int32_t *)(d_res + 1), c->d_aux.p, c->d_aux2.p, (csb_stream_t)s);
				if (e > 1) {
					rc = set_err("stream decoder launch", e);
					break;
				}
			}
			if (e == 1) {
				if ((e = (int)cudaMemcpyAsync(d_res + 2, &src_len, 4, cudaMemcpyHostToDevice, s))) {
					rc = set_err("H2D len", e);
					break;
				}
				fill_decompress_args(&a);
				if (a.stage_input == 4)
					a.stage_input = 0;
				a.in = (const uint8_t *)sl->d_in.p;
				a.in_len = d_res + 2;
				a.n_blocks = 1;
				a.out = (uint8_t *)sl->d_out.p;
				a.uniform_cap = cap;
				a.out_len = d_res;
				a.status = (int32_t *)(d_res + 1);
				a.max_in_len = src_len;
				a.counter = (uint32_t *)sl->d_ctr.p;
				if ((e = csb_launch_decompress(&a, (csb_stream_t)s))) {
					rc = set_err("decompress launch", e);
					break;
				}
			}
			if ((e = (int)cudaMemcpyAsync(&res, d_res, 8, cudaMemcpyDeviceToHost, s)) || (e = (int)cudaStreamSynchronize(s))) {
				rc = set_err("D2H result", e);
				break;
			}
			rc = res.status;
			if (rc == 0) {
				if (res.out_len && ((e = (int)cudaMemcpyAsync(dst, sl->d_out.p, res.out_len, cudaMemcpyDeviceToHost, s)) ||
						    (e = (int)cudaStreamSynchronize(s)))) {
					rc = set_err("D2H data", e);
					break;
				}
				*produced = res.out_len;
			}
		} while (0);
		hostreg_end(&r1);
		hostreg_end(&r2);
	}
out:
	ctx_release(c);
	return rc;
}

int csnappy_decompress_noheader(const char *src, uint32_t src_len, char *dst, uint32_t *dst_len)
{
	uint32_t produced = 0;
	int rc = decompress_host((const uint8_t *)src, src_len, (uint8_t *)dst, *dst_len, &produced);
	if (rc == 0)
		*dst_len = produced; /* written only on success, csnappy_decompress.c:385 */
	return rc;
}

int csnappy_decompress(const char *src, uint32_t src_len, char *dst, uint32_t dst_len)
{
	uint32_t olen = 0, produced = 0;
	int n = csnappy_get_uncompressed_length(src, src_len, &olen);
	if (n < 0)
		return n;
	if (olen > dst_len)
		return CSNAPPY_E_OUTPUT_INSUF;
	return decompress_host((const uint8_t *)src + n, src_len - (uint32_t)n, (uint8_t *)dst, olen, &produced);
}

/* ---- host-buffer batches of strided slots: chunked, H2D / kernel / D2H overlap ---- */
static size_t pick_chunk_blocks(uint64_t in_stride, uint64_t out_stride, uint32_t n_blocks)
{
	/* ~32 MiB of the larger side per chunk keeps PCIe busy and the kernels full */
	uint64_t per = in_stride > out_stride ? in_stride : out_stride;
	uint64_t blocks = per ? ((uint64_t)(g_chunk_mb > 0 ? g_chunk_mb : 32) << 20) / per : n_blocks;
	if (blocks < 1024)
		blocks = 1024;
	if (blocks > n_blocks)
		blocks = n_blocks;
	return (size_t)blocks;
}

int csnappy_batch_compress_fragments_host(const void *h_in, uint64_t in_stride, uint32_t uniform_in_len,
					  uint32_t n_blocks, void *h_out, uint64_t out_stride,
					  uint32_t *h_out_len, int workmem_bytes_power_of_two)
{
	int rc = 0, k, in_pg, out_pg;
	size_t chunk, done, width;
	struct ctx *c = NULL;
	if (workmem_bytes_power_of_two < 9 || workmem_bytes_power_of_two > 16)
		return set_err("workmem_bytes_power_of_two outside 9..16", 0);
	if (uniform_in_len > CSB_FRAGMENT_MAX || in_stride < uniform_in_len ||
	    out_stride < csnappy_max_compressed_length(uniform_in_len))
		return set_err("bad block geometry", 0);
	width = csnappy_max_compressed_length(uniform_in_len); /* bytes of a slot the kernel may write */
	if (n_blocks == 0)
		return 0;
	if (!h_in || !h_out || !h_out_len)
		return set_err("null buffer", 0);

	TRY("context", ctx_acquire(&c));
	chunk = pick_chunk_blocks(in_stride, out_stride, n_blocks);
	in_pg = is_pageable(h_in);
	out_pg = is_pageable(h_out) || is_pageable(h_out_len);
	for (k = 0; k < PIPE; k++) {
		TRY("cudaMalloc(in)", grow_dev_retry(&c->sl[k].d_in, chunk * in_stride + 64));
		TRY("cudaMalloc(out)", grow_dev_retry(&c->sl[k].d_slots, chunk * out_stride + 64));
		TRY("cudaMalloc(len)", grow_dev_retry(&c->sl[k].d_len, chunk * 4 + 64));
		TRY("cudaMalloc(ctr)", grow_dev_retry(&c->sl[k].d_ctr, 64));
		if (in_pg)
			TRY("cudaMallocHost(in)", grow_pin(&c->sl[k].h_in, chunk * in_stride + 64));
		if (out_pg) {
			TRY("cudaMallocHost(out)", grow_pin(&c->sl[k].h_out, chunk * out_stride + 64));
			TRY("cudaMallocHost(len)", grow_pin(&c->sl[k].h_idx, chunk * 8 + 64));
		}
		c->sl[k].npend = 0;
	}
	for (done = 0, k = 0; done < n_blocks; done += chunk, k = (k + 1) % PIPE) {
		size_t nb = n_blocks - done < chunk ? n_blocks - done : chunk;
		/* the last chunk ends with its last block: the caller's buffer need not extend to a whole stride */
		const size_t in_bytes = done + nb == n_blocks ? (nb - 1) * in_stride + uniform_in_len : nb * in_stride;
		struct slot *b = &c->sl[k];
		struct csb_compress_args a;
		const uint8_t *src = (const uint8_t *)h_in + done * in_stride;
		TRY("copy-out of the slot's previous chunk", slot_drain(b));
		if (in_pg) { /* pageable caller memory: through the slot's pinned staging (see par_memcpy) */
			par_memcpy(b->h_in.p, src, in_bytes);
			src = (const uint8_t *)b->h_in.p;
		}
		if (in_bytes)
			TRY("H2D", cudaMemcpyAsync(b->d_in.p, src, in_bytes, cudaMemcpyHostToDevice, b->s));
		fill_compress_args(&a);
		a.in = (const uint8_t *)b->d_in.p;
		a.in_stride = in_stride;
		a.uniform_len = uniform_in_len;
		a.n_blocks = (uint32_t)nb;
		a.out = (uint8_t *)b->d_slots.p;
		a.out_stride = out_stride;
		a.out_len = (uint32_t *)b->d_len.p;
		a.wm = workmem_bytes_power_of_two;
		a.counter = (uint32_t *)b->d_ctr.p;
		TRY("compress launch", csb_launch_compress(&a, (csb_stream_t)b->s));
		if (out_pg) {
			TRY("D2H data", cudaMemcpyAsync(b->h_out.p, b->d_slots.p, nb * out_stride, cudaMemcpyDeviceToHost, b->s));
			TRY("D2H len", cudaMemcpyAsync(b->h_idx.p, b->d_len.p, nb * 4, cudaMemcpyDeviceToHost, b->s));
			slot_owe2(b, b->h_out.p, (uint8_t *)h_out + done * out_stride, width, out_stride, nb);
			slot_owe(b, b->h_idx.p, h_out_len + done, nb * 4);
		} else {
			TRY("D2H data", d2h_slots((uint8_t *)h_out + done * out_stride, b->d_slots.p, width, out_stride, nb, b->s));
			TRY("D2H len", cudaMemcpyAsync(h_out_len + done, b->d_len.p, nb * 4, cudaMemcpyDeviceToHost, b->s));
		}
	}
out:
	if (c)
		for (k = 0; k < PIPE; k++) {
			int e = slot_drain(&c->sl[k]);
			if (!e)
				e = (int)cudaStreamSynchronize(c->sl[k].s);
			if (e && !rc)
				rc = set_err("sync", e);
		}
	ctx_release(c);
	return rc;
}

int csnappy_batch_decompress_host(const void *h_in, uint64_t in_stride, const uint32_t *h_in_len,
				  uint32_t n_blocks, void *h_out, uint64_t out_stride, uint32_t uniform_out_cap,
				  uint32_t *h_out_len, int32_t *h_status, uint32_t flags)
{
	int rc = 0, k, in_pg, out_pg;
	size_t chunk, done;
	struct ctx *c = NULL;
	if (out_stride < uniform_out_cap)
		return set_err("bad block geometry", 0);
	if (n_blocks == 0)
		return 0;
	if (!h_in || !h_in_len || !h_out || !h_out_len || !h_status)
		return set_err("null buffer", 0);
	{
		/* a length beyond the stride would make the kernel read past the staged chunk (csnappy_bc_decompress_host
		 * checks its index the same way) */
		uint32_t i;
		for (i = 0; i < n_blocks; i++)
			if (h_in_len[i] > in_stride)
				return set_err("h_in_len[i] larger than in_stride", 0);
	}

	TRY("context", ctx_acquire(&c));
	chunk = pick_chunk_blocks(in_stride, out_stride, n_blocks);
	in_pg = is_pageable(h_in);
	out_pg = is_pageable(h_out) || is_pageable(h_out_len) || is_pageable(h_status);
	for (k = 0; k < PIPE; k++) {
		TRY("cudaMalloc(in)", grow_dev_retry(&c->sl[k].d_in, chunk * in_stride + 64));
		TRY("cudaMalloc(out)", grow_dev_retry(&c->sl[k].d_out, chunk * out_stride + 64));
		TRY("cudaMalloc(aux)", grow_dev_retry(&c->sl[k].d_res, chunk * 12 + 64));
		TRY("cudaMalloc(ctr)", grow_dev_retry(&c->sl[k].d_ctr, 64));
		if (in_pg)
			TRY("cudaMallocHost(in)", grow_pin(&c->sl[k].h_in, chunk * in_stride + 64));
		if (out_pg) {
			TRY("cudaMallocHost(out)", grow_pin(&c->sl[k].h_out, chunk * out_stride + 64));
			TRY("cudaMallocHost(len)", grow_pin(&c->sl[k].h_idx, chunk * 8 + 64));
		}
		c->sl[k].npend = 0;
	}
	for (done = 0, k = 0; done < n_blocks; done += chunk, k = (k + 1) % PIPE) {
		size_t nb = n_blocks - done < chunk ? n_blocks - done : chunk;
		struct slot *b = &c->sl[k];
		uint32_t *d_ilen = (uint32_t *)b->d_res.p, *d_olen = d_ilen + chunk;
		int32_t *d_st = (int32_t *)(d_olen + chunk);
		/* the last chunk ends with its last block: the caller's buffer need not extend to a whole stride */
		const size_t in_bytes = done + nb == n_blocks ? (nb - 1) * in_stride + h_in_len[n_blocks - 1] : nb * in_stride;
		struct csb_decompress_args a;
		const uint8_t *src = (const uint8_t *)h_in + done * in_stride;
		TRY("copy-out of the slot's previous chunk", slot_drain(b));
		if (in_pg) {
			par_memcpy(b->h_in.p, src, in_bytes);
			src = (const uint8_t *)b->h_in.p;
		}
		if (in_bytes)
			TRY("H2D", cudaMemcpyAsync(b->d_in.p, src, in_bytes, cudaMemcpyHostToDevice, b->s));
		TRY("H2D len", cudaMemcpyAsync(d_ilen, h_in_len + done, nb * 4, cudaMemcpyHostToDevice, b->s));
		fill_decompress_args(&a);
		a.in = (const uint8_t *)b->d_in.p;
		a.in_stride = in_stride;
		a.in_len = d_ilen;
		a.n_blocks = (uint32_t)nb;
		a.out = (uint8_t *)b->d_out.p;
		a.out_stride = out_stride;
		a.uniform_cap = uniform_out_cap;
		a.out_len = d_olen;
		a.status = d_st;
		a.flags = flags;
		a.counter = (uint32_t *)b->d_ctr.p;
		TRY("decompress launch", csb_launch_decompress(&a, (csb_stream_t)b->s));
		if (out_pg) {
			uint8_t *h_len = (uint8_t *)b->h_idx.p, *h_st = h_len + chunk * 4;
			TRY("D2H data", cudaMemcpyAsync(b->h_out.p, b->d_out.p, nb * out_stride, cudaMemcpyDeviceToHost, b->s));
			TRY("D2H len", cudaMemcpyAsync(h_len, d_olen, nb * 4, cudaMemcpyDeviceToHost, b->s));
			TRY("D2H status", cudaMemcpyAsync(h_st, d_st, nb * 4, cudaMemcpyDeviceToHost, b->s));
			slot_owe2(b, b->h_out.p, (uint8_t *)h_out + done * out_stride, uniform_out_cap, out_stride, nb);
			slot_owe(b, h_len, h_out_len + done, nb * 4);
			slot_owe(b, h_st, h_status + done, nb * 4);
		} else {
			TRY("D2H data", d2h_slots((uint8_t *)h_out + done * out_stride, b->d_out.p, uniform_out_cap, out_stride, nb, b->s));
			TRY("D2H len", cudaMemcpyAsync(h_out_len + done, d_olen, nb * 4, cudaMemcpyDeviceToHost, b->s));
			TRY("D2H status", cudaMemcpyAsync(h_status + done, d_st, nb * 4, cudaMemcpyDeviceToHost, b->s));
		}
	}
out:
	if (c)
		for (k = 0; k < PIPE; k++) {
			int e = slot_drain(&c->sl[k]);
			if (!e)
				e = (int)cudaStreamSynchronize(c->sl[k].s);
			if (e && !rc)
				rc = set_err("sync", e);
		}
	ctx_release(c);
	return rc;
}

/* ---- block_compressor-style container on host buffers ----------------------------------
 * Layout (reference block_compressor.c:275-394):
 *     [u32 nr_pages][u32 clen[nr_pages]][payload_0]...[payload_{nr_pages-1}]
 * payload_i is csnappy_compress_fragment(page_i, wm) or, when that is not smaller than the
 * page, the page itself with clen_i = its length (:316-318); the reader treats
 * clen_i == page_size as stored (:378).  Pages are compressed, size-scanned and packed on the
 * device chunk by chunk (compress pipeline above); only COMPRESSED bytes cross the bus on the
 * compressed side.
 */
uint64_t csnappy_bc_max_container_length(uint64_t input_length, uint32_t page_size)
{
	uint64_t nr = page_size ? (input_length + page_size - 1) / page_size : 0;
	return 4 + 4 * nr + input_length;
}

static int bc_compress(const void *h_in, uint64_t input_length, uint32_t page_size, void *h_container,
		       uint64_t container_capacity, uint64_t *container_length, int wm, const int *devs, int G)
{
	uint64_t nr;
	uint8_t *cont = (uint8_t *)h_container;
	struct cjob j;
	struct hostreg r1, r2;
	int rc;
	if (wm < 9 || wm > 16)
		return set_err("workmem_bytes_power_of_two outside 9..16", 0);
	if (page_size == 0 || page_size > CSB_FRAGMENT_MAX)
		return set_err("page_size outside 1..32768", 0);
	nr = (input_length + page_size - 1) / page_size;
	if (nr > 0xffffffffull)
		return set_err("input too big", 0);
	if (!h_container || !container_length || (input_length && !h_in) ||
	    container_capacity < csnappy_bc_max_container_length(input_length, page_size))
		return set_err("container buffer missing or smaller than csnappy_bc_max_container_length", 0);
	{
		uint32_t nr32 = (uint32_t)nr;
		memcpy(cont, &nr32, 4);
	}
	*container_length = 4 + 4 * nr;
	if (nr == 0)
		return 0;
	memset(&j, 0, sizeof(j));
	j.in = (const uint8_t *)h_in;
	j.in_len = input_length;
	j.page = page_size;
	j.wm = wm;
	j.stored = 1;
	j.index_out = cont + 4;
	j.payload_out = cont + 4 + 4 * nr;
	j.nr = nr;
	j.G = G;
	j.devs = devs;
	j.chunk = chunk_units(page_size, nr, G);
	j.n_chunks = (nr + j.chunk - 1) / j.chunk;
	hostreg_begin(&r1, h_in, input_length);
	hostreg_begin(&r2, h_container, container_capacity);
	j.in_pageable = is_pageable(h_in);
	j.out_pageable = is_pageable(h_container);
	rc = run_cjob(&j);
	hostreg_end(&r1);
	hostreg_end(&r2);
	if (rc)
		return rc;
	*container_length = 4 + 4 * nr + j.pos;
	return 0;
}

int csnappy_bc_compress_host(const void *h_in, uint64_t input_length, uint32_t page_size, void *h_container,
			     uint64_t container_capacity, uint64_t *container_length,
			     int workmem_bytes_power_of_two)
{
	return bc_compress(h_in, input_length, page_size, h_container, container_capacity, container_length,
			   workmem_bytes_power_of_two, NULL, 1);
}

int csnappy_bc_compress_host_multi(const void *h_in, uint64_t input_length, uint32_t page_size, void *h_container,
				   uint64_t container_capacity, uint64_t *container_length,
				   int workmem_bytes_power_of_two, const int *devices, int n_devices)
{
	int list[MAX_DEV], G = resolve_devices(devices, n_devices, list);
	if (G < 0)
		return G;
	return bc_compress(h_in, input_length, page_size, h_container, container_capacity, container_length,
			   workmem_bytes_power_of_two, list, G);
}

/* ---- container reader: chunks of pages, chunk c on device c mod G; positions come from the index ---------- */
struct djob {
	const uint8_t *cont;
	const uint8_t *idx; /* u32 per page (any alignment) */
	uint32_t page, chunk;
	uint8_t *out;
	uint64_t nr; /* pages to decode (up to the first malformed index entry) */
	uint64_t n_chunks;
	const uint64_t *chunk_at;     /* container offset of each chunk's first payload byte (n_chunks + 1) */
	const uint32_t *chunk_longest; /* longest compressed page of each chunk */
	int G;
	const int *devs;
	int in_pageable, out_pageable; /* stage the chunks through pinned slot buffers (see par_memcpy) */
	pthread_mutex_t mu;
	int first_err;
	uint64_t err_page, produced;
	int err;
	char errtext[256];
};

struct dworker {
	struct djob *j;
	int g;
	pthread_t th;
};

static void djob_fail(struct djob *j, int rc)
{
	pthread_mutex_lock(&j->mu);
	if (!j->err) {
		j->err = rc;
		memcpy(j->errtext, tls_err, sizeof(j->errtext));
	}
	pthread_mutex_unlock(&j->mu);
}

static void *decompress_worker(void *arg)
{
	struct dworker *w = (struct dworker *)arg;
	struct djob *j = w->j;
	struct ctx *c = NULL;
	const uint32_t max_clen = csnappy_max_compressed_length(j->page);
	const uint64_t n_mine = (uint64_t)w->g < j->n_chunks ? (j->n_chunks - (uint64_t)w->g + (uint64_t)j->G - 1) / (uint64_t)j->G : 0;
	uint64_t issued = 0, retired = 0;
	int rc = 0, k;
	if (j->devs)
		TRY("cudaSetDevice", cudaSetDevice(j->devs[w->g]));
	if (n_mine == 0)
		return NULL;
	TRY("context", ctx_acquire(&c));
	for (k = 0; k < PIPE && (uint64_t)k < n_mine; k++) {
		struct slot *b = &c->sl[k];
		TRY("cudaMalloc(packed)", grow_dev_retry(&b->d_packed, (size_t)j->chunk * max_clen + 64));
		TRY("cudaMalloc(clen)", grow_dev_retry(&b->d_clen, (size_t)j->chunk * 4 + 64));
		TRY("cudaMalloc(off)", grow_dev_retry(&b->d_off, ((size_t)j->chunk + 1) * 8 + 64));
		TRY("cudaMalloc(out)", grow_dev_retry(&b->d_out, (size_t)j->chunk * j->page + 64));
		TRY("cudaMalloc(res)", grow_dev_retry(&b->d_res, (size_t)j->chunk * 8 + 64));
		TRY("cudaMallocHost(res)", grow_pin(&b->h_res, (size_t)j->chunk * 8 + 64));
		TRY("cudaMalloc(ctr)", grow_dev_retry(&b->d_ctr, 64));
		if (j->in_pageable)
			TRY("cudaMallocHost(in)", grow_pin(&b->h_in, (size_t)j->chunk * max_clen + 64));
		if (j->out_pageable)
			TRY("cudaMallocHost(out)", grow_pin(&b->h_out, (size_t)j->chunk * j->page + 64));
	}
	while (retired < n_mine) {
		if (j->err)
			goto out;
		if (retired < issued && (issued - retired >= PIPE || issued == n_mine)) {
			struct slot *b = &c->sl[retired % PIPE];
			const uint32_t *olen = (const uint32_t *)b->h_res.p;
			const int32_t *st = (const int32_t *)b->h_res.p + b->n;
			uint64_t produced = 0, bad_page = 0;
			int bad = 0;
			uint32_t i;
			TRY("sync", cudaStreamSynchronize(b->s));
			if (j->out_pageable)
				par_memcpy(j->out + b->first * j->page, b->h_out.p, (size_t)b->n * j->page);
			for (i = 0; i < b->n; i++) {
				if (st[i] != 0 && !bad) {
					bad = st[i];
					bad_page = b->first + i;
				}
				produced += olen[i];
			}
			pthread_mutex_lock(&j->mu);
			j->produced += produced;
			if (bad && (!j->first_err || bad_page < j->err_page)) {
				j->first_err = bad;
				j->err_page = bad_page;
			}
			pthread_mutex_unlock(&j->mu);
			retired++;
			continue;
		}
		{
			struct slot *b = &c->sl[issued % PIPE];
			const uint64_t gc = (uint64_t)w->g + issued * (uint64_t)j->G;
			const uint64_t first = gc * j->chunk, left_pages = j->nr - first;
			const uint32_t nb = left_pages < j->chunk ? (uint32_t)left_pages : j->chunk;
			const uint64_t bytes = j->chunk_at[gc + 1] - j->chunk_at[gc];
			struct csb_decompress_args a;
			if (bytes && j->in_pageable) {
				par_memcpy(b->h_in.p, j->cont + j->chunk_at[gc], bytes);
				TRY("H2D payload", cudaMemcpyAsync(b->d_packed.p, b->h_in.p, bytes, cudaMemcpyHostToDevice, b->s));
			} else if (bytes) {
				TRY("H2D payload", cudaMemcpyAsync(b->d_packed.p, j->cont + j->chunk_at[gc], bytes, cudaMemcpyHostToDevice, b->s));
			}
			TRY("H2D index", cudaMemcpyAsync(b->d_clen.p, j->idx + 4 * first, (size_t)nb * 4, cudaMemcpyHostToDevice, b->s));
			TRY("scan launch", csb_launch_scan((const uint32_t *)b->d_clen.p, nb, (uint64_t *)b->d_off.p, (csb_stream_t)b->s));
			fill_decompress_args(&a);
			a.in = (const uint8_t *)b->d_packed.p;
			a.in_off = (const uint64_t *)b->d_off.p;
			a.in_len = (const uint32_t *)b->d_clen.p;
			a.n_blocks = nb;
			a.out = (uint8_t *)b->d_out.p;
			a.out_stride = j->page;
			a.uniform_cap = j->page;
			a.out_len = (uint32_t *)b->d_res.p;
			a.status = (int32_t *)b->d_res.p + nb;
			a.flags = CSNAPPY_BATCH_RAW_IF_FULL;
			a.max_in_len = j->chunk_longest[gc];
			a.counter = (uint32_t *)b->d_ctr.p;
			TRY("decompress launch", csb_launch_decompress(&a, (csb_stream_t)b->s));
			TRY("D2H pages", cudaMemcpyAsync(j->out_pageable ? (uint8_t *)b->h_out.p : j->out + first * j->page, b->d_out.p,
							 (size_t)nb * j->page, cudaMemcpyDeviceToHost, b->s));
			TRY("D2H result", cudaMemcpyAsync(b->h_res.p, b->d_res.p, (size_t)nb * 8, cudaMemcpyDeviceToHost, b->s));
			b->first = first;
			b->n = nb;
			issued++;
		}
	}
out:
	if (c)
		for (k = 0; k < PIPE; k++)
			cudaStreamSynchronize(c->sl[k].s);
	if (rc)
		djob_fail(j, rc);
	ctx_release(c);
	return NULL;
}

static int bc_decompress(const void *h_container, uint64_t container_length, uint32_t page_size, void *h_out,
			 uint64_t out_capacity, uint64_t *out_length, uint32_t *failed_page, const int *devs, int G)
{
	const uint8_t *cont = (const uint8_t *)h_container;
	uint32_t nr32 = 0, max_clen;
	uint64_t nr, i, ipos, n_chunks;
	uint64_t *chunk_at = NULL;
	uint32_t *chunk_longest = NULL;
	struct djob j;
	struct dworker w[MAX_DEV];
	struct hostreg r1, r2;
	int rc = 0, g, index_err = 0;
	uint64_t index_err_page = 0;
	if (page_size == 0 || page_size > CSB_FRAGMENT_MAX)
		return set_err("page_size outside 1..32768", 0);
	if (!h_container || !out_length || container_length < 4)
		return set_err("container missing or shorter than its header", 0);
	memcpy(&nr32, cont, 4);
	nr = nr32;
	if (container_length < 4 + 4 * nr)
		return CSNAPPY_E_DATA_MALFORMED;
	if (out_capacity < nr * page_size || (nr && !h_out))
		return CSNAPPY_E_OUTPUT_INSUF;
	*out_length = 0;
	if (nr == 0)
		return 0;
	max_clen = csnappy_max_compressed_length(page_size);
	memset(&j, 0, sizeof(j));
	j.cont = cont;
	j.idx = cont + 4;
	j.page = page_size;
	j.out = (uint8_t *)h_out;
	j.G = G;
	j.devs = devs;
	j.chunk = chunk_units(page_size, nr, G);
	n_chunks = (nr + j.chunk - 1) / j.chunk;
	chunk_at = (uint64_t *)malloc((size_t)(n_chunks + 1) * 8);
	chunk_longest = (uint32_t *)calloc((size_t)n_chunks, 4);
	if (!chunk_at || !chunk_longest) {
		free(chunk_at);
		free(chunk_longest);
		return set_err("host index", (int)cudaErrorMemoryAllocation);
	}
	/* payload positions from the index; a size no writer produces, or a payload past the end of the container,
	 * ends the decodable prefix (pages before it are still decoded: an earlier failing page wins) */
	ipos = 4 + 4 * nr;
	j.nr = nr;
	for (i = 0; i < nr; i++) {
		uint32_t cl;
		if (i % j.chunk == 0)
			chunk_at[i / j.chunk] = ipos;
		memcpy(&cl, j.idx + 4 * i, 4);
		if (cl > max_clen || ipos + cl > container_length) {
			index_err = CSNAPPY_E_DATA_MALFORMED;
			index_err_page = i;
			j.nr = i;
			break;
		}
		if (cl > chunk_longest[i / j.chunk])
			chunk_longest[i / j.chunk] = cl;
		ipos += cl;
	}
	j.n_chunks = (j.nr + j.chunk - 1) / j.chunk;
	chunk_at[j.n_chunks] = ipos;
	j.chunk_at = chunk_at;
	j.chunk_longest = chunk_longest;
	pthread_mutex_init(&j.mu, NULL);
	hostreg_begin(&r1, h_container, container_length);
	hostreg_begin(&r2, h_out, j.nr * page_size);
	j.in_pageable = is_pageable(h_container);
	j.out_pageable = is_pageable(h_out);
	if (j.n_chunks) {
		if (!devs) {
			w[0].j = &j;
			w[0].g = 0;
			decompress_worker(&w[0]);
		} else {
			int started = 0;
			for (g = 0; g < G; g++) {
				w[g].j = &j;
				w[g].g = g;
				if (pthread_create(&w[g].th, NULL, decompress_worker, &w[g])) {
					set_err("pthread_create", (int)cudaErrorUnknown);
					djob_fail(&j, CSNAPPY_E_DEVICE);
					break;
				}
				started++;
			}
			for (g = 0; g < started; g++)
				pthread_join(w[g].th, NULL);
		}
	}
	hostreg_end(&r1);
	hostreg_end(&r2);
	pthread_mutex_destroy(&j.mu);
	free(chunk_at);
	free(chunk_longest);
	if (j.err) {
		memcpy(tls_err, j.errtext, sizeof(tls_err));
		return j.err;
	}
	*out_length = j.produced;
	if (index_err && (!j.first_err || index_err_page < j.err_page)) {
		j.first_err = index_err;
		j.err_page = index_err_page;
	}
	if (j.first_err) {
		if (failed_page)
			*failed_page = (uint32_t)j.err_page;
		rc = j.first_err;
	}
	return rc;
}

int csnappy_bc_decompress_host(const void *h_container, uint64_t container_length, uint32_t page_size, void *h_out,
			       uint64_t out_capacity, uint64_t *out_length, uint32_t *failed_page)
{
	return bc_decompress(h_container, container_length, page_size, h_out, out_capacity, out_length, failed_page, NULL, 1);
}

int csnappy_bc_decompress_host_multi(const void *h_container, uint64_t container_length, uint32_t page_size, void *h_out,
				     uint64_t out_capacity, uint64_t *out_length, uint32_t *failed_page,
				     const int *devices, int n_devices)
{
	int list[MAX_DEV], G = resolve_devices(devices, n_devices, list);
	if (G < 0)
		return G;
	return bc_decompress(h_container, container_length, page_size, h_out, out_capacity, out_length, failed_page, list, G);
}

/* ---- the same container on DEVICE buffers (csnappy_bc_compress / _index / _decompress_pages / _decompress) ---------
 * Writer: one compress launch over every page (total_len clips the short last page), the stored-page rule
 * (csb_launch_clamp), the grid-wide index scan for the payload offsets, the gather of fragments and stored pages to
 * their offsets, and the header and index at d_container (bc_kernel.cu; any alignment).
 * Readers: the page count is read back (one synchronisation); the index scan gives each page's payload offset, or
 * CSNAPPY_BC_NO_PAGE from the first malformed entry on.  A batch of page requests gathers (offset, length) per request
 * and runs the batched decoder on those; the whole-container read runs the decoder on every page with the index as
 * its offsets, and a finish step reduces the page results to the host reader's (status, out_length, failed_page). */
#define BC_MAX_PAGES 0xffffffffull

static uint64_t bc_pages_of(uint64_t input_length, uint32_t page) { return input_length / page + (input_length % page != 0); }

static uint64_t bc_slot(uint32_t page) { return ((uint64_t)csnappy_max_compressed_length(page) + 15) & ~(uint64_t)15; }

static int bc_page_size_ok(uint32_t page) { return page >= 1 && page <= CSB_FRAGMENT_MAX; }

/* writer workspace: fragment slots | fragment sizes | stored-rule sizes | payload offsets | claim counter */
static uint64_t bc_compress_layout(uint64_t nr, uint32_t page, uint64_t *o_len, uint64_t *o_clen, uint64_t *o_off,
				   uint64_t *o_ctr)
{
	uint64_t p = al256(nr * bc_slot(page));
	*o_len = p;
	p = al256(p + nr * 4);
	*o_clen = p;
	p = al256(p + nr * 4);
	*o_off = p;
	p = al256(p + nr * 8);
	*o_ctr = p;
	return p + 256;
}

uint64_t csnappy_bc_compress_workspace(uint64_t input_length, uint32_t page_size)
{
	uint64_t nr, a, b, c, d;
	if (!bc_page_size_ok(page_size))
		return UINT64_MAX;
	nr = bc_pages_of(input_length, page_size);
	if (nr > BC_MAX_PAGES)
		return UINT64_MAX;
	return bc_compress_layout(nr, page_size, &a, &b, &c, &d);
}

int csnappy_bc_compress(const void *d_in, uint64_t input_length, uint32_t page_size, void *d_container,
			uint64_t container_capacity, uint64_t *d_container_length, int workmem_bytes_power_of_two,
			void *d_workspace, uint64_t workspace_bytes, void *stream)
{
	uint64_t nr, o_len, o_clen, o_off, o_ctr;
	uint8_t *ws = (uint8_t *)d_workspace;
	csb_stream_t s = (csb_stream_t)stream;
	struct csb_compress_args a;
	int e;
	if (workmem_bytes_power_of_two < 9 || workmem_bytes_power_of_two > 16)
		return set_err("workmem_bytes_power_of_two outside 9..16", 0);
	if (!bc_page_size_ok(page_size))
		return set_err("page_size outside 1..32768", 0);
	nr = bc_pages_of(input_length, page_size);
	if (nr > BC_MAX_PAGES)
		return set_err("more than 2^32 - 1 pages", 0);
	if (!d_container || !d_container_length || !d_workspace || (input_length && !d_in))
		return set_err("null buffer", 0);
	if (container_capacity < csnappy_bc_max_container_length(input_length, page_size))
		return set_err("container_capacity smaller than csnappy_bc_max_container_length()", 0);
	if (workspace_bytes < bc_compress_layout(nr, page_size, &o_len, &o_clen, &o_off, &o_ctr))
		return set_err("workspace smaller than csnappy_bc_compress_workspace()", 0);
	if (nr) {
		fill_compress_args(&a);
		a.in = (const uint8_t *)d_in;
		a.in_stride = page_size;
		a.uniform_len = page_size;
		a.total_len = input_length;
		a.n_blocks = (uint32_t)nr;
		a.out = ws;
		a.out_stride = bc_slot(page_size);
		a.out_len = (uint32_t *)(ws + o_len);
		a.wm = workmem_bytes_power_of_two;
		a.counter = (uint32_t *)(ws + o_ctr);
		if ((e = csb_launch_compress(&a, s)))
			return set_err("compress launch", e);
		if ((e = csb_launch_clamp((const uint32_t *)(ws + o_len), (uint32_t)nr, page_size, input_length,
					  (uint32_t *)(ws + o_clen), s)))
			return set_err("clamp launch", e);
		/* every size is valid here: no bound, no room limit */
		if ((e = csb_launch_bc_index(ws + o_clen, (uint32_t)nr, 0xffffffffu, 4 + 4 * nr, UINT64_MAX, 0,
					     (uint64_t *)(ws + o_off), NULL, NULL, s)))
			return set_err("index launch", e);
		if ((e = csb_launch_gather(ws, bc_slot(page_size), (const uint32_t *)(ws + o_clen), (uint32_t)nr,
					   (uint8_t *)d_container, (const uint64_t *)(ws + o_off), (const uint8_t *)d_in, page_size,
					   input_length, (const uint32_t *)(ws + o_len), s)))
			return set_err("gather launch", e);
	}
	e = csb_launch_bc_header((const uint32_t *)(ws + o_clen), (uint32_t)nr, (const uint64_t *)(ws + o_off),
				 (uint8_t *)d_container, d_container_length, s);
	return e ? set_err("header launch", e) : 0;
}

/* the page count at the container's start: the readers' one synchronisation */
static int bc_read_count(const void *d_container, uint32_t *nr, cudaStream_t s)
{
	int e;
	if ((e = (int)cudaMemcpyAsync(nr, d_container, 4, cudaMemcpyDeviceToHost, s)) || (e = (int)cudaStreamSynchronize(s)))
		return set_err("D2H page count", e);
	return 0;
}

int csnappy_bc_index(const void *d_container, uint64_t container_length, uint32_t page_size, uint64_t *d_index,
		     uint64_t index_entries, uint32_t *nr_pages, void *stream)
{
	uint32_t nr = 0;
	int e;
	if (!bc_page_size_ok(page_size))
		return set_err("page_size outside 1..32768", 0);
	if (!d_container || !nr_pages || container_length < 4)
		return set_err("container missing or shorter than its header", 0);
	if (index_entries && !d_index)
		return set_err("null buffer", 0);
	if ((e = bc_read_count(d_container, &nr, (cudaStream_t)stream)))
		return e;
	*nr_pages = nr;
	if (container_length < 4 + 4 * (uint64_t)nr)
		return CSNAPPY_E_DATA_MALFORMED;
	if (index_entries < nr)
		return set_err("index_entries smaller than the page count", 0);
	e = csb_launch_bc_index((const uint8_t *)d_container + 4, nr, csnappy_max_compressed_length(page_size),
				4 + 4 * (uint64_t)nr, container_length - 4 - 4 * (uint64_t)nr, CSNAPPY_BC_NO_PAGE, d_index,
				NULL, NULL, (csb_stream_t)stream);
	return e ? set_err("index launch", e) : 0;
}

/* page reads workspace: decoder offsets | decoder lengths | request tags | claim counter */
static uint64_t bc_pages_layout(uint64_t n, uint64_t *o_len, uint64_t *o_tag, uint64_t *o_ctr)
{
	uint64_t p = al256(n * 8);
	*o_len = p;
	p = al256(p + n * 4);
	*o_tag = p;
	p = al256(p + n * 4);
	*o_ctr = p;
	return p + 256;
}

uint64_t csnappy_bc_decompress_pages_workspace(uint32_t n_requests)
{
	uint64_t a, b, c;
	return bc_pages_layout(n_requests, &a, &b, &c);
}

int csnappy_bc_decompress_pages(const void *d_container, uint64_t container_length, uint32_t page_size,
				const uint64_t *d_index, uint32_t nr_pages, const uint32_t *d_pages, uint32_t n_requests,
				void *d_out, uint64_t out_stride, uint32_t *d_out_len, int32_t *d_status,
				void *d_workspace, uint64_t workspace_bytes, void *stream)
{
	uint64_t o_len, o_tag, o_ctr;
	uint8_t *ws = (uint8_t *)d_workspace;
	csb_stream_t s = (csb_stream_t)stream;
	struct csb_decompress_args a;
	int e;
	if (!bc_page_size_ok(page_size))
		return set_err("page_size outside 1..32768", 0);
	if (out_stride < page_size)
		return set_err("out_stride smaller than page_size", 0);
	if (n_requests == 0)
		return 0;
	if (!d_container || !d_pages || !d_out || !d_out_len || !d_status || !d_workspace || (nr_pages && !d_index))
		return set_err("null buffer", 0);
	if (container_length < 4 + 4 * (uint64_t)nr_pages)
		return set_err("container shorter than the index of nr_pages pages", 0);
	if (workspace_bytes < bc_pages_layout(n_requests, &o_len, &o_tag, &o_ctr))
		return set_err("workspace smaller than csnappy_bc_decompress_pages_workspace()", 0);
	if ((e = csb_launch_bc_requests((const uint8_t *)d_container, container_length, csnappy_max_compressed_length(page_size),
					d_index, nr_pages, d_pages, n_requests, (uint64_t *)ws, (uint32_t *)(ws + o_len),
					(int32_t *)(ws + o_tag), s)))
		return set_err("request launch", e);
	fill_decompress_args(&a);
	a.in = (const uint8_t *)d_container;
	a.in_off = (const uint64_t *)ws;
	a.in_len = (const uint32_t *)(ws + o_len);
	a.n_blocks = n_requests;
	a.out = (uint8_t *)d_out;
	a.out_stride = out_stride;
	a.uniform_cap = page_size;
	a.out_len = d_out_len;
	a.status = d_status;
	a.flags = CSNAPPY_BATCH_RAW_IF_FULL;
	a.counter = (uint32_t *)(ws + o_ctr);
	if ((e = csb_launch_decompress(&a, s)))
		return set_err("decompress launch", e);
	e = csb_launch_bc_request_status((const int32_t *)(ws + o_tag), n_requests, d_out_len, d_status, s);
	return e ? set_err("request status launch", e) : 0;
}

/* whole-container workspace, for the most pages a container of this length and an output of this capacity can take:
 * index | decoder lengths | page out_len | page status | result words | claim counter */
static uint64_t bc_decompress_layout(uint64_t container_length, uint32_t page, uint64_t out_capacity, uint64_t *o_len,
				     uint64_t *o_olen, uint64_t *o_st, uint64_t *o_res, uint64_t *o_ctr)
{
	uint64_t n = container_length >= 4 ? (container_length - 4) / 4 : 0, p;
	if (n > out_capacity / page)
		n = out_capacity / page;
	if (n > BC_MAX_PAGES)
		n = BC_MAX_PAGES;
	p = al256(n * 8);
	*o_len = p;
	p = al256(p + n * 4);
	*o_olen = p;
	p = al256(p + n * 4);
	*o_st = p;
	p = al256(p + n * 4);
	*o_res = p;
	p = al256(p + sizeof(struct csb_bc_result));
	*o_ctr = p;
	return p + 256;
}

uint64_t csnappy_bc_decompress_workspace(uint64_t container_length, uint32_t page_size, uint64_t out_capacity)
{
	uint64_t a, b, c, d, e;
	if (!bc_page_size_ok(page_size))
		return UINT64_MAX;
	return bc_decompress_layout(container_length, page_size, out_capacity, &a, &b, &c, &d, &e);
}

int csnappy_bc_decompress(const void *d_container, uint64_t container_length, uint32_t page_size, void *d_out,
			  uint64_t out_capacity, uint64_t *d_out_length, int32_t *d_status, uint32_t *d_failed_page,
			  void *d_workspace, uint64_t workspace_bytes, void *stream)
{
	uint64_t o_len, o_olen, o_st, o_res, o_ctr;
	uint8_t *ws = (uint8_t *)d_workspace;
	cudaStream_t s = (cudaStream_t)stream;
	struct csb_bc_result *res;
	struct csb_decompress_args a;
	uint32_t nr = 0;
	int32_t hdr = 0;
	int e;
	if (!bc_page_size_ok(page_size))
		return set_err("page_size outside 1..32768", 0);
	if (!d_container || container_length < 4)
		return set_err("container missing or shorter than its header", 0);
	if (!d_out_length || !d_status || !d_workspace || (out_capacity && !d_out))
		return set_err("null buffer", 0);
	if (workspace_bytes < bc_decompress_layout(container_length, page_size, out_capacity, &o_len, &o_olen, &o_st, &o_res, &o_ctr))
		return set_err("workspace smaller than csnappy_bc_decompress_workspace()", 0);
	res = (struct csb_bc_result *)(ws + o_res);
	if ((e = bc_read_count(d_container, &nr, s)))
		return e;
	if (container_length < 4 + 4 * (uint64_t)nr)
		hdr = CSNAPPY_E_DATA_MALFORMED;
	else if (out_capacity < (uint64_t)nr * page_size)
		hdr = CSNAPPY_E_OUTPUT_INSUF;
	if (!hdr && nr) {
		if ((e = (int)cudaMemsetAsync(res, 0xff, offsetof(struct csb_bc_result, sum), s)) ||
		    (e = (int)cudaMemsetAsync(&res->sum, 0, sizeof(res->sum), s)))
			return set_err("result words", e);
		/* pages behind the prefix decode an empty block at the container start: no output, and the finish step
		 * does not count them */
		if ((e = csb_launch_bc_index((const uint8_t *)d_container + 4, nr, csnappy_max_compressed_length(page_size),
					     4 + 4 * (uint64_t)nr, container_length - 4 - 4 * (uint64_t)nr, 0, (uint64_t *)ws,
					     (uint32_t *)(ws + o_len), &res->prefix, (csb_stream_t)s)))
			return set_err("index launch", e);
		fill_decompress_args(&a);
		a.in = (const uint8_t *)d_container;
		a.in_off = (const uint64_t *)ws;
		a.in_len = (const uint32_t *)(ws + o_len);
		a.n_blocks = nr;
		a.out = (uint8_t *)d_out;
		a.out_stride = page_size;
		a.uniform_cap = page_size;
		a.out_len = (uint32_t *)(ws + o_olen);
		a.status = (int32_t *)(ws + o_st);
		a.flags = CSNAPPY_BATCH_RAW_IF_FULL;
		a.counter = (uint32_t *)(ws + o_ctr);
		if ((e = csb_launch_decompress(&a, (csb_stream_t)s)))
			return set_err("decompress launch", e);
	}
	e = csb_launch_bc_finish((const uint32_t *)(ws + o_olen), (const int32_t *)(ws + o_st), nr, hdr, res, d_out_length,
				 d_status, d_failed_page, (csb_stream_t)s);
	return e ? set_err("finish launch", e) : 0;
}

/* ---- Snappy framing format (include/csnappy_batch.h csnappy_framed_*; kernels in framed_kernel.cu) ------------------
 * Writer: ONE compress launch over the whole input as 32 KiB fragments (only the global last fragment is short, and it
 * gets csnappy_compress()'s short-chunk table rule), so fragments 2k and 2k+1 behind a varint are exactly
 * csnappy_compress(chunk k).  Then one warp per chunk computes its masked CRC-32C and record size, a scan places the
 * records, and one warp per chunk writes header, CRC and payload.
 * Reader: one thread walks the chunk headers (a dependent chain) into a table of data chunks; the host reads the
 * counts back to size the launches; the batched decoder writes every compressed chunk straight to its output offset;
 * one warp per data chunk copies stored chunks and checks lengths and CRCs; one thread writes the result.           */
#define FRAMED_CHUNK ((uint64_t)CSB_FRAMED_CHUNK)
#define FRAMED_IDENT 10u

static uint64_t chunks_of(uint64_t n) { return (n + FRAMED_CHUNK - 1) / FRAMED_CHUNK; }

uint64_t csnappy_framed_max_length(uint64_t input_length)
{
	return FRAMED_IDENT + 8 * chunks_of(input_length) + input_length;
}

/* workspace of the writer: fragment slots | fragment sizes | crc | record sizes | record offsets | counter */
static uint64_t framed_compress_layout(uint64_t n, uint64_t *o_flen, uint64_t *o_crc, uint64_t *o_rec, uint64_t *o_off,
				       uint64_t *o_ctr)
{
	const uint64_t F = (n + CSB_FRAGMENT_MAX - 1) / CSB_FRAGMENT_MAX, K = chunks_of(n);
	uint64_t p = al256(F * SLOT_STRIDE_32K);
	*o_flen = p;
	p = al256(p + F * 4);
	*o_crc = p;
	p = al256(p + K * 4);
	*o_rec = p;
	p = al256(p + K * 4);
	*o_off = p;
	p = al256(p + (K + 1) * 8);
	*o_ctr = p;
	return p + 256;
}

uint64_t csnappy_framed_compress_workspace(uint64_t input_length)
{
	uint64_t a, b, c, d, e;
	return framed_compress_layout(input_length, &a, &b, &c, &d, &e);
}

/* the longest input: 2^32 - 1 fragments of 32 KiB for the compress launch */
#define FRAMED_MAX_INPUT (((uint64_t)0xffffffffu - 1) * CSB_FRAGMENT_MAX)

int csnappy_framed_compress(const void *d_in, uint64_t input_length, void *d_out, uint64_t out_capacity,
			    uint64_t *d_out_length, int workmem_bytes_power_of_two, void *d_workspace, uint64_t workspace_bytes,
			    void *stream)
{
	uint64_t o_flen, o_crc, o_rec, o_off, o_ctr, need;
	const uint64_t F = (input_length + CSB_FRAGMENT_MAX - 1) / CSB_FRAGMENT_MAX;
	uint8_t *ws = (uint8_t *)d_workspace;
	csb_stream_t s = (csb_stream_t)stream;
	struct csb_compress_args a;
	int e;
	if (workmem_bytes_power_of_two < 9 || workmem_bytes_power_of_two > 16)
		return set_err("workmem_bytes_power_of_two outside 9..16", 0);
	if (input_length > FRAMED_MAX_INPUT)
		return set_err("input longer than (2^32 - 2) * 32768 bytes", 0);
	if ((input_length && !d_in) || !d_out || !d_out_length || !d_workspace)
		return set_err("null buffer", 0);
	if (out_capacity < csnappy_framed_max_length(input_length))
		return set_err("out_capacity smaller than csnappy_framed_max_length()", 0);
	need = framed_compress_layout(input_length, &o_flen, &o_crc, &o_rec, &o_off, &o_ctr);
	if (workspace_bytes < need)
		return set_err("workspace smaller than csnappy_framed_compress_workspace()", 0);
	if (F) {
		fill_compress_args(&a);
		a.in = (const uint8_t *)d_in;
		a.in_stride = CSB_FRAGMENT_MAX;
		a.uniform_len = CSB_FRAGMENT_MAX;
		a.total_len = input_length;
		a.n_blocks = (uint32_t)F;
		a.out = ws;
		a.out_stride = SLOT_STRIDE_32K;
		a.out_len = (uint32_t *)(ws + o_flen);
		a.wm = workmem_bytes_power_of_two;
		a.flags = CSNAPPY_BATCH_SHRINK_TABLE;
		a.counter = (uint32_t *)(ws + o_ctr);
		if ((e = csb_launch_compress(&a, s)))
			return set_err("compress launch", e);
		if ((e = csb_launch_framed_crc((const uint8_t *)d_in, input_length, (uint32_t *)(ws + o_crc),
					       (const uint32_t *)(ws + o_flen), (uint32_t)F, (uint32_t *)(ws + o_rec), s)))
			return set_err("crc launch", e);
	}
	if ((e = csb_launch_scan((const uint32_t *)(ws + o_rec), (uint32_t)chunks_of(input_length), (uint64_t *)(ws + o_off), s)))
		return set_err("scan launch", e);
	e = csb_launch_framed_write((const uint8_t *)d_in, input_length, ws, SLOT_STRIDE_32K, (const uint32_t *)(ws + o_flen),
				    (uint32_t)F, (const uint32_t *)(ws + o_crc), (const uint32_t *)(ws + o_rec),
				    (const uint64_t *)(ws + o_off), (uint8_t *)d_out, d_out_length, s);
	return e ? set_err("framed write launch", e) : 0;
}

int csnappy_framed_crc32c(const void *d_in, uint64_t length, uint32_t *d_crc, void *stream)
{
	int e;
	if (length > FRAMED_MAX_INPUT)
		return set_err("input longer than (2^32 - 2) * 32768 bytes", 0);
	if (length && (!d_in || !d_crc))
		return set_err("null buffer", 0);
	e = csb_launch_framed_crc((const uint8_t *)d_in, length, d_crc, NULL, 0, NULL, (csb_stream_t)stream);
	return e ? set_err("crc launch", e) : 0;
}

/* Reader workspace: result words, then the tables of csb_framed_table for at most src_length / 8 + 1 data chunks (a
 * data chunk takes at least 8 bytes of the stream), then the decoder's block counter. */
#define FRAMED_MAX_SRC ((uint64_t)0xfffffffeu * 8)

static uint64_t framed_decompress_layout(uint64_t src_length, struct csb_framed_table *t, uint8_t *ws, uint32_t **ctr)
{
	const uint64_t D = src_length / 8 + 1;
	uint64_t p = 0;
#define FRAMED_TAB(field, type, per)                              \
	do {                                                      \
		if (t)                                            \
			t->field = (type *)(ws + p);              \
		p = al256(p + (per));                             \
	} while (0)
	FRAMED_TAB(res, struct csb_framed_result, sizeof(struct csb_framed_result));
	FRAMED_TAB(pos, uint64_t, D * 8);
	FRAMED_TAB(out_off, uint64_t, D * 8);
	FRAMED_TAB(out_len, uint32_t, D * 4);
	FRAMED_TAB(crc, uint32_t, D * 4);
	FRAMED_TAB(cidx, uint32_t, D * 4);
	FRAMED_TAB(c_pos, uint64_t, D * 8);
	FRAMED_TAB(c_out_off, uint64_t, D * 8);
	FRAMED_TAB(c_len, uint32_t, D * 4);
	FRAMED_TAB(c_produced, uint32_t, D * 4);
	FRAMED_TAB(c_status, int32_t, D * 4);
#undef FRAMED_TAB
	if (ctr)
		*ctr = (uint32_t *)(ws + p);
	return p + 256;
}

uint64_t csnappy_framed_decompress_workspace(uint64_t src_length)
{
	return framed_decompress_layout(src_length, NULL, NULL, NULL);
}

int csnappy_framed_decompress(const void *d_src, uint64_t src_length, void *d_dst, uint64_t out_capacity,
			      uint64_t *d_out_length, int32_t *d_status, uint64_t *d_failed_offset, void *d_workspace,
			      uint64_t workspace_bytes, void *stream)
{
	struct csb_framed_table t;
	struct csb_framed_result r;
	struct csb_decompress_args a;
	uint32_t *ctr = NULL;
	cudaStream_t s = (cudaStream_t)stream;
	const uint8_t *src = (const uint8_t *)d_src;
	int e;
	if (src_length > FRAMED_MAX_SRC)
		return set_err("src_length above 2^35 bytes", 0);
	if ((src_length && !d_src) || (out_capacity && !d_dst) || !d_out_length || !d_status || !d_workspace)
		return set_err("null buffer", 0);
	if (workspace_bytes < csnappy_framed_decompress_workspace(src_length))
		return set_err("workspace smaller than csnappy_framed_decompress_workspace()", 0);
	framed_decompress_layout(src_length, &t, (uint8_t *)d_workspace, &ctr);
	if ((e = csb_launch_framed_walk(src, src_length, out_capacity, &t, (csb_stream_t)s)))
		return set_err("framed walk launch", e);
	/* the only synchronisation: the chunk counts size the launches below */
	if ((e = (int)cudaMemcpyAsync(&r, t.res, sizeof(r), cudaMemcpyDeviceToHost, s)) || (e = (int)cudaStreamSynchronize(s)))
		return set_err("D2H chunk counts", e);
	if (r.n_comp) {
		fill_decompress_args(&a);
		a.in = src + 8; /* block j = the body behind chunk j's header and CRC */
		a.in_off = t.c_pos;
		a.in_len = t.c_len;
		a.n_blocks = r.n_comp;
		a.out = (uint8_t *)d_dst;
		a.out_off = t.c_out_off;
		a.uniform_cap = CSB_FRAMED_CHUNK; /* WITH_HEADER: the capacity becomes the varint's value, <= 65536 */
		a.out_len = t.c_produced;
		a.status = t.c_status;
		a.flags = CSNAPPY_BATCH_WITH_HEADER;
		a.counter = ctr;
		if ((e = csb_launch_decompress(&a, (csb_stream_t)s)))
			return set_err("decompress launch", e);
	}
	e = csb_launch_framed_verify(src, (uint8_t *)d_dst, r.n_data, &t, d_out_length, d_status, d_failed_offset,
				     (csb_stream_t)s);
	return e ? set_err("framed verify launch", e) : 0;
}

/* Host buffers: the whole input and output staged through one pooled context. */
int csnappy_framed_compress_host(const void *h_in, uint64_t input_length, void *h_out, uint64_t out_capacity,
				 uint64_t *out_length, int workmem_bytes_power_of_two)
{
	int rc = 0;
	struct ctx *c = NULL;
	struct slot *sl;
	uint64_t max_len = csnappy_framed_max_length(input_length), olen = 0;
	if (workmem_bytes_power_of_two < 9 || workmem_bytes_power_of_two > 16)
		return set_err("workmem_bytes_power_of_two outside 9..16", 0);
	if (input_length > FRAMED_MAX_INPUT)
		return set_err("input longer than (2^32 - 2) * 32768 bytes", 0);
	if ((input_length && !h_in) || !h_out || !out_length)
		return set_err("null buffer", 0);
	if (out_capacity < max_len)
		return set_err("out_capacity smaller than csnappy_framed_max_length()", 0);
	TRY("context", ctx_acquire(&c));
	sl = &c->sl[0];
	TRY("cudaMalloc(in)", grow_dev_retry(&sl->d_in, (size_t)input_length + 64));
	TRY("cudaMalloc(out)", grow_dev_retry(&sl->d_out, (size_t)max_len + 64));
	TRY("cudaMalloc(res)", grow_dev_retry(&sl->d_res, 64));
	TRY("cudaMalloc(workspace)", grow_dev_retry(&c->d_aux, (size_t)csnappy_framed_compress_workspace(input_length)));
	if (input_length)
		TRY("H2D", cudaMemcpyAsync(sl->d_in.p, h_in, (size_t)input_length, cudaMemcpyHostToDevice, sl->s));
	rc = csnappy_framed_compress(sl->d_in.p, input_length, sl->d_out.p, max_len, (uint64_t *)sl->d_res.p,
				     workmem_bytes_power_of_two, c->d_aux.p, c->d_aux.cap, sl->s);
	if (rc)
		goto out;
	TRY("D2H length", cudaMemcpyAsync(&olen, sl->d_res.p, 8, cudaMemcpyDeviceToHost, sl->s));
	TRY("sync", cudaStreamSynchronize(sl->s));
	TRY("D2H data", cudaMemcpyAsync(h_out, sl->d_out.p, (size_t)olen, cudaMemcpyDeviceToHost, sl->s));
	TRY("sync", cudaStreamSynchronize(sl->s));
	*out_length = olen;
out:
	ctx_release(c);
	return rc;
}

int csnappy_framed_decompress_host(const void *h_src, uint64_t src_length, void *h_dst, uint64_t out_capacity,
				   uint64_t *out_length, uint64_t *failed_offset)
{
	int rc = 0;
	struct ctx *c = NULL;
	struct slot *sl;
	/* no stream can produce more than 65536 bytes per 9 of its bytes: a larger capacity needs no device memory */
	const uint64_t most = (src_length / 9 + 1) * FRAMED_CHUNK, cap = out_capacity < most ? out_capacity : most;
	struct {
		uint64_t out_length;
		uint64_t failed_offset;
		int32_t status;
		int32_t pad;
	} res = {0, 0, 0, 0};
	if (src_length > FRAMED_MAX_SRC)
		return set_err("src_length above 2^35 bytes", 0);
	if ((src_length && !h_src) || (out_capacity && !h_dst) || !out_length)
		return set_err("null buffer", 0);
	TRY("context", ctx_acquire(&c));
	sl = &c->sl[0];
	TRY("cudaMalloc(in)", grow_dev_retry(&sl->d_in, (size_t)src_length + 64));
	TRY("cudaMalloc(out)", grow_dev_retry(&sl->d_out, (size_t)cap + 64));
	TRY("cudaMalloc(res)", grow_dev_retry(&sl->d_res, 64));
	TRY("cudaMalloc(workspace)", grow_dev_retry(&c->d_aux, (size_t)csnappy_framed_decompress_workspace(src_length)));
	if (src_length)
		TRY("H2D", cudaMemcpyAsync(sl->d_in.p, h_src, (size_t)src_length, cudaMemcpyHostToDevice, sl->s));
	{
		uint8_t *d_res = (uint8_t *)sl->d_res.p;
		rc = csnappy_framed_decompress(sl->d_in.p, src_length, sl->d_out.p, cap, (uint64_t *)d_res, (int32_t *)(d_res + 16),
					       (uint64_t *)(d_res + 8), c->d_aux.p, c->d_aux.cap, sl->s);
		if (rc)
			goto out;
	}
	TRY("D2H result", cudaMemcpyAsync(&res, sl->d_res.p, sizeof(res), cudaMemcpyDeviceToHost, sl->s));
	TRY("sync", cudaStreamSynchronize(sl->s));
	if (res.out_length) {
		TRY("D2H data", cudaMemcpyAsync(h_dst, sl->d_out.p, (size_t)res.out_length, cudaMemcpyDeviceToHost, sl->s));
		TRY("sync", cudaStreamSynchronize(sl->s));
	}
	*out_length = res.out_length;
	rc = res.status;
	if (rc && failed_offset)
		*failed_offset = res.failed_offset;
out:
	ctx_release(c);
	return rc;
}

/* ---- many framed streams in one call (csnappy_framed_batch_*) --------------------------------------------------------
 * Exactly N independent single calls, with a launch count that does not grow with N.
 * Writer: the host lays out every stream's chunks and their 32 KiB fragments (a chunk's short last fragment takes the
 * short-chunk table rule, as csnappy_compress(chunk) does); one compress launch over all fragments, one warp per chunk
 * for CRC and record size, one scan over all records, one warp per chunk to write, one thread per stream for the
 * identifier and the length.
 * Reader: one thread per stream walks its headers into its own table region; scans of the per-stream counts and a
 * compaction make the tables contiguous; the host reads the two totals back (the one synchronisation); then one decode
 * launch, one warp per data chunk to verify and one thread per stream for the result.                               */
#define FRAMED_BATCH_NONE (~(uint64_t)0)

/* writer workspace after the fragment slots: device-written tables, then the host-built ones (one upload) */
enum { WB_FLEN, WB_CRC, WB_REC, WB_OFF, WB_CTR, WB_FIN, WB_FOFF, WB_CIN, WB_CLEN, WB_CSTREAM, WB_CFRAG, WB_SOUT, WB_SFIRST, WB_END };

static uint64_t framed_batch_compress_layout(uint64_t F, uint64_t K, uint64_t n, uint64_t o[WB_END + 1])
{
	const uint64_t per[WB_END] = {F * 4, K * 4, K * 4, (K + 1) * 8, 256, F * 4, F * 8, K * 8, K * 4, K * 4, K * 4, n * 8, (n + 1) * 4};
	uint64_t p = al256(F * SLOT_STRIDE_32K);
	int i;
	for (i = 0; i < WB_END; i++) {
		o[i] = p;
		p = al256(p + per[i]);
	}
	o[WB_END] = p;
	return p;
}

/* fragments and chunks of a batch; 0 when a stream is too long or the fragments leave uint32 (chunks <= fragments) */
static int framed_batch_counts(const uint64_t *h_len, uint32_t n, uint64_t *F, uint64_t *K)
{
	uint32_t i;
	*F = *K = 0;
	for (i = 0; i < n; i++) {
		if (h_len[i] > FRAMED_MAX_INPUT)
			return 0;
		*F += (h_len[i] + CSB_FRAGMENT_MAX - 1) / CSB_FRAGMENT_MAX;
		*K += chunks_of(h_len[i]);
		if (*F > 0xffffffffull)
			return 0;
	}
	return 1;
}

uint64_t csnappy_framed_batch_compress_workspace(const uint64_t *h_in_len, uint32_t n_streams)
{
	uint64_t F, K, o[WB_END + 1];
	if ((n_streams && !h_in_len) || !framed_batch_counts(h_in_len, n_streams, &F, &K))
		return FRAMED_BATCH_NONE;
	return framed_batch_compress_layout(F, K, n_streams, o);
}

int csnappy_framed_batch_compress(const void *d_in, const uint64_t *h_in_off, const uint64_t *h_in_len, uint32_t n_streams,
				  void *d_out, const uint64_t *h_out_off, uint64_t out_capacity, uint64_t *d_out_len,
				  int workmem_bytes_power_of_two, void *d_workspace, uint64_t workspace_bytes, void *stream)
{
	uint64_t F, K, o[WB_END + 1], at = 0, f = 0, k = 0, total_in = 0;
	uint8_t *ws = (uint8_t *)d_workspace, *tab;
	csb_stream_t s = (csb_stream_t)stream;
	struct csb_framed_batch_wtable t;
	struct csb_compress_args a;
	uint32_t i;
	int e;
	if (workmem_bytes_power_of_two < 9 || workmem_bytes_power_of_two > 16)
		return set_err("workmem_bytes_power_of_two outside 9..16", 0);
	if (n_streams == 0)
		return 0;
	if (!h_in_off || !h_in_len || !d_out || !d_out_len || !d_workspace)
		return set_err("null buffer", 0);
	if (!framed_batch_counts(h_in_len, n_streams, &F, &K))
		return set_err("a stream longer than (2^32 - 2) * 32768 bytes, or more than 2^32 - 1 fragments", 0);
	for (i = 0; i < n_streams; i++) {
		const uint64_t base = h_out_off ? h_out_off[i] : at, m = csnappy_framed_max_length(h_in_len[i]);
		if (base > out_capacity || m > out_capacity - base)
			return set_err("output slot ending past out_capacity", 0);
		at = base + m;
		total_in += h_in_len[i];
	}
	if (total_in && !d_in)
		return set_err("null buffer", 0);
	if (workspace_bytes < framed_batch_compress_layout(F, K, n_streams, o))
		return set_err("workspace smaller than csnappy_framed_batch_compress_workspace()", 0);
	/* host image of the tables [o[WB_FIN], o[WB_END]) */
	tab = (uint8_t *)malloc((size_t)(o[WB_END] - o[WB_FIN]));
	if (!tab)
		return set_err("host table", (int)cudaErrorMemoryAllocation);
	{
#define HT(idx, type) ((type *)(tab + (o[idx] - o[WB_FIN])))
		uint32_t *fin = HT(WB_FIN, uint32_t), *c_len = HT(WB_CLEN, uint32_t), *c_stream = HT(WB_CSTREAM, uint32_t);
		uint32_t *c_frag = HT(WB_CFRAG, uint32_t), *s_first = HT(WB_SFIRST, uint32_t);
		uint64_t *foff = HT(WB_FOFF, uint64_t), *c_in = HT(WB_CIN, uint64_t), *s_out = HT(WB_SOUT, uint64_t);
#undef HT
		at = 0;
		for (i = 0; i < n_streams; i++) {
			const uint64_t base = h_in_off[i], n = h_in_len[i];
			uint64_t c;
			s_out[i] = h_out_off ? h_out_off[i] : at;
			s_first[i] = (uint32_t)k;
			at += csnappy_framed_max_length(n);
			for (c = 0; c < n; c += FRAMED_CHUNK) {
				const uint32_t m = n - c < FRAMED_CHUNK ? (uint32_t)(n - c) : (uint32_t)FRAMED_CHUNK;
				uint32_t q;
				c_in[k] = base + c;
				c_len[k] = m;
				c_stream[k] = i;
				c_frag[k] = (uint32_t)f;
				for (q = 0; q < m; q += CSB_FRAGMENT_MAX) {
					foff[f] = base + c + q;
					fin[f] = m - q < CSB_FRAGMENT_MAX ? m - q : CSB_FRAGMENT_MAX;
					f++;
				}
				k++;
			}
		}
		s_first[n_streams] = (uint32_t)k;
	}
	/* pageable source: the copy is staged before the call returns, the table can be freed right after */
	e = (int)cudaMemcpyAsync(ws + o[WB_FIN], tab, (size_t)(o[WB_END] - o[WB_FIN]), cudaMemcpyHostToDevice, (cudaStream_t)s);
	free(tab);
	if (e)
		return set_err("H2D chunk tables", e);
	t.flen = (const uint32_t *)(ws + o[WB_FLEN]);
	t.c_in = (const uint64_t *)(ws + o[WB_CIN]);
	t.c_len = (const uint32_t *)(ws + o[WB_CLEN]);
	t.c_stream = (const uint32_t *)(ws + o[WB_CSTREAM]);
	t.c_frag = (const uint32_t *)(ws + o[WB_CFRAG]);
	t.crc = (uint32_t *)(ws + o[WB_CRC]);
	t.rec = (uint32_t *)(ws + o[WB_REC]);
	t.off = (const uint64_t *)(ws + o[WB_OFF]);
	t.s_out = (const uint64_t *)(ws + o[WB_SOUT]);
	t.s_first = (const uint32_t *)(ws + o[WB_SFIRST]);
	if (F) {
		fill_compress_args(&a);
		a.in = (const uint8_t *)d_in;
		a.in_off = (const uint64_t *)(ws + o[WB_FOFF]);
		a.in_len = (const uint32_t *)(ws + o[WB_FIN]);
		a.n_blocks = (uint32_t)F;
		a.out = ws;
		a.out_stride = SLOT_STRIDE_32K;
		a.out_len = (uint32_t *)(ws + o[WB_FLEN]);
		a.wm = workmem_bytes_power_of_two;
		a.flags = CSNAPPY_BATCH_SHRINK_TABLE; /* applies to fragments below 32768 bytes: a chunk's short last one */
		a.counter = (uint32_t *)(ws + o[WB_CTR]);
		if ((e = csb_launch_compress(&a, s)))
			return set_err("compress launch", e);
		if ((e = csb_launch_framed_batch_crc((const uint8_t *)d_in, (uint32_t)K, &t, s)))
			return set_err("crc launch", e);
	}
	if ((e = csb_launch_scan(t.rec, (uint32_t)K, (uint64_t *)(ws + o[WB_OFF]), s)))
		return set_err("scan launch", e);
	e = csb_launch_framed_batch_write((const uint8_t *)d_in, (uint32_t)K, n_streams, ws, SLOT_STRIDE_32K, &t,
					  (uint8_t *)d_out, d_out_len, s);
	return e ? set_err("framed write launch", e) : 0;
}

/* reader workspace: per-stream table (uploaded) and results, the two scans and the totals, then the region tables and
 * the compacted tables for D = sum(src_len / 8 + 1) data chunks (a data chunk takes at least 8 bytes of its stream),
 * then the decoder's block counter */
enum { RB_SSRC, RB_SLEN, RB_SDST, RB_SCAP, RB_SREG, RB_ND, RB_NC, RB_WKEY, RB_WOUT, RB_VKEY, RB_DBASE, RB_CBASE, RB_TOT,
       RB_RPOS, RB_ROUT, RB_RLEN, RB_RCRC, RB_RCIDX, RB_RPLEN, RB_POS, RB_OUTOFF, RB_OUTLEN, RB_CRC, RB_CIDX, RB_STREAM,
       RB_CPOS, RB_COUTOFF, RB_CLEN, RB_CPROD, RB_CSTATUS, RB_CTR, RB_END };

static uint64_t framed_batch_decompress_layout(uint64_t D, uint64_t n, uint8_t *ws, uint64_t o[RB_END + 1],
					       struct csb_framed_batch_rtable *t)
{
	const uint64_t per[RB_END] = {n * 8, n * 8, n * 8, n * 8, n * 8, n * 4, n * 4, n * 8, n * 8, n * 8, (n + 1) * 8,
				      (n + 1) * 8, 16, D * 8, D * 8, D * 4, D * 4, D * 4, D * 4, D * 8, D * 8, D * 4,
				      D * 4, D * 4, D * 4, D * 8, D * 8, D * 4, D * 4, D * 4, 256};
	uint64_t p = 0;
	int i;
	for (i = 0; i < RB_END; i++) {
		o[i] = p;
		p = al256(p + per[i]);
	}
	o[RB_END] = p;
	if (t) {
#define RT(idx, type) ((type *)(ws + o[idx]))
		t->s_src = RT(RB_SSRC, const uint64_t);
		t->s_len = RT(RB_SLEN, const uint64_t);
		t->s_dst = RT(RB_SDST, const uint64_t);
		t->s_cap = RT(RB_SCAP, const uint64_t);
		t->s_reg = RT(RB_SREG, const uint64_t);
		t->nd = RT(RB_ND, uint32_t);
		t->nc = RT(RB_NC, uint32_t);
		t->walk_key = RT(RB_WKEY, uint64_t);
		t->walk_out = RT(RB_WOUT, uint64_t);
		t->verify_key = RT(RB_VKEY, uint64_t);
		t->d_base = RT(RB_DBASE, uint64_t);
		t->c_base = RT(RB_CBASE, uint64_t);
		t->totals = RT(RB_TOT, uint64_t);
		t->r_pos = RT(RB_RPOS, uint64_t);
		t->r_out = RT(RB_ROUT, uint64_t);
		t->r_len = RT(RB_RLEN, uint32_t);
		t->r_crc = RT(RB_RCRC, uint32_t);
		t->r_cidx = RT(RB_RCIDX, uint32_t);
		t->r_plen = RT(RB_RPLEN, uint32_t);
		t->pos = RT(RB_POS, uint64_t);
		t->out_off = RT(RB_OUTOFF, uint64_t);
		t->out_len = RT(RB_OUTLEN, uint32_t);
		t->crc = RT(RB_CRC, uint32_t);
		t->cidx = RT(RB_CIDX, uint32_t);
		t->stream = RT(RB_STREAM, uint32_t);
		t->c_pos = RT(RB_CPOS, uint64_t);
		t->c_out_off = RT(RB_COUTOFF, uint64_t);
		t->c_len = RT(RB_CLEN, uint32_t);
		t->c_produced = RT(RB_CPROD, uint32_t);
		t->c_status = RT(RB_CSTATUS, int32_t);
#undef RT
	}
	return p;
}

/* table entries of a batch (sum of src_len / 8 + 1); 0 when a stream is longer than 2^35 bytes or D leaves uint32 */
static int framed_batch_entries(const uint64_t *h_len, uint32_t n, uint64_t *D)
{
	uint32_t i;
	*D = 0;
	for (i = 0; i < n; i++) {
		if (h_len[i] > FRAMED_MAX_SRC)
			return 0;
		*D += h_len[i] / 8 + 1;
		if (*D > 0xffffffffull)
			return 0;
	}
	return 1;
}

uint64_t csnappy_framed_batch_decompress_workspace(const uint64_t *h_src_len, uint32_t n_streams)
{
	uint64_t D, o[RB_END + 1];
	if ((n_streams && !h_src_len) || !framed_batch_entries(h_src_len, n_streams, &D))
		return FRAMED_BATCH_NONE;
	return framed_batch_decompress_layout(D, n_streams, NULL, o, NULL);
}

int csnappy_framed_batch_decompress(const void *d_src, const uint64_t *h_src_off, const uint64_t *h_src_len,
				    uint32_t n_streams, void *d_dst, const uint64_t *h_dst_off, const uint64_t *h_dst_cap,
				    uint64_t *d_out_len, int32_t *d_status, uint64_t *d_failed_offset, void *d_workspace,
				    uint64_t workspace_bytes, void *stream)
{
	struct csb_framed_batch_rtable t;
	struct csb_decompress_args a;
	uint64_t D, o[RB_END + 1], totals[2], reg = 0, total_src = 0, total_cap = 0, *h;
	uint8_t *ws = (uint8_t *)d_workspace;
	cudaStream_t s = (cudaStream_t)stream;
	const uint8_t *src = (const uint8_t *)d_src;
	uint32_t i;
	int e;
	if (n_streams == 0)
		return 0;
	if (!h_src_off || !h_src_len || !h_dst_off || !h_dst_cap || !d_out_len || !d_status || !d_workspace)
		return set_err("null buffer", 0);
	if (!framed_batch_entries(h_src_len, n_streams, &D))
		return set_err("a stream longer than 2^35 bytes, or more than 2^32 - 1 chunk table entries", 0);
	for (i = 0; i < n_streams; i++) {
		total_src |= h_src_len[i];
		total_cap |= h_dst_cap[i];
	}
	if ((total_src && !d_src) || (total_cap && !d_dst))
		return set_err("null buffer", 0);
	if (workspace_bytes < framed_batch_decompress_layout(D, n_streams, ws, o, &t))
		return set_err("workspace smaller than csnappy_framed_batch_decompress_workspace()", 0);
	/* the per-stream table [o[RB_SSRC], o[RB_ND]): source offset, length, output offset, capacity, table region */
	h = (uint64_t *)malloc((size_t)(o[RB_ND] - o[RB_SSRC]));
	if (!h)
		return set_err("host table", (int)cudaErrorMemoryAllocation);
	for (i = 0; i < n_streams; i++) {
		h[(o[RB_SSRC] / 8) + i] = h_src_off[i];
		h[(o[RB_SLEN] / 8) + i] = h_src_len[i];
		h[(o[RB_SDST] / 8) + i] = h_dst_off[i];
		h[(o[RB_SCAP] / 8) + i] = h_dst_cap[i];
		h[(o[RB_SREG] / 8) + i] = reg;
		reg += h_src_len[i] / 8 + 1;
	}
	e = (int)cudaMemcpyAsync(ws + o[RB_SSRC], h, (size_t)(o[RB_ND] - o[RB_SSRC]), cudaMemcpyHostToDevice, s);
	free(h);
	if (e)
		return set_err("H2D stream table", e);
	if ((e = csb_launch_framed_batch_walk(src, n_streams, &t, NULL, NULL, (csb_stream_t)s)))
		return set_err("framed walk launch", e);
	if ((e = csb_launch_scan(t.nd, n_streams, t.d_base, (csb_stream_t)s)) ||
	    (e = csb_launch_scan(t.nc, n_streams, t.c_base, (csb_stream_t)s)))
		return set_err("scan launch", e);
	if ((e = csb_launch_framed_batch_compact(n_streams, &t, (csb_stream_t)s)))
		return set_err("compact launch", e);
	/* the only synchronisation: the batch totals size the launches below */
	if ((e = (int)cudaMemcpyAsync(totals, t.totals, sizeof(totals), cudaMemcpyDeviceToHost, s)) ||
	    (e = (int)cudaStreamSynchronize(s)))
		return set_err("D2H chunk totals", e);
	if (totals[1]) {
		fill_decompress_args(&a);
		a.in = src + 8; /* block j = the body behind chunk j's header and CRC */
		a.in_off = t.c_pos;
		a.in_len = t.c_len;
		a.n_blocks = (uint32_t)totals[1];
		a.out = (uint8_t *)d_dst;
		a.out_off = t.c_out_off;
		a.uniform_cap = CSB_FRAMED_CHUNK; /* WITH_HEADER: the capacity becomes the varint's value, <= 65536 */
		a.out_len = t.c_produced;
		a.status = t.c_status;
		a.flags = CSNAPPY_BATCH_WITH_HEADER;
		a.counter = (uint32_t *)(ws + o[RB_CTR]);
		if ((e = csb_launch_decompress(&a, (csb_stream_t)s)))
			return set_err("decompress launch", e);
	}
	e = csb_launch_framed_batch_verify(src, (uint8_t *)d_dst, (uint32_t)totals[0], n_streams, &t, d_out_len, d_status,
					   d_failed_offset, (csb_stream_t)s);
	return e ? set_err("framed verify launch", e) : 0;
}

int csnappy_framed_batch_decompressed_length(const void *d_src, const uint64_t *h_src_off, const uint64_t *h_src_len,
					     uint32_t n_streams, uint64_t *d_length, int32_t *d_status, void *stream)
{
	struct csb_framed_batch_rtable t;
	cudaStream_t s = (cudaStream_t)stream;
	uint64_t *h, total_src = 0;
	void *d_tab = NULL;
	uint32_t i;
	int e;
	if (n_streams == 0)
		return 0;
	if (!h_src_off || !h_src_len || !d_length || !d_status)
		return set_err("null buffer", 0);
	for (i = 0; i < n_streams; i++) {
		if (h_src_len[i] > FRAMED_MAX_SRC)
			return set_err("a stream longer than 2^35 bytes", 0);
		total_src |= h_src_len[i];
	}
	if (total_src && !d_src)
		return set_err("null buffer", 0);
	/* the offsets and lengths go to a stream-ordered allocation, freed behind the walk */
	h = (uint64_t *)malloc((size_t)n_streams * 16);
	if (!h)
		return set_err("host table", (int)cudaErrorMemoryAllocation);
	memcpy(h, h_src_off, (size_t)n_streams * 8);
	memcpy(h + n_streams, h_src_len, (size_t)n_streams * 8);
	e = (int)cudaMallocAsync(&d_tab, (size_t)n_streams * 16, s);
	if (!e)
		e = (int)cudaMemcpyAsync(d_tab, h, (size_t)n_streams * 16, cudaMemcpyHostToDevice, s);
	free(h);
	if (e) {
		if (d_tab)
			cudaFreeAsync(d_tab, s);
		return set_err("H2D stream table", e);
	}
	memset(&t, 0, sizeof(t));
	t.s_src = (const uint64_t *)d_tab;
	t.s_len = (const uint64_t *)d_tab + n_streams;
	e = csb_launch_framed_batch_walk((const uint8_t *)d_src, n_streams, &t, d_length, d_status, (csb_stream_t)s);
	if (e) {
		cudaFreeAsync(d_tab, s);
		return set_err("framed length walk launch", e);
	}
	e = (int)cudaFreeAsync(d_tab, s);
	return e ? set_err("cudaFreeAsync(stream table)", e) : 0;
}
