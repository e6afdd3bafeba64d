/* agrep_b200/csrc/aux.cu -- the small kernels around the stages: bitmap density sample, bitmap -> candidate list,
 * exclusive scans, ordinals (delimiter counts), the synthetic corpus generator */
#include "automaton.cuh"
#include "corpus.h"

/* how often does each candidate gram of the pattern start in a chunk?  One thread per 16-byte chunk of a sample of
 * the text (nblk stretches of blk_chunks chunks, evenly spread); the anchor planner (scan.cu) picks the k+1 disjoint
 * grams with the fewest hits: stage 1.5's work is proportional to the chunks stage 1 flags */
__global__ void __launch_bounds__(256) k_gram_sample(const uint8_t *text, uint64_t n_chunks, uint32_t nblk, uint32_t blk_chunks,
                                                    int ngram, const uint32_t *gram, const uint32_t *gmask, uint32_t fold, unsigned int *counts)
{
	__shared__ unsigned int s_cnt[128];
	if (threadIdx.x < 128) s_cnt[threadIdx.x] = 0;
	__syncthreads();
	const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const uint64_t b = t / blk_chunks, i = t % blk_chunks;
	if (b < nblk) {
		const uint64_t chunk = (n_chunks / nblk) * b + i;
		if (chunk + 2 < n_chunks) {
			const uint4 v = __ldg(reinterpret_cast<const uint4 *>(text) + chunk);
			const uint32_t x4 = __ldg(reinterpret_cast<const uint32_t *>(text) + (chunk + 1) * 4);
			const uint32_t x[5] = { v.x | fold, v.y | fold, v.z | fold, v.w | fold, x4 | fold };
			uint32_t wv[16];
#pragma unroll
			for (int w = 0; w < 4; w++) {
				wv[4 * w] = x[w]; wv[4 * w + 1] = __funnelshift_r(x[w], x[w + 1], 8);
				wv[4 * w + 2] = __funnelshift_r(x[w], x[w + 1], 16); wv[4 * w + 3] = __funnelshift_r(x[w], x[w + 1], 24);
			}
			for (int g = 0; g < ngram; g++) {
				const uint32_t G = gram[g], M = gmask[g];
				bool hit = false;
#pragma unroll
				for (int s = 0; s < 16; s++) hit = hit || ((wv[s] & M) == G);
				if (hit) atomicAdd(&s_cnt[g], 1u);
			}
		}
	}
	__syncthreads();
	if (threadIdx.x < ngram && s_cnt[threadIdx.x]) atomicAdd(&counts[threadIdx.x], s_cnt[threadIdx.x]);
}

/* how dense are the flags?  popcount of every `stride`-th bitmap word (an estimate is all the host needs to pick the
 * record stage's form before it spends time on stage 1.5) */
__global__ void __launch_bounds__(256) k_bitmap_sample(const uint32_t *bitmap, uint64_t n_words, uint32_t stride, unsigned long long *out)
{
	unsigned long long c = 0;
	for (uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * stride; i < n_words; i += (uint64_t)gridDim.x * blockDim.x * stride)
		c += __popc(bitmap[i]);
	c = __reduce_add_sync(0xffffffffu, (uint32_t)c);
	if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

/* bitmap -> ordered list of flagged chunk numbers: per-block popcounts, scan (k_scan_tiles), scatter */
__global__ void __launch_bounds__(COMPACT_THREADS) k_compact_count(const uint32_t *bitmap, uint64_t n_words, uint32_t *block_counts, unsigned long long *totals)
{
	const uint64_t w0 = ((uint64_t)blockIdx.x * COMPACT_THREADS + threadIdx.x) * COMPACT_WPT;
	uint32_t c = 0;
#pragma unroll
	for (int j = 0; j < COMPACT_WPT; j++) if (w0 + j < n_words) c += __popc(bitmap[w0 + j]);
	__shared__ uint32_t s_part[COMPACT_THREADS / 32];
	uint32_t sum = __reduce_add_sync(0xffffffffu, c);
	if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = sum;
	__syncthreads();
	if (threadIdx.x == 0) {
		uint32_t t = 0;
		for (int j = 0; j < COMPACT_THREADS / 32; j++) t += s_part[j];
		block_counts[blockIdx.x] = t;
		if (t) atomicAdd(&totals[1], (unsigned long long)t);
	}
}

__global__ void __launch_bounds__(COMPACT_THREADS) k_compact_write(const uint32_t *bitmap, uint64_t n_words, const uint64_t *block_offsets,
                                                                   uint64_t *list, uint64_t cap)
{
	const uint64_t w0 = ((uint64_t)blockIdx.x * COMPACT_THREADS + threadIdx.x) * COMPACT_WPT;
	uint32_t wd[COMPACT_WPT], c = 0;
#pragma unroll
	for (int j = 0; j < COMPACT_WPT; j++) { wd[j] = (w0 + j < n_words) ? bitmap[w0 + j] : 0u; c += __popc(wd[j]); }
	__shared__ uint32_t s_scan[COMPACT_THREADS];
	s_scan[threadIdx.x] = c;
	__syncthreads();
	for (int off = 1; off < COMPACT_THREADS; off <<= 1) {
		uint32_t v = (threadIdx.x >= (unsigned)off) ? s_scan[threadIdx.x - off] : 0;
		__syncthreads();
		s_scan[threadIdx.x] += v;
		__syncthreads();
	}
	uint64_t at = block_offsets[blockIdx.x] + (s_scan[threadIdx.x] - c);
#pragma unroll
	for (int j = 0; j < COMPACT_WPT; j++)
		for (uint32_t b = wd[j]; b; b &= b - 1) { if (at < cap) list[at] = (w0 + j) * 32 + (uint64_t)(__ffs(b) - 1); at++; }
}

/* exclusive scan of 32-bit counts into 64-bit offsets (one block, coalesced tiles of 4096 with a running carry);
 * the grand total goes to *total when given */
__global__ void __launch_bounds__(1024) k_scan_tiles(const uint32_t *counts, uint64_t *offsets, uint64_t n_tiles, unsigned long long *total)
{
	__shared__ unsigned long long s_warp[32];
	__shared__ unsigned long long s_carry;
	const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
	if (tid == 0) s_carry = 0;
	__syncthreads();
	for (uint64_t base = 0; base < n_tiles; base += 4096) {
		uint32_t v[4]; unsigned long long sum = 0;
#pragma unroll
		for (int j = 0; j < 4; j++) { const uint64_t i = base + (uint64_t)tid * 4 + j; v[j] = i < n_tiles ? counts[i] : 0u; sum += v[j]; }
		unsigned long long inc = sum;
#pragma unroll
		for (int o = 1; o < 32; o <<= 1) { unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= (uint32_t)o) inc += t; }
		if (lane == 31) s_warp[wid] = inc;
		__syncthreads();
		if (wid == 0) {
			unsigned long long w = s_warp[lane], winc = w;
#pragma unroll
			for (int o = 1; o < 32; o <<= 1) { unsigned long long t = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= (uint32_t)o) winc += t; }
			s_warp[lane] = winc - w;                 /* exclusive prefix of the warp sums */
		}
		__syncthreads();
		unsigned long long run = s_carry + s_warp[wid] + (inc - sum);
#pragma unroll
		for (int j = 0; j < 4; j++) { const uint64_t i = base + (uint64_t)tid * 4 + j; if (i < n_tiles) offsets[i] = run; run += v[j]; }
		__syncthreads();
		if (tid == 1023) s_carry = run;
		__syncthreads();
	}
	if (total && tid == 0) *total = s_carry;
}

/* two-level exclusive scan for long count arrays (the per-candidate counts of the list form):
 * k_scan_partial sums blocks of 16384 counts, k_scan_tiles scans those sums, k_scan_apply finishes each block */
__global__ void __launch_bounds__(1024) k_scan_partial(const uint32_t *counts, uint64_t n, uint32_t *block_sums, const unsigned long long *n_dev)
{
	if (n_dev && *n_dev < n) n = *n_dev;                    /* the length lives on the device; the grid covers the capacity */
	__shared__ uint32_t s_w[32];
	const uint64_t base = (uint64_t)blockIdx.x * SCAN_BLOCK;
	uint32_t sum = 0;
#pragma unroll
	for (int j = 0; j < SCAN_BLOCK / 1024; j++) { const uint64_t i = base + (uint64_t)j * 1024 + threadIdx.x; if (i < n) sum += counts[i]; }
	sum = __reduce_add_sync(0xffffffffu, sum);
	if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = sum;
	__syncthreads();
	if (threadIdx.x < 32) { uint32_t v = __reduce_add_sync(0xffffffffu, s_w[threadIdx.x]); if (threadIdx.x == 0) block_sums[blockIdx.x] = v; }
}

__global__ void __launch_bounds__(1024) k_scan_apply(const uint32_t *counts, uint64_t n, const uint64_t *block_offsets, uint64_t *offsets, const unsigned long long *n_dev)
{
	if (n_dev && *n_dev < n) n = *n_dev;
	__shared__ unsigned long long s_warp[32];
	__shared__ unsigned long long s_carry;
	const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
	const uint64_t base0 = (uint64_t)blockIdx.x * SCAN_BLOCK;
	if (tid == 0) s_carry = block_offsets[blockIdx.x];
	__syncthreads();
	for (uint64_t base = base0; base < base0 + SCAN_BLOCK && base < n; base += 4096) {
		uint32_t v[4]; unsigned long long sum = 0;
#pragma unroll
		for (int j = 0; j < 4; j++) { const uint64_t i = base + (uint64_t)tid * 4 + j; v[j] = i < n ? counts[i] : 0u; sum += v[j]; }
		unsigned long long inc = sum;
#pragma unroll
		for (int o = 1; o < 32; o <<= 1) { unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= (uint32_t)o) inc += t; }
		if (lane == 31) s_warp[wid] = inc;
		__syncthreads();
		if (wid == 0) {
			unsigned long long w = s_warp[lane], winc = w;
#pragma unroll
			for (int o = 1; o < 32; o <<= 1) { unsigned long long t = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= (uint32_t)o) winc += t; }
			s_warp[lane] = winc - w;
		}
		__syncthreads();
		unsigned long long run = s_carry + s_warp[wid] + (inc - sum);
#pragma unroll
		for (int j = 0; j < 4; j++) { const uint64_t i = base + (uint64_t)tid * 4 + j; if (i < n) offsets[i] = run; run += v[j]; }
		__syncthreads();
		if (tid == 1023) s_carry = run;
		__syncthreads();
	}
}

/* ================================================================================================
 * synthetic corpus
 * ============================================================================================== */
__constant__ char     c_vocab[sizeof(AGB_VOCAB_STR)];
__constant__ uint16_t c_woff[257];
static const char h_vocab[] = AGB_VOCAB_STR;

struct CorpusParams { agb_corpus_spec s; int needle_len; };

#define CORPUS_THREADS 32
#define CORPUS_STRIDE  (AGB_PAGE + 4)     /* +1 word: the 32 generator threads hit different banks */
__global__ void __launch_bounds__(CORPUS_THREADS) k_corpus(uint8_t *out, uint64_t n_pages, const CorpusParams P)
{
	/* one thread generates one 4 KiB page (the generator is inherently sequential) into shared memory,
	 * then the warp writes the 32 pages out with coalesced 128-byte stores */
	extern __shared__ __align__(16) uint8_t s_pages[];
	const uint64_t pg0 = (uint64_t)blockIdx.x * CORPUS_THREADS, pg = pg0 + threadIdx.x;
	if (pg < n_pages)
		agb_corpus_page(s_pages + threadIdx.x * CORPUS_STRIDE, P.s.seed, P.s.first_page + pg, c_vocab, c_woff,
		                P.s.paragraphs, P.s.needle_every, P.s.needle, P.needle_len, P.s.needle_maxedits);
	__syncwarp();
	for (int q = 0; q < CORPUS_THREADS && pg0 + q < n_pages; q++) {
		const uint32_t *src = reinterpret_cast<const uint32_t *>(s_pages + q * CORPUS_STRIDE);
		uint32_t *dst = reinterpret_cast<uint32_t *>(out + (pg0 + q) * AGB_PAGE);
		for (int j = threadIdx.x; j < AGB_PAGE / 4; j += CORPUS_THREADS) dst[j] = src[j];
	}
}

static int corpus_check(const agb_corpus_spec *s, uint16_t *woff)
{
	if (!s || (s->n_bytes % AGB_PAGE) != 0) { snprintf(g_err, sizeof g_err, "corpus size must be a multiple of %d", AGB_PAGE); return AGB_ERR_ARG; }
	if (agb_vocab_offsets(h_vocab, woff) != 256) { snprintf(g_err, sizeof g_err, "vocabulary must hold 256 words"); return AGB_ERR_ARG; }
	return AGB_OK;
}

extern "C" int agb_corpus_fill_device(const agb_corpus_spec *s, void *d_text, void *stream)
{
	uint16_t woff[257]; int rc = corpus_check(s, woff); if (rc) return rc;
	cudaStream_t st = (cudaStream_t)stream;
	CUDA_TRY(cudaMemcpyToSymbolAsync(c_vocab, h_vocab, sizeof h_vocab, 0, cudaMemcpyHostToDevice, st));
	CUDA_TRY(cudaMemcpyToSymbolAsync(c_woff, woff, sizeof woff, 0, cudaMemcpyHostToDevice, st));
	CorpusParams P; P.s = *s; P.s.needle[63] = 0; P.needle_len = (int)strlen(P.s.needle);
	uint64_t n_pages = s->n_bytes / AGB_PAGE;
	if (n_pages) {
		const int smem = CORPUS_THREADS * CORPUS_STRIDE;
		CUDA_TRY(cudaFuncSetAttribute(k_corpus, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
		k_corpus<<<(unsigned)((n_pages + CORPUS_THREADS - 1) / CORPUS_THREADS), CORPUS_THREADS, smem, st>>>((uint8_t *)d_text, n_pages, P);
		g_launches++;
		CUDA_TRY(cudaGetLastError());
	}
	return AGB_OK;
}

extern "C" int agb_corpus_fill_host(const agb_corpus_spec *s, void *h_text)
{
	uint16_t woff[257]; int rc = corpus_check(s, woff); if (rc) return rc;
	agb_corpus_spec t = *s; t.needle[63] = 0;
	int nl = (int)strlen(t.needle);
	for (uint64_t pg = 0; pg < s->n_bytes / AGB_PAGE; pg++)
		agb_corpus_page((uint8_t *)h_text + pg * AGB_PAGE, t.seed, t.first_page + pg, h_vocab, woff,
		                t.paragraphs, t.needle_every, t.needle, nl, t.needle_maxedits);
	return AGB_OK;
}

/* ================================================================================================
 * ordinals: j of the reference's loops (bitap.c:178, asearch.c:120), what -n prints minus one.
 *
 * j is incremented at every record close, the virtual '\n' included, so the ordinal of a record is the number of
 * delimiter ends at or before the delimiter that closes it -- a property of the text alone.  k_delim_count counts
 * the delimiter ends of every 512-byte block (16-bit) and every 32 KiB tile (one more HBM-bound pass, only when
 * ordinals are asked for); the tile counts are scanned; k_ordinals gives every record tile prefix + the blocks
 * of its tile before its own + the delimiter ends of its own block up to its close.  Same delimiter rule as
 * delim_ends_at() / agb_fill_ordinals(): every occurrence of a border-free delimiter, greedy pairing from the
 * start of the run for c^L ("$$"), the virtual '\n' and the delimiter appended at EOF included.
 * ============================================================================================== */

/* delimiter ends in [from, to) (file offsets; to <= n + L), sequentially; run: the length of the run of delim[0]
 * that ends at from - 1 (kind 1) */
__device__ __forceinline__ uint32_t ord_count_seq(Reader &R, const OrdParams &P, int64_t from, int64_t to)
{
	uint32_t cnt = 0;
	if (P.L == 1) { for (int64_t q = from; q < to; q++) cnt += (R.get(q) | P.dfold[0]) == P.delim[0]; return cnt; }
	if (P.kind == 0) {
		for (int64_t q = from; q < to; q++) {
			bool m = true;
			for (int u = 0; u < P.L && m; u++) m = (R.get(q - u) | P.dfold[P.L - 1 - u]) == P.delim[P.L - 1 - u];
			cnt += m ? 1u : 0u;
		}
		return cnt;
	}
	if (P.kind == 2) {
		/* the occurrence taken last before `from` that can still shadow one ending at or after it, then greedily on */
		int64_t last = -(1ll << 60);
		for (int64_t e = from - 1; e > from - P.L; e--) if (delim_ends_at(R, e, P.delim, P.dfold, P.L, 2)) { last = e; break; }
		for (int64_t q = from; q < to; q++) if (q - P.L + 1 > last && delim_occurs(R, q, P.delim, P.dfold, P.L)) { cnt++; last = q; }
		return cnt;
	}
	const int c = P.delim[0], f = P.dfold[0];
	int64_t run = 0;
	for (int64_t q = from - 1; q >= -1 && (R.get(q) | f) == c; q--) run++;       /* (-1 is the virtual '\n') */
	for (int64_t q = from; q < to; q++) {
		run = (R.get(q) | f) == c ? run + 1 : 0;
		cnt += (run > 0 && run % P.L == 0) ? 1u : 0u;
	}
	return cnt;
}

__global__ void __launch_bounds__(ORD_THREADS) k_delim_count(const OrdParams P)
{
	__shared__ uint32_t s_warp[ORD_THREADS / 32];
	const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
	const int64_t n = (int64_t)P.n, limit = n + P.L, tile0 = (int64_t)blockIdx.x * ORD_TILE;
	uint32_t cnt = 0;                                           /* this thread's share of the tile */
	if (P.L == 1 && tile0 + ORD_TILE <= n) {
		/* a warp takes a 512-byte block per iteration, 16 bytes per lane (coalesced): exact per-byte equality by
		 * SWAR (0x80 where the byte equals the delimiter), one warp reduction per block */
		const uint32_t d4 = P.delim[0] * 0x01010101u, f4 = P.dfold[0] * 0x01010101u;
#pragma unroll
		for (int it = 0; it < ORD_TILE / ORD_BLOCK / (ORD_THREADS / 32); it++) {
			const uint32_t blk = wid * (ORD_TILE / ORD_BLOCK / (ORD_THREADS / 32)) + it;
			const uint4 x = __ldg(reinterpret_cast<const uint4 *>(P.text + tile0 + (int64_t)blk * ORD_BLOCK) + lane);
			const uint32_t xs[4] = { x.x, x.y, x.z, x.w };
			uint32_t c = 0;
#pragma unroll
			for (int w = 0; w < 4; w++) {
				const uint32_t t = (xs[w] | f4) ^ d4;
				c += __popc(~(((t & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | t | 0x7F7F7F7Fu));
			}
			const uint32_t b = __reduce_add_sync(0xffffffffu, c);
			if (lane == 0) P.blocks[(uint64_t)blockIdx.x * (ORD_TILE / ORD_BLOCK) + blk] = (uint16_t)b;
			cnt += c;
		}
	} else {
		/* other delimiters and the last tile: every thread walks its 128 bytes; 4 threads = one block */
		const int64_t s0 = tile0 + (int64_t)tid * ORD_PER, s1 = s0 + ORD_PER < limit ? s0 + ORD_PER : limit;
		if (s0 < limit) {
			Reader R; R.init(P.text, P.n, P.delim, P.L);
			cnt = ord_count_seq(R, P, s0, s1);
		}
		uint32_t b = cnt;
		b += __shfl_xor_sync(0xffffffffu, b, 1); b += __shfl_xor_sync(0xffffffffu, b, 2);
		if ((tid & 3) == 0) P.blocks[(uint64_t)blockIdx.x * (ORD_TILE / ORD_BLOCK) + (tid >> 2)] = (uint16_t)b;
	}
	const uint32_t w = __reduce_add_sync(0xffffffffu, cnt);
	if (lane == 0) s_warp[wid] = w;
	__syncthreads();
	if (tid == 0) { uint32_t t = 0; for (int i = 0; i < ORD_THREADS / 32; i++) t += s_warp[i]; P.tiles[blockIdx.x] = t; }
}

/* the tile counts from block counts that stage 1 already took (front.cu, COUNT): 64 blocks per tile, plus the
 * delimiter appended at EOF, which no block of the text has seen (position n; L = 1 on this path).  That one is added
 * to the tile sum only, never written back to its block: a rerun of the record stage (stages_after_front) runs this
 * kernel again over the same block counts and must count it once.  No reader needs it in the block -- k_ordinals and
 * k_shard_aux sum only the blocks below their own, and the EOF block is the last one that holds text. */
__global__ void __launch_bounds__(256) k_ord_tiles(const OrdParams P, uint64_t n_tiles)
{
	/* a warp per tile: its 64 block counts are 128 consecutive bytes */
	static_assert(ORD_TILE / ORD_BLOCK == 64, "two block counts per lane");
	const uint64_t t = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const uint32_t lane = threadIdx.x & 31;
	if (t >= n_tiles) return;
	const uint64_t b = t * 64 + 2 * lane, eof_blk = P.n / ORD_BLOCK;
	const uint32_t two = *reinterpret_cast<const uint32_t *>(P.blocks + b);
	uint32_t lo = two & 0xFFFFu, hi = two >> 16;
	if (b == eof_blk) lo += 1;
	if (b + 1 == eof_blk) hi += 1;
	const uint32_t sum = __reduce_add_sync(0xffffffffu, lo + hi);
	if (lane == 0) P.tiles[t] = sum;
}

/* delimiter bytes (L = 1) in [from, to), from a multiple of 16: sixteen bytes per load, exact per-byte equality by SWAR;
 * positions from n on are not text -- the delimiter appended at EOF sits at n */
__device__ __forceinline__ uint32_t ord_count_swar(const OrdParams &P, int64_t from, int64_t to)
{
	const int64_t n = (int64_t)P.n, end = to < n ? to : n;
	const uint32_t d4 = P.delim[0] * 0x01010101u, f4 = P.dfold[0] * 0x01010101u;
	uint32_t cnt = (to > n && from <= n) ? 1u : 0u;
	for (int64_t p = from; p < end; p += 16) {
		const uint4 x = __ldg(reinterpret_cast<const uint4 *>(P.text + p));
		const uint32_t xs[4] = { x.x, x.y, x.z, x.w };
		const int64_t left = end - p;                         /* bytes of this group that count */
#pragma unroll
		for (int w = 0; w < 4; w++) {
			const uint32_t t = (xs[w] | f4) ^ d4;
			uint32_t z = ~(((t & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | t | 0x7F7F7F7Fu);
			const int64_t v = left - 4 * w;
			if (v <= 0) z = 0; else if (v < 4) z &= (1u << (8 * (uint32_t)v)) - 1u;
			cnt += __popc(z);
		}
	}
	return cnt;
}

__global__ void __launch_bounds__(256) k_ordinals(const OrdParams P)
{
	unsigned long long nrec = P.totals[0];
	if (nrec > P.capacity) nrec = P.capacity;
	const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= nrec) return;
	const int64_t q = P.records[i].end + P.L - 1;                          /* the last byte of the closing delimiter */
	const uint64_t tile = (uint64_t)q / ORD_TILE, blk = (uint64_t)q / ORD_BLOCK;
	unsigned long long j = P.tile_off[tile];
	for (uint64_t b = tile * (ORD_TILE / ORD_BLOCK); b < blk; b++) j += P.blocks[b];
	if (P.L == 1) j += ord_count_swar(P, (int64_t)(blk * ORD_BLOCK), q + 1);
	else { Reader R; R.init(P.text, P.n, P.delim, P.L); j += ord_count_seq(R, P, (int64_t)(blk * ORD_BLOCK), q + 1); }
	/* the virtual '\n' closes a record of its own when it completes a delimiter: only a 1-byte '\n' can */
	const long long virt = (P.L == 1 && P.delim[0] == '\n') ? 1 : 0;
	P.records[i].ordinal = (long long)j + virt + P.j0;
}

/* after stage 1: is the bitmap so full that thinning it (stage 1.5) and walking a candidate list cannot pay?  Then the
 * record stage walks every byte anyway (slices / dense tile form) and stage 1.5 is skipped.  Estimated from every
 * 61st bitmap word; same 5 % threshold as the list/dense switch in records_launch(). */
int front_is_dense(Workspace &W, uint64_t n, cudaStream_t st, bool *dense)
{
	const uint64_t n_chunks = (n + 15) / 16, n_words = (n_chunks + 31) / 32;
	const uint32_t stride = n_words > (1u << 16) ? 61u : 1u;
	CUDA_TRY(cudaMemsetAsync(W.totals + 14, 0, sizeof(unsigned long long), st));
	const uint64_t samples = (n_words + stride - 1) / stride;
	const unsigned grid = (unsigned)std::min<uint64_t>((samples + 255) / 256, (uint64_t)W.sm_count * 8);
	k_bitmap_sample<<<grid ? grid : 1, 256, 0, st>>>(W.bitmap, n_words, stride, W.totals + 14); g_launches++;
	CUDA_TRY(cudaMemcpyAsync(W.h_totals + 14, W.totals + 14, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
	CUDA_TRY(cudaStreamSynchronize(st));
	*dense = W.h_totals[14] * stride > n_chunks / 20 + 1024;
	return AGB_OK;
}

/* AGB_WANT_ORDINALS: fill agb_record.ordinal of the list just written and leave the number of record closes of the
 * whole text (j after the last record, the basis of the next shard's ordinals) in totals[13].  Runs after the
 * record stage, whose tile scratch it reuses. */
/* the block array of the ordinals pass: (n + L) / 512 entries, zeroed where stage 1 will not write */
int ordinals_reserve(const agb_desc &d, Workspace &W, uint64_t n)
{
	const uint64_t limit = n + (uint64_t)d.L, tiles = (limit + ORD_TILE - 1) / ORD_TILE;
	const size_t nb = (size_t)tiles * (ORD_TILE / ORD_BLOCK);
	if (nb > W.ord_blocks_cap) {
		if (W.ord_blocks) cudaFree(W.ord_blocks);
		W.ord_blocks = nullptr; W.ord_blocks_cap = 0;
		CUDA_TRY(cudaMalloc(&W.ord_blocks, nb * sizeof(uint16_t))); W.ord_blocks_cap = nb;
	}
	return AGB_OK;
}

int ordinals_launch(const agb_desc &d, Workspace &W, const void *d_text, uint64_t n, agb_record *d_records,
                           uint64_t capacity, cudaStream_t st, bool blocks_counted)
{
	uint8_t *h_head = reinterpret_cast<uint8_t *>(W.h_totals + 14);      /* pinned scratch: the first bytes of the text */
	if (n >= (uint64_t)d.L && d.user_delim) {
		CUDA_TRY(cudaMemcpyAsync(h_head, d_text, (size_t)d.L, cudaMemcpyDeviceToHost, st));
		CUDA_TRY(cudaStreamSynchronize(st));
	}
	const uint64_t limit = n + (uint64_t)d.L, tiles = (limit + ORD_TILE - 1) / ORD_TILE;
	if (tiles + 1 > W.tiles) return AGB_ERR_NOMEM;                       /* (ws_prepare sized them for n + one tile) */
	{ int rc0 = ordinals_reserve(d, W, n); if (rc0) return rc0; }
	OrdParams P; memset(&P, 0, sizeof P);
	P.text = (const uint8_t *)d_text; P.n = n; P.blocks = W.ord_blocks; P.tiles = W.tile_counts; P.tile_off = W.tile_offsets;
	P.records = d_records; P.totals = W.totals; P.capacity = capacity;
	for (int i = 0; i < AGB_MAXDELIM + 2; i++) { P.dfold[i] = d.delim_fold[i]; P.delim[i] = d.delim[i] | d.delim_fold[i]; }
	P.L = d.L; P.kind = d.delim_kind;
	W.ord_virt = (d.L == 1 && d.delim[0] == '\n') ? 1 : 0;
	/* bitap.c:151-156: j starts at -1 when the text begins with the user's delimiter (asearch0() has no such correction) */
	/* (this one check is byte for byte against the delimiter as typed, also under -i: bitap.c:151-154 compares old_D_pat) */
	P.j0 = (d.user_delim && d.engine != AGB_ENGINE_ASEARCH0 && n >= (uint64_t)d.L && memcmp(h_head, d.delim, (size_t)d.L) == 0) ? -1 : 0;
	W.ord_j0 = P.j0;
	if (blocks_counted) { k_ord_tiles<<<(unsigned)((tiles * 32 + 255) / 256), 256, 0, st>>>(P, tiles); g_launches++; }     /* stage 1 counted the blocks */
	else { k_delim_count<<<(unsigned)tiles, ORD_THREADS, 0, st>>>(P); g_launches++; }
	const uint64_t nb = (tiles + SCAN_BLOCK - 1) / SCAN_BLOCK;
	if (tiles > 4 * SCAN_BLOCK && nb <= W.scan_cap) {
		/* two million tile counts at 64 GiB: one block would take 1.6 ms over them */
		k_scan_partial<<<(unsigned)nb, 1024, 0, st>>>(W.tile_counts, tiles, W.scan_sums, nullptr);
		k_scan_tiles<<<1, 1024, 0, st>>>(W.scan_sums, W.scan_offs, nb, W.totals + 13);
		k_scan_apply<<<(unsigned)nb, 1024, 0, st>>>(W.tile_counts, tiles, W.scan_offs, W.tile_offsets, nullptr);
		g_launches += 3;
	} else { k_scan_tiles<<<1, 1024, 0, st>>>(W.tile_counts, W.tile_offsets, tiles, W.totals + 13); g_launches++; }
	if (d_records && capacity) {
		/* the list length is on the device (totals[0]); one thread per possible entry, bounded by the capacity */
		CUDA_TRY(cudaMemcpyAsync(W.h_totals, W.totals, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
		CUDA_TRY(cudaStreamSynchronize(st));
		const uint64_t nrec = std::min<uint64_t>(W.h_totals[0], capacity);
		if (nrec) { k_ordinals<<<(unsigned)((nrec + 255) / 256), 256, 0, st>>>(P); g_launches++; }
	}
	CUDA_TRY(cudaGetLastError());
	return AGB_OK;
}

