// Gzip output on the device: the compression half of Writer::writeInternal (src/writer.cpp:110-126, libdeflate_gzip_compress
// once per buffer flush on the writer thread), for the text the writers receive.  Every FPL_GZIP_SEGMENT-byte segment of a
// piece becomes one complete RFC 1952 member; segments are independent (no match reaches outside its segment), so one CTA
// compresses one segment with everything it needs in shared memory:
//   k_gzip_deflate   load the segment; CRC-32 per thread over 256-byte chunks, combined by GF(2) shifts
//                    match finding: 4-byte hash, a candidate per position = the nearest earlier position with the same hash
//                      (exact among a thread's own 8 positions of a 2048-position tile, else the table as the previous tiles
//                      left it; each bucket keeps the largest position by compare-and-swap), verified for 3 bytes and
//                      within 32 KiB
//                    greedy parse: one lane walks p += len, skipping candidate-free runs 32 positions at a time; a
//                      length-3 match farther than 4 KiB is left as literals (it costs more than they do)
//                    symbol histograms; code lengths by the in-place minimum-redundancy algorithm of Moffat and Katajainen,
//                      limited to 15 (literal/length, distance) and 7 (code-length alphabet) bits by moving leaves down until
//                      the Kraft sum is exactly one; canonical codes; the 16/17/18 run-length coding of RFC 1951 §3.2.7
//                    one dynamic-Huffman block, or stored blocks when those are not larger; the token bits are placed by an
//                      exclusive scan of the per-thread bit counts, whole words stored, boundary words atomicOr-ed
//   cub scan         member sizes -> offsets
//   k_gzip_compact   the members back to back
// The bytes are a pure function of the input: no step depends on which thread wins a race.
// Included once, by fpl_emit.cu: the encoder is compiled in the translation unit that assembles the output text.
#pragma once
#include <cub/device/device_scan.cuh>
#include "fpl_gzip.h"

namespace {

constexpr int GZ_THREADS = 256;
constexpr int GZ_SEG = FPL_GZIP_SEGMENT;
constexpr int GZ_CHUNK = GZ_SEG / GZ_THREADS;     // positions per thread in the scan / CRC phases
constexpr int GZ_TILE = 8;                        // positions per thread per match-finding tile
constexpr int GZ_HASH_BITS = 14;
constexpr int GZ_WINDOW = 32768;
constexpr int GZ_MAX_MATCH = 258;
constexpr int GZ_WORDS = GZ_SEG / 32;
constexpr int GZ_DATA_BYTES = GZ_SEG + 16;
constexpr int GZ_DIST_BYTES = GZ_SEG * 2;
constexpr int GZ_HEAD_BYTES = (1 << GZ_HASH_BITS) * 2;
constexpr int GZ_SMEM = GZ_DATA_BYTES + GZ_DIST_BYTES + GZ_HEAD_BYTES;
constexpr uint32_t GZ_NONE = 0xFFFFFFFFu;

// Everything after match finding; lives where the hash table was.
struct GzWork {
    uint32_t mbits[GZ_WORDS];        // position has a verified candidate
    uint32_t sbits[GZ_WORDS];        // position starts a token of the parse
    uint32_t hist[288];              // literal/length symbols
    uint32_t histd[32];              // distance symbols
    int32_t A[288];                  // minimum-redundancy workspace: weights in, code lengths out
    int32_t Ad[32];
    uint16_t sym[288];               // used symbols by ascending (count, symbol)
    uint16_t symd[32];
    uint8_t len[288], lend[32], cllen[20];
    uint16_t code[288], coded[32], clcode[20];   // bit-reversed canonical codes
    int32_t cnt[16], cntd[16];
    uint32_t clhist[20];
    int32_t clA[20];
    uint16_t clsym[20];
    uint16_t rle[320];               // code-length sequence: symbol | extra << 5
    uint32_t chunk_bits[GZ_THREADS];
    uint32_t chunk_crc[GZ_THREADS];
    int32_t hlit, hdist, hclen, nrle, header_bits, stored;
    uint32_t deflate_bytes, token_bits;
};
static_assert(sizeof(GzWork) <= GZ_HEAD_BYTES, "GzWork must fit in the hash table's space");

__constant__ uint8_t c_clorder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
// x^(2^k) mod the CRC-32 polynomial, reflected
__constant__ uint32_t c_x2n[32] = {
    0x40000000, 0x20000000, 0x08000000, 0x00800000, 0x00008000, 0xedb88320, 0xb1e6b092, 0xa06a2517, 0xed627dae, 0x88d14467,
    0xd7bbfe6a, 0xec447f11, 0x8e7ea170, 0x6427800e, 0x4d47bae0, 0x09fe548f, 0x83852d0f, 0x30362f1a, 0x7b5a9cc3, 0x31fec169,
    0x9fec022a, 0x6c8dedc4, 0x15d6874d, 0x5fde7a4e, 0xbad90e37, 0x2e4e5eef, 0x4eaba214, 0xa8a472c0, 0x429a969e, 0x148d302a,
    0xc40ba6d0, 0xc4e22c3c};

__device__ __forceinline__ uint32_t gf2_mult(uint32_t a, uint32_t b) {    // a * b mod P (reflected)
    uint32_t m = 1u << 31, p = 0;
    while (m) {
        if (a & m) p ^= b;
        m >>= 1;
        b = (b >> 1) ^ (0xedb88320u & (0u - (b & 1u)));
    }
    return p;
}

// crc32(A || B) from crc32(A), crc32(B) and |B|
__device__ uint32_t crc32_combine(uint32_t a, uint32_t b, uint32_t len_b) {
    uint32_t x = 1u << 31;                        // x^(8 |B|) mod P
    for (int k = 3; len_b; len_b >>= 1, k++)
        if (len_b & 1) x = gf2_mult(c_x2n[k & 31], x);
    return gf2_mult(x, a) ^ b;
}

__device__ __forceinline__ void len_code(int L, int& sym, int& nb, int& extra) {
    if (L == 258) { sym = 285; nb = 0; extra = 0; return; }
    const int v = L - 3;
    if (v < 8) { sym = 257 + v; nb = 0; extra = 0; return; }
    const int lg = 31 - __clz(v);
    nb = lg - 2;
    sym = 257 + 4 * (nb + 1) + ((v >> nb) & 3);
    extra = v & ((1 << nb) - 1);
}

__device__ __forceinline__ void dist_code(int d, int& sym, int& nb, int& extra) {
    const int v = d - 1;
    if (v < 4) { sym = v; nb = 0; extra = 0; return; }
    const int lg = 31 - __clz(v);
    nb = lg - 1;
    sym = 2 * lg + ((v >> nb) & 1);
    extra = v & ((1 << nb) - 1);
}

// Writes a run of bits that one thread owns: words wholly inside the run are stored, the first and the last (shared with
// whoever owns the neighbouring runs) are OR-ed in.  The target words start at zero.
struct BitSink {
    uint32_t* words;
    int64_t word;
    uint64_t acc;
    int nacc;
    bool first;
    __device__ __forceinline__ BitSink(uint32_t* w, int64_t bitpos) : words(w), word(bitpos >> 5), acc(0), nacc((int)(bitpos & 31)), first(true) {}
    __device__ __forceinline__ void put(uint32_t v, int nb) {      // nb <= 32
        acc |= (uint64_t)v << nacc;
        nacc += nb;
        if (nacc >= 32) {
            if (first) atomicOr(&words[word], (uint32_t)acc);
            else words[word] = (uint32_t)acc;
            first = false;
            word++;
            acc >>= 32;
            nacc -= 32;
        }
    }
    __device__ __forceinline__ void finish() { if (nacc > 0) atomicOr(&words[word], (uint32_t)acc); }
};

__device__ void set_range(uint32_t* bits, int lo, int hi) {
    while (lo < hi) {
        const int s = lo & 31, k = min(32 - s, hi - lo);
        bits[lo >> 5] |= (k == 32 ? ~0u : ((1u << k) - 1u)) << s;
        lo += k;
    }
}

// Code lengths for m >= 2 used symbols whose counts A[0..m) ascend (sym[] names them), limited to maxbits.  len[] must be 0.
__device__ void huff_lengths(int32_t* A, const uint16_t* sym, int m, int maxbits, uint8_t* len, int32_t* cnt) {
    // Moffat & Katajainen, in place: pass 1 pairs the two lightest items (leaf or internal) and records parents, pass 2 turns
    // parents into internal-node depths, pass 3 turns those into leaf depths (A[0] = deepest)
    A[0] += A[1];
    int root = 0, leaf = 2;
    for (int next = 1; next < m - 1; next++) {
        if (leaf >= m || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = next; }
        else A[next] = A[leaf++];
        if (leaf >= m || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = next; }
        else A[next] += A[leaf++];
    }
    A[m - 2] = 0;
    for (int next = m - 3; next >= 0; next--) A[next] = A[A[next]] + 1;
    int avail = 1, used = 0, depth = 0, next = m - 1;
    root = m - 2;
    while (avail > 0) {
        while (root >= 0 && A[root] == depth) { used++; root--; }
        while (avail > used) { A[next--] = depth; avail--; }
        avail = 2 * used; depth++; used = 0;
    }
    for (int i = 0; i <= maxbits; i++) cnt[i] = 0;
    for (int i = 0; i < m; i++) cnt[min(A[i], maxbits)]++;
    // too-deep leaves now sit at maxbits; while the Kraft sum exceeds one, move a leaf one level down and hang a
    // maxbits leaf beside it (each step lowers the sum by one unit of 2^-maxbits)
    uint32_t total = 0;
    for (int i = maxbits; i > 0; i--) total += (uint32_t)cnt[i] << (maxbits - i);
    while (total != (1u << maxbits)) {
        cnt[maxbits]--;
        for (int i = maxbits - 1; i > 0; i--)
            if (cnt[i]) { cnt[i]--; cnt[i + 1] += 2; break; }
        total--;
    }
    int j = m;                      // the most frequent symbols get the shortest codes
    for (int b = 1; b <= maxbits; b++)
        for (int k = cnt[b]; k > 0; k--) len[sym[--j]] = (uint8_t)b;
}

// fewer than two used symbols: the used one (if any) and symbol 0 or 1 get length 1 (a complete code, as zlib's build_tree)
__device__ void huff_lengths_small(const uint16_t* sym, int m, uint8_t* len) {
    if (m == 0) { len[0] = 1; len[1] = 1; }
    else { len[sym[0]] = 1; len[sym[0] == 0 ? 1 : 0] = 1; }
}

// canonical codes (RFC 1951 §3.2.2), stored bit-reversed for LSB-first output
__device__ void huff_codes(const uint8_t* len, int nsym, uint16_t* code, int32_t* cnt) {
    for (int i = 0; i < 16; i++) cnt[i] = 0;
    for (int s = 0; s < nsym; s++) cnt[len[s]]++;
    cnt[0] = 0;
    int c = 0, prev = 0;
    for (int b = 1; b < 16; b++) { c = (c + prev) << 1; prev = cnt[b]; cnt[b] = c; }
    for (int s = 0; s < nsym; s++)
        if (len[s]) code[s] = (uint16_t)(__brev((unsigned)cnt[len[s]]++) >> (32 - len[s]));
}

__global__ void __launch_bounds__(GZ_THREADS, 1)
k_gzip_deflate(const GzSeg* __restrict__ segs, uint8_t* __restrict__ slots, int64_t* __restrict__ sizes) {
    extern __shared__ __align__(16) uint8_t gz_smem[];
    uint8_t* data = gz_smem;
    uint16_t* dist = reinterpret_cast<uint16_t*>(gz_smem + GZ_DATA_BYTES);
    uint16_t* head = reinterpret_cast<uint16_t*>(gz_smem + GZ_DATA_BYTES + GZ_DIST_BYTES);
    GzWork& W = *reinterpret_cast<GzWork*>(gz_smem + GZ_DATA_BYTES + GZ_DIST_BYTES);
    const GzSeg sg = segs[blockIdx.x];
    const int n = sg.len;
    const int tid = threadIdx.x;
    uint8_t* out = slots + (int64_t)blockIdx.x * FPL_GZIP_SLOT;

    for (int i = tid; i < n; i += GZ_THREADS) data[i] = sg.src[i];
    if (tid < 16) data[n + tid] = 0;
    for (int i = tid; i < (1 << GZ_HASH_BITS); i += GZ_THREADS) head[i] = 0;
    __syncthreads();

    // CRC-32 of this thread's chunk (kept in a register until the hash table's space is free)
    uint32_t crc = 0;
    {
        const int lo = tid * GZ_CHUNK, hi = min(n, lo + GZ_CHUNK);
        if (lo < hi) {
            uint32_t c = 0xFFFFFFFFu;
            for (int i = lo; i < hi; i++) {
                c ^= data[i];
#pragma unroll
                for (int k = 0; k < 8; k++) c = (c >> 1) ^ (0xedb88320u & (0u - (c & 1u)));
            }
            crc = ~c;
        }
    }

    // ---- match finding, tile by tile in position order ----
    for (int base = 0; base < n; base += GZ_THREADS * GZ_TILE) {
        const int p0 = base + tid * GZ_TILE;
        uint32_t hs[GZ_TILE];
        int cand[GZ_TILE];
#pragma unroll
        for (int k = 0; k < GZ_TILE; k++) {
            const int p = p0 + k;
            hs[k] = GZ_NONE;
            if (p + 4 <= n) {
                const uint32_t v = (uint32_t)data[p] | (uint32_t)data[p + 1] << 8 | (uint32_t)data[p + 2] << 16 | (uint32_t)data[p + 3] << 24;
                hs[k] = (v * 2654435761u) >> (32 - GZ_HASH_BITS);
            }
        }
#pragma unroll
        for (int k = 0; k < GZ_TILE; k++) {
            int c = -1;
#pragma unroll
            for (int j = 0; j < k; j++)
                if (hs[j] == hs[k]) c = p0 + j;
            if (hs[k] != GZ_NONE && c < 0) c = (int)head[hs[k]] - 1;
            cand[k] = hs[k] == GZ_NONE ? -1 : c;
        }
        __syncthreads();
        // each bucket ends up holding the largest position that hashes to it (+1; 0 = empty): a thread offers its last
        // position of each hash, and a compare-and-swap on the 32-bit word holding the bucket keeps the larger value
#pragma unroll
        for (int k = 0; k < GZ_TILE; k++) {
            bool last = hs[k] != GZ_NONE;
#pragma unroll
            for (int j = k + 1; j < GZ_TILE; j++)
                if (hs[j] == hs[k]) last = false;
            if (!last) continue;
            uint32_t* word = reinterpret_cast<uint32_t*>(head) + (hs[k] >> 1);
            const unsigned sh = (hs[k] & 1u) * 16;
            const uint32_t mine = (uint32_t)(p0 + k + 1);
            uint32_t cur = atomicCAS(word, 0u, 0u);
            while (((cur >> sh) & 0xFFFFu) < mine) {
                const uint32_t prev = atomicCAS(word, cur, (cur & ~(0xFFFFu << sh)) | mine << sh);
                if (prev == cur) break;
                cur = prev;
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < GZ_TILE; k++) {
            const int p = p0 + k, c = cand[k];
            if (p >= n) break;
            int d = 0;
            if (c >= 0 && p - c <= GZ_WINDOW && data[c] == data[p] && data[c + 1] == data[p + 1] && data[c + 2] == data[p + 2]) d = p - c;
            dist[p] = (uint16_t)d;
        }
    }
    __syncthreads();

    // ---- the hash table's space becomes GzWork ----
    const int nwords = (n + 31) >> 5;
    for (int w = tid; w < GZ_WORDS; w += GZ_THREADS) {
        uint32_t m = 0;
        if (w < nwords)
            for (int i = 0; i < 32; i++) {
                const int p = w * 32 + i;
                if (p < n && dist[p]) m |= 1u << i;
            }
        W.mbits[w] = m;
        W.sbits[w] = 0;
    }
    for (int i = tid; i < 288; i += GZ_THREADS) W.hist[i] = 0;
    if (tid < 32) W.histd[tid] = 0;
    W.chunk_crc[tid] = crc;
    __syncthreads();

    // ---- greedy parse: one lane ----
    if (tid == 0) {
        int p = 0;
        while (p < n) {
            int w = p >> 5;
            uint32_t m = W.mbits[w] & (~0u << (p & 31));
            while (!m && ++w < nwords) m = W.mbits[w];
            const int q = m ? (w << 5) + __ffs((int)m) - 1 : n;
            set_range(W.sbits, p, q);                          // literals
            if (q >= n) break;
            const int d = dist[q];
            const int maxl = min(GZ_MAX_MATCH, n - q);
            const uint8_t* a = data + q;
            const uint8_t* b = a - d;
            int L = 3;
            while (L < maxl && a[L] == b[L]) L++;
            W.sbits[q >> 5] |= 1u << (q & 31);
            if (L == 3 && d > 4096) { dist[q] = 0; p = q + 1; }
            else { dist[q + 1] = (uint16_t)L; p = q + L; }    // q + 1 lies inside the match: it carries the length
        }
    }
    // CRC-32 of the segment: pairwise combination of the chunks' CRCs
    for (int s = 1; s < GZ_THREADS; s <<= 1) {
        __syncthreads();
        if ((tid & (2 * s - 1)) == 0) {
            const int rlo = (tid + s) * GZ_CHUNK;
            const int rlen = min(n - rlo, s * GZ_CHUNK);
            if (rlen > 0) W.chunk_crc[tid] = crc32_combine(W.chunk_crc[tid], W.chunk_crc[tid + s], (uint32_t)rlen);
        }
    }
    __syncthreads();

    // ---- symbol histograms ----
    const int clo = tid * GZ_CHUNK, chi = min(n, clo + GZ_CHUNK);
    for (int p = clo; p < chi; p++) {
        if (!(W.sbits[p >> 5] >> (p & 31) & 1u)) continue;
        const int d = dist[p];
        if (!d) { atomicAdd(&W.hist[data[p]], 1u); continue; }
        int ls, lnb, lx, ds, dnb, dx;
        len_code(dist[p + 1], ls, lnb, lx);
        dist_code(d, ds, dnb, dx);
        atomicAdd(&W.hist[ls], 1u);
        atomicAdd(&W.histd[ds], 1u);
    }
    if (tid == 0) atomicAdd(&W.hist[256], 1u);       // end of block
    __syncthreads();

    // ---- used symbols in ascending (count, symbol) order ----
    for (int s = tid; s < 286 + 30; s += GZ_THREADS) {
        const bool isd = s >= 286;
        const uint32_t* h = isd ? W.histd : W.hist;
        const int ns = isd ? 30 : 286, x = isd ? s - 286 : s;
        const uint32_t f = h[x];
        if (!f) continue;
        int r = 0;
        for (int y = 0; y < ns; y++) {
            const uint32_t g = h[y];
            r += g && (g < f || (g == f && y < x));
        }
        if (isd) { W.Ad[r] = (int32_t)f; W.symd[r] = (uint16_t)x; }
        else { W.A[r] = (int32_t)f; W.sym[r] = (uint16_t)x; }
    }
    __syncthreads();

    // ---- code lengths and codes: literal/length on lane 0 of warp 0, distance on lane 0 of warp 1 ----
    if (tid == 0 || tid == 32) {
        const bool isd = tid == 32;
        const uint32_t* h = isd ? W.histd : W.hist;
        const int ns = isd ? 30 : 286;
        uint8_t* len = isd ? W.lend : W.len;
        int m = 0;
        for (int s = 0; s < (isd ? 32 : 288); s++) { len[s] = 0; if (s < ns) m += h[s] != 0; }
        if (m < 2) huff_lengths_small(isd ? W.symd : W.sym, m, len);
        else huff_lengths(isd ? W.Ad : W.A, isd ? W.symd : W.sym, m, 15, len, isd ? W.cntd : W.cnt);
        huff_codes(len, ns, isd ? W.coded : W.code, isd ? W.cntd : W.cnt);
    }
    __syncthreads();

    // ---- block header: code-length sequence, its code, the header's size ----
    if (tid == 0) {
        int hlit = 286, hdist = 30;
        while (hlit > 257 && !W.len[hlit - 1]) hlit--;
        while (hdist > 1 && !W.lend[hdist - 1]) hdist--;
        const int total = hlit + hdist;
        int nr = 0, i = 0;
        for (int s = 0; s < 20; s++) W.clhist[s] = 0;
        while (i < total) {
            const int v = i < hlit ? W.len[i] : W.lend[i - hlit];
            int r = 1;
            while (i + r < total && (i + r < hlit ? W.len[i + r] : W.lend[i + r - hlit]) == v) r++;
            i += r;
            if (v == 0) {
                while (r >= 11) { const int k = min(r, 138); W.rle[nr++] = (uint16_t)(18 | (k - 11) << 5); W.clhist[18]++; r -= k; }
                if (r >= 3) { W.rle[nr++] = (uint16_t)(17 | (r - 3) << 5); W.clhist[17]++; r = 0; }
            } else {
                W.rle[nr++] = (uint16_t)v; W.clhist[v]++; r--;
                while (r >= 3) { const int k = min(r, 6); W.rle[nr++] = (uint16_t)(16 | (k - 3) << 5); W.clhist[16]++; r -= k; }
            }
            for (; r > 0; r--) { W.rle[nr++] = (uint16_t)v; W.clhist[v]++; }
        }
        // code-length alphabet: 19 symbols, sorted by insertion
        int m = 0;
        for (int s = 0; s < 19; s++) {
            W.cllen[s] = 0;
            const uint32_t f = W.clhist[s];
            if (!f) continue;
            int j = m++;
            while (j > 0 && (uint32_t)W.clA[j - 1] > f) { W.clA[j] = W.clA[j - 1]; W.clsym[j] = W.clsym[j - 1]; j--; }
            W.clA[j] = (int32_t)f; W.clsym[j] = (uint16_t)s;
        }
        if (m < 2) huff_lengths_small(W.clsym, m, W.cllen);
        else huff_lengths(W.clA, W.clsym, m, 7, W.cllen, W.cnt);
        huff_codes(W.cllen, 19, W.clcode, W.cnt);
        int hclen = 19;
        while (hclen > 4 && !W.cllen[c_clorder[hclen - 1]]) hclen--;
        int bits = 3 + 5 + 5 + 4 + 3 * hclen;
        for (int k = 0; k < nr; k++) {
            const int s = W.rle[k] & 31;
            bits += W.cllen[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
        }
        W.hlit = hlit; W.hdist = hdist; W.hclen = hclen; W.nrle = nr; W.header_bits = bits;
    }
    __syncthreads();

    // ---- bits of this thread's tokens ----
    uint32_t mybits = 0;
    for (int p = clo; p < chi; p++) {
        if (!(W.sbits[p >> 5] >> (p & 31) & 1u)) continue;
        const int d = dist[p];
        if (!d) { mybits += W.len[data[p]]; continue; }
        int ls, lnb, lx, ds, dnb, dx;
        len_code(dist[p + 1], ls, lnb, lx);
        dist_code(d, ds, dnb, dx);
        mybits += W.len[ls] + lnb + W.lend[ds] + dnb;
    }
    W.chunk_bits[tid] = mybits;
    __syncthreads();
    if (tid == 0) {
        uint32_t run = 0;
        for (int t = 0; t < GZ_THREADS; t++) { const uint32_t b = W.chunk_bits[t]; W.chunk_bits[t] = run; run += b; }
        W.token_bits = run;
        const uint32_t dbits = (uint32_t)W.header_bits + run + W.len[256];
        const uint32_t dbytes = (dbits + 7) >> 3;
        const uint32_t nblk = (uint32_t)(n + 65534) / 65535;
        const uint32_t sbytes = (uint32_t)n + 5 * nblk;
        W.stored = dbytes > sbytes;
        W.deflate_bytes = W.stored ? sbytes : dbytes;
        sizes[blockIdx.x] = 10 + (int64_t)W.deflate_bytes + 8;
    }
    __syncthreads();
    const uint32_t crc_all = W.chunk_crc[0];
    const int member = 10 + (int)W.deflate_bytes + 8;

    if (W.stored) {
        // stored blocks of at most 65535 bytes, each behind a 5-byte header (byte-aligned: the member header is 10 bytes)
        for (int i = tid; i < n; i += GZ_THREADS) out[10 + 5 * (i / 65535 + 1) + i] = data[i];
        if (tid == 0) {
            const uint8_t hdr[10] = {0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 0, 0xff};
            for (int k = 0; k < 10; k++) out[k] = hdr[k];
            const int nblk = (n + 65534) / 65535;
            for (int b = 0; b < nblk; b++) {
                uint8_t* o = out + 10 + b * (65535 + 5);
                const int len = min(65535, n - b * 65535);
                o[0] = (uint8_t)(b == nblk - 1);
                o[1] = (uint8_t)len; o[2] = (uint8_t)(len >> 8);
                o[3] = (uint8_t)~len; o[4] = (uint8_t)(~len >> 8);
            }
            uint8_t* t = out + member - 8;
            for (int k = 0; k < 4; k++) { t[k] = (uint8_t)(crc_all >> (8 * k)); t[4 + k] = (uint8_t)((uint32_t)n >> (8 * k)); }
        }
        return;
    }

    uint32_t* words = reinterpret_cast<uint32_t*>(out);
    for (int i = tid; i < (member + 3) / 4; i += GZ_THREADS) words[i] = 0;
    __syncthreads();
    if (tid == 0) {
        BitSink o(words, 0);
        o.put(0x00088b1fu, 32);                             // ID1 ID2 CM=8 FLG=0
        o.put(0, 32);                                       // MTIME
        o.put(0xff00u, 16);                                 // XFL=0 OS=255
        o.put(1, 1);                                        // BFINAL
        o.put(2, 2);                                        // BTYPE 10: dynamic Huffman codes
        o.put((uint32_t)(W.hlit - 257), 5);
        o.put((uint32_t)(W.hdist - 1), 5);
        o.put((uint32_t)(W.hclen - 4), 4);
        for (int k = 0; k < W.hclen; k++) o.put(W.cllen[c_clorder[k]], 3);
        for (int k = 0; k < W.nrle; k++) {
            const int s = W.rle[k] & 31, x = W.rle[k] >> 5;
            o.put(W.clcode[s], W.cllen[s]);
            if (s >= 16) o.put((uint32_t)x, s == 16 ? 2 : s == 17 ? 3 : 7);
        }
        o.finish();
    }
    {
        BitSink o(words, 80 + (int64_t)W.header_bits + W.chunk_bits[tid]);
        for (int p = clo; p < chi; p++) {
            if (!(W.sbits[p >> 5] >> (p & 31) & 1u)) continue;
            const int d = dist[p];
            if (!d) { const int c = data[p]; o.put(W.code[c], W.len[c]); continue; }
            int ls, lnb, lx, ds, dnb, dx;
            len_code(dist[p + 1], ls, lnb, lx);
            dist_code(d, ds, dnb, dx);
            o.put((uint32_t)W.code[ls] | (uint32_t)lx << W.len[ls], W.len[ls] + lnb);
            o.put((uint32_t)W.coded[ds] | (uint32_t)dx << W.lend[ds], W.lend[ds] + dnb);
        }
        o.finish();
    }
    __syncthreads();
    if (tid == 0) {                                         // end of block, then CRC-32 and ISIZE
        BitSink o(words, 80 + (int64_t)W.header_bits + W.token_bits);
        o.put(W.code[256], W.len[256]);
        o.finish();
        BitSink t(words, (int64_t)(member - 8) * 8);
        t.put(crc_all, 32);
        t.put((uint32_t)n, 32);
        t.finish();
    }
}

__global__ void __launch_bounds__(256)
k_gzip_compact(const uint8_t* __restrict__ slots, const int64_t* __restrict__ off, uint8_t* __restrict__ dst) {
    const int64_t s = blockIdx.x;
    const int64_t o = off[s];
    const int n = (int)(off[s + 1] - o);
    const uint32_t* src = reinterpret_cast<const uint32_t*>(slots + s * FPL_GZIP_SLOT);
    uint8_t* d = dst + o;
    for (int i = threadIdx.x; 4 * i < n; i += blockDim.x) {
        const uint32_t w = src[i];
        const int k = min(4, n - 4 * i);
        for (int j = 0; j < k; j++) d[4 * i + j] = (uint8_t)(w >> (8 * j));
    }
}

}  // namespace

#define CKG(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { snprintf(err, errlen, "%s failed: %s", #call, cudaGetErrorString(e_)); return -1; } } while (0)

int fpl_gzip_grow(void** p, int64_t* cap, int64_t need, char* err, size_t errlen) {
    if (need <= *cap) return 0;
    int64_t c = *cap ? *cap : (1 << 16);
    while (c < need) c *= 2;
    cudaFree(*p); *p = nullptr; *cap = 0;
    CKG(cudaMalloc(p, (size_t)c));
    *cap = c;
    return 0;
}

int fpl_gzip_plan(FplGzip* g, const uint8_t* const* piece, const int64_t* piece_bytes, int n_pieces, cudaStream_t s, char* err,
                  size_t errlen) {
    g->h_segs.clear();
    g->h_first.assign(1, 0);
    int64_t total = 0;
    for (int i = 0; i < n_pieces; i++) {
        for (int64_t o = 0; o < piece_bytes[i]; o += FPL_GZIP_SEGMENT)
            g->h_segs.push_back({piece[i] + o, (int32_t)(piece_bytes[i] - o < FPL_GZIP_SEGMENT ? piece_bytes[i] - o : FPL_GZIP_SEGMENT), 0});
        g->h_first.push_back((int64_t)g->h_segs.size());
        total += piece_bytes[i];
    }
    const int64_t m = g->n_segs = (int64_t)g->h_segs.size();
    if (!m) return 0;
    if (fpl_gzip_grow((void**)&g->d_segs, &g->cap_segs, (int64_t)sizeof(GzSeg) * m, err, errlen)) return -1;
    if (fpl_gzip_grow((void**)&g->d_slots, &g->cap_slots, (int64_t)FPL_GZIP_SLOT * m, err, errlen)) return -1;
    if (fpl_gzip_grow((void**)&g->d_size, &g->cap_size, (int64_t)sizeof(int64_t) * (m + 1), err, errlen)) return -1;
    if (fpl_gzip_grow((void**)&g->d_off, &g->cap_off, (int64_t)sizeof(int64_t) * (m + 1), err, errlen)) return -1;
    if (fpl_gzip_grow((void**)&g->d_out, &g->cap_out, FPL_GZIP_BOUND(total, n_pieces) + 16, err, errlen)) return -1;
    CKG(cudaMemcpyAsync(g->d_segs, g->h_segs.data(), sizeof(GzSeg) * m, cudaMemcpyHostToDevice, s));
    CKG(cudaMemsetAsync(g->d_size + m, 0, sizeof(int64_t), s));
    CKG(cudaFuncSetAttribute(k_gzip_deflate, cudaFuncAttributeMaxDynamicSharedMemorySize, GZ_SMEM));
    return 0;
}

void fpl_gzip_deflate(FplGzip* g, cudaStream_t s) {
    k_gzip_deflate<<<(unsigned)g->n_segs, GZ_THREADS, GZ_SMEM, s>>>(g->d_segs, g->d_slots, g->d_size);
}

int fpl_gzip_offsets(FplGzip* g, cudaStream_t s, char* err, size_t errlen) {
    size_t tb = 0;
    CKG(cub::DeviceScan::ExclusiveSum(nullptr, tb, g->d_size, g->d_off, g->n_segs + 1, s));
    if (fpl_gzip_grow(&g->d_tmp, &g->cap_tmp, (int64_t)tb + 256, err, errlen)) return -1;
    CKG(cub::DeviceScan::ExclusiveSum(g->d_tmp, tb, g->d_size, g->d_off, g->n_segs + 1, s));
    return 0;
}

void fpl_gzip_compact(FplGzip* g, cudaStream_t s) {
    k_gzip_compact<<<(unsigned)g->n_segs, 256, 0, s>>>(g->d_slots, g->d_off, g->d_out);
}

int fpl_gzip_piece_sizes(FplGzip* g, int64_t* out_piece_bytes, cudaStream_t s, char* err, size_t errlen) {
    const int64_t m = g->n_segs;
    g->h_off.assign((size_t)m + 1, 0);
    if (m) CKG(cudaMemcpyAsync(g->h_off.data(), g->d_off, sizeof(int64_t) * (m + 1), cudaMemcpyDeviceToHost, s));
    CKG(cudaStreamSynchronize(s));
    for (size_t i = 0; i + 1 < g->h_first.size(); i++) out_piece_bytes[i] = g->h_off[g->h_first[i + 1]] - g->h_off[g->h_first[i]];
    return 0;
}

void fpl_gzip_free(FplGzip* g) {
    cudaFree(g->d_in); cudaFree(g->d_segs); cudaFree(g->d_slots); cudaFree(g->d_size); cudaFree(g->d_off); cudaFree(g->d_tmp);
    cudaFree(g->d_out);
    *g = FplGzip();
}
