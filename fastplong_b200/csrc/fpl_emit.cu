// Output assembly on the device (SURVEY §8f row 2, device half): Read::appendToString / appendToStringWithTag
// (src/read.cpp:119-173) for every output read of a chunk of FASTQ text that fpl_process_fastq_host has just processed,
// in the order processSingleEnd emits them (src/seprocessor.cpp:264-288).  The chunk, its record table, the per-read
// results and — with --mask / --break — the list of output reads and the masked bases are already in HBM, so the text
// the two writer threads receive is a stream compaction:
//   k_emit_sizes   thread per read: bytes this read contributes to --out and to --failed_out
//   cub scan       one exclusive sum over both size vectors -> where each read's text starts
//   k_emit_copy    warp per read: name (+ "r<k>-" / "split-by-adapter-…-" after the '@', or " <reason>" behind it), the
//                  window of the bases, the '+' line as it was, the window of the qualities; 16-byte stores, source words
//                  re-aligned by funnel shifts
// Both kernels walk a read with the same code (walk_read) and differ in the sink only, so the sizes cannot drift from
// the text.
#include <cub/device/device_scan.cuh>
#include "fpl_device.cuh"
#include "fpl_emit.h"

namespace {

// Read::breakByGap's name tags (src/read.cpp:204,209) and the --failed_out reasons by filter result code
// (src/common.h:55-64)
__constant__ char c_left[24] = "split-by-adapter-left-";
__constant__ char c_right[24] = "split-by-adapter-right-";
__constant__ char c_failed[32][24] = {
    "passed", "", "", "", "failed_polyx_filter", "", "", "", "failed_bad_overlap", "", "", "",
    "failed_too_many_n_bases", "", "", "", "failed_too_short", "failed_too_long", "", "",
    "failed_quality_filter", "", "", "", "failed_low_complexity", "", "", "", "", "", "", ""};
__constant__ int c_failed_len[32] = {6, 0, 0, 0, 19, 0, 0, 0, 18, 0, 0, 0, 23, 0, 0, 0, 16, 15, 0, 0, 21, 0, 0, 0, 21, 0, 0, 0, 0, 0, 0, 0};

__device__ __forceinline__ int dec_digits(int v) {
    int nd = 1;
    for (unsigned t = (unsigned)v; t >= 10; t /= 10) nd++;
    return nd;
}

// counts bytes (one thread walks a read)
struct SizeSink {
    int64_t n = 0;
    __device__ __forceinline__ void bytes(const uint8_t*, int64_t k) { n += k; }
    __device__ __forceinline__ void lit(const char*, int k) { n += k; }
    __device__ __forceinline__ void ch(char) { n++; }
    __device__ __forceinline__ void dec(int v) { n += dec_digits(v); }
};

// n bytes from src to dst, any alignment, by one warp.  May read up to 3 bytes past src + n (inside the 64-byte pad every
// source buffer carries).
__device__ __forceinline__ void warp_copy(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, int64_t n, int lane) {
    if (n <= 0) return;
    int head = (int)((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15);
    if (head > n) head = (int)n;
    if (lane < head) dst[lane] = src[lane];
    dst += head; src += head; n -= head;
    const int64_t nv = n >> 4;
    if (nv) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(src);
        const uint32_t* sw = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
        const unsigned sh = (unsigned)(a & 3) * 8;
        uint4* dv = reinterpret_cast<uint4*>(dst);
        for (int64_t k = lane; k < nv; k += 32) {
            const uint32_t* p = sw + 4 * k;
            const uint32_t w0 = __ldg(p), w1 = __ldg(p + 1), w2 = __ldg(p + 2), w3 = __ldg(p + 3);
            uint4 o = make_uint4(w0, w1, w2, w3);
            if (sh) {
                const uint32_t w4 = __ldg(p + 4);
                o = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
                               __funnelshift_r(w3, w4, sh));
            }
            dv[k] = o;
        }
    }
    const int64_t done = nv << 4;
    if (lane < (int)(n - done)) dst[done + lane] = src[done + lane];
}

// writes bytes (one warp walks a read; p is warp-uniform)
struct CopySink {
    uint8_t* p;
    int lane;
    __device__ __forceinline__ void bytes(const uint8_t* s, int64_t k) { warp_copy(p, s, k, lane); p += k; }
    __device__ __forceinline__ void lit(const char* s, int k) { if (lane < k) p[lane] = (uint8_t)s[lane]; p += k; }   // k <= 32
    __device__ __forceinline__ void ch(char c) { if (lane == 0) *p = (uint8_t)c; p++; }
    __device__ __forceinline__ void dec(int v) {
        const int nd = dec_digits(v);
        if (lane < nd) {
            unsigned d = 1;
            for (int i = 0; i < nd - 1 - lane; i++) d *= 10;
            p[lane] = (uint8_t)('0' + ((unsigned)v / d) % 10);
        }
        p += nd;
    }
};

template <class Sink>
__device__ __forceinline__ void put_record(Sink& o, const uint8_t* name, int name_len, int bidx, int side, const char* reason,
                                           int reason_len, const uint8_t* bases, const uint8_t* plus, int plus_len,
                                           const uint8_t* qual, int lo, int len) {
    if ((bidx || side) && name_len > 0) {        // the tag goes between the '@' and the rest of the name line
        o.bytes(name, 1);
        if (bidx) { o.ch('r'); o.dec(bidx); o.ch('-'); }
        if (side) o.lit(side == 2 ? c_right : c_left, side == 2 ? 23 : 22);
        o.bytes(name + 1, name_len - 1);
    } else {
        o.bytes(name, name_len);
    }
    if (reason) { o.ch(' '); o.lit(reason, reason_len); }
    o.ch('\n');
    o.bytes(bases + lo, len);
    o.ch('\n');
    o.bytes(plus, plus_len);
    o.ch('\n');
    o.bytes(qual + lo, len);
    o.ch('\n');
}

// Everything read r sends to the two writers, in the reference's order (src/seprocessor.cpp:264-288): a passing output
// read goes to --out; a failing one goes to --failed_out only when it is the read's only output read, and then as r1
// after the trims (the record's trim window), masked only if that output read is r1 itself.
template <class Sink>
__device__ __forceinline__ void walk_read(const EmitSource& S, int64_t r, bool want_failed, Sink& out, Sink& failed) {
    const fpl_fastq_record fq = S.rec[r];
    const fpl_read_result* rr = S.res + r;
    const int nseg = rr->n_segments;
    const uint32_t flags = rr->flags;
    const uint8_t* name = S.text + fq.name_off;
    const uint8_t* seq = S.text + fq.seq_off;
    const uint8_t* plus = S.text + fq.plus_off;
    const uint8_t* qual = S.text + fq.qual_off;
    const uint8_t* mseq = S.mseq ? S.mseq + S.offsets[r] : seq;
    const int s0 = S.segs ? S.seg_off[2 * r] : 0;
    for (int k = 0; k < nseg; k++) {
        int lo, len, code, side, bidx, is_r1;
        if (S.segs) {
            const fpl_segment sg = S.segs[s0 + k];
            lo = sg.lo; len = sg.len; code = sg.result; side = sg.split_side; bidx = sg.break_index; is_r1 = sg.is_r1;
        } else {
            lo = rr->seg_lo[k]; len = rr->seg_len[k]; code = rr->seg_result[k];
            side = (flags & FPL_FLAG_MIDDLE_ADAPTER) ? ((k == 1 || (flags & FPL_FLAG_SEG0_IS_RIGHT)) ? 2 : 1) : 0;
            bidx = 0; is_r1 = side == 0;
        }
        if (code == FPL_PASS_FILTER) {
            put_record(out, name, fq.name_len, bidx, side, nullptr, 0, mseq, plus, fq.plus_len, qual, lo, len);
        } else if (want_failed && nseg == 1) {
            put_record(failed, name, fq.name_len, 0, 0, c_failed[code & 31], c_failed_len[code & 31], is_r1 ? mseq : seq, plus,
                       fq.plus_len, qual, rr->trim_lo, rr->trim_len);
        }
    }
}

// size[r] = --out bytes of read r, size[n + 1 + r] = --failed_out bytes (size[n] and size[2n + 1] stay 0: the totals
// appear there after the exclusive sum)
__global__ void k_emit_sizes(const EmitSource S, bool want_failed, int64_t* __restrict__ size) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= S.n_reads) return;
    SizeSink out, failed;
    walk_read(S, r, want_failed, out, failed);
    size[r] = out.n;
    size[S.n_reads + 1 + r] = failed.n;
}

__global__ void __launch_bounds__(256)
k_emit_copy(const EmitSource S, bool want_failed, const int64_t* __restrict__ off, uint8_t* __restrict__ d_out,
            uint8_t* __restrict__ d_failed) {
    const int lane = lane_id();
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t n = S.n_reads;
    const int64_t total_out = off[n];
    for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n; r += nwarps) {
        CopySink out{d_out + off[r], lane}, failed{d_failed + (off[n + 1 + r] - total_out), lane};
        walk_read(S, r, want_failed, out, failed);
    }
}

}  // namespace

#define CKM(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { snprintf(err, errlen, "%s failed: %s", #call, cudaGetErrorString(e_)); return -1; } } while (0)

static int growm(void** p, int64_t* cap, int64_t need, char* err, size_t errlen) {
    if (need <= *cap) return 0;
    int64_t c = *cap ? *cap : (1 << 16);
    while (c < need) c *= 2;
    cudaFree(*p); *p = nullptr; *cap = 0;
    CKM(cudaMalloc(p, (size_t)c));
    *cap = c;
    return 0;
}

int fpl_emit_build(FplEmit* e, const EmitSource& src, bool want_failed, cudaStream_t s, char* err, size_t errlen) {
    e->built = false; e->out_bytes = e->failed_bytes = 0; e->with_failed = want_failed;
    const int64_t n = src.n_reads;
    if (n == 0) { e->built = true; return 0; }
    const int64_t m = 2 * n + 2;
    if (growm((void**)&e->d_size, &e->cap_size, (int64_t)sizeof(int64_t) * m, err, errlen)) return -1;
    if (growm((void**)&e->d_off, &e->cap_off, (int64_t)sizeof(int64_t) * m, err, errlen)) return -1;
    CKM(cudaMemsetAsync(e->d_size + n, 0, sizeof(int64_t), s));
    CKM(cudaMemsetAsync(e->d_size + 2 * n + 1, 0, sizeof(int64_t), s));
    k_emit_sizes<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, want_failed, e->d_size);
    size_t tb = 0;
    CKM(cub::DeviceScan::ExclusiveSum(nullptr, tb, e->d_size, e->d_off, m, s));
    if (growm(&e->d_tmp, &e->cap_tmp, (int64_t)tb + 256, err, errlen)) return -1;
    CKM(cub::DeviceScan::ExclusiveSum(e->d_tmp, tb, e->d_size, e->d_off, m, s));
    int64_t total_out = 0, total_both = 0;
    CKM(cudaMemcpyAsync(&total_out, e->d_off + n, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CKM(cudaMemcpyAsync(&total_both, e->d_off + 2 * n + 1, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CKM(cudaStreamSynchronize(s));
    e->out_bytes = total_out;
    e->failed_bytes = total_both - total_out;
    // + 16: a warp's last 16-byte store never needs a bounds test against the next buffer
    if (growm((void**)&e->d_out, &e->cap_out, e->out_bytes + 16, err, errlen)) return -1;
    if (growm((void**)&e->d_failed, &e->cap_failed, e->failed_bytes + 16, err, errlen)) return -1;
    const int64_t want = (n + 7) / 8;
    k_emit_copy<<<(unsigned)(want < 148 * 16 ? want : 148 * 16), 256, 0, s>>>(src, want_failed, e->d_off, e->d_out, e->d_failed);
    CKM(cudaGetLastError());
    e->built = true;
    return 0;
}

void fpl_emit_free(FplEmit* e) {
    cudaFree(e->d_size); cudaFree(e->d_off); cudaFree(e->d_out); cudaFree(e->d_failed); cudaFree(e->d_tmp);
    *e = FplEmit();
}

// The gzip encoder that compresses this text (fpl_emit_fastq_gzip_host) and any other (fpl_gzip_host) is compiled in
// this translation unit.
#include "fpl_gzip.cuh"
