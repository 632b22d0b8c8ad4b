// C-ABI implementation of include/fplgpu.h: context management, device tables, batch tiling and kernel sequencing.
// No CPU fallback anywhere: every entry point fails loudly when CUDA is unusable.
#include <cuda_runtime.h>
#include <limits.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <algorithm>
#include <string>
#include <vector>
#include <dlfcn.h>
#include <nccl.h>
#include "fpl_device.cuh"
#include "fpl_scanplan.h"
#include "fpl_stats.h"
#include "fpl_jit.h"
#include "fpl_ingest.h"
#include "fpl_ext.h"
#include "fpl_emit.h"
#include "fpl_gzip.h"

static_assert(sizeof(fpl_options) == 144, "fpl_options ABI size");
static_assert(sizeof(fpl_segment) == 20 && sizeof(fpl_region) == 12, "segment / region ABI size");
static_assert(sizeof(fpl_read_result) == 64, "fpl_read_result ABI size");
static_assert(sizeof(ReadState) == 64, "ReadState size");
static_assert(sizeof(StatSeg) == 24, "StatSeg size");

// kernel launchers (fpl_trim.cu, fpl_scan.cu, fpl_stats.cu)
void launch_trim(const DevParams&, const DevBatch&, ReadState*, fpl_read_result*, unsigned long long*, cudaStream_t);
void launch_scan(const DevParams&, const DevBatch&, ReadState*, cudaStream_t);
void launch_scan_fast(const DevParams&, const ScanPlan&, const DevBatch&, ReadState*, cudaStream_t);
void launch_final(const DevParams&, const DevBatch&, const ReadState*, fpl_read_result*, StatSeg*, cudaStream_t);
void launch_count(const fpl_read_result*, int64_t, unsigned long long*, bool, cudaStream_t);
int launch_cycle_stats(CycleWs*, const uint8_t*, const uint8_t*, const StatSeg*, int64_t, int64_t, unsigned long long*, int64_t,
                        bool, unsigned long long*, bool, cudaStream_t);
void launch_kmer_fix(const DevBatch&, const fpl_read_result*, unsigned long long*, cudaStream_t);
void launch_read_qual(const DevBatch&, unsigned long long*, unsigned long long*, int64_t, fpl_read_result*, bool, cudaStream_t);
void launch_make_preseg(const DevBatch&, StatSeg*, cudaStream_t);

static thread_local char g_err[512] = "";

static int fail(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return -1;
}

#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) return fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

enum { K_PRESEG, K_CYCLE_PRE, K_QUAL_PRE, K_TRIM, K_SCAN, K_FINAL, K_COUNT, K_CYCLE_POST, K_QUAL_POST, K_KMER_FIX, K_ALLREDUCE, K_GZ_DEFLATE, K_GZ_COMPACT, K_NKERNELS };
static const char* const kKernelNames[K_NKERNELS] = {"k_make_preseg", "k_cycle_stats(pre)", "k_read_qual(pre+post)",
                                                     "k_trim", "k_scan", "k_final", "k_count",
                                                     "k_cycle_stats(post)", "k_read_qual(post)", "k_kmer_fix",
                                                     "nccl_allreduce(stats)", "k_gzip_deflate", "k_gzip_compact"};

struct fpl_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    DevParams P;
    ScanPlan plan;
    FplJitKernel jit;   // specialised scan kernel (NVRTC), fn == nullptr if not used
    FplIngest ingest;   // device-side FASTQ parsing state
    FplExt ext;         // --mask / --break state (variable number of output reads)
    FplEmit emit;       // device-side output text of the last fpl_process_fastq_host chunk (fpl_emit_fastq_host)
    bool emit_valid = false;            // the last call was a successful fpl_process_fastq_host: chunk + records + results in HBM
    FplGzip gz;         // device gzip encoder state (fpl_gzip_host, fpl_emit_fastq_gzip_host)
    bool emit_gz_built = false;         // gz.d_out holds the compressed emit text (out piece, then failed piece)
    bool emit_gz_failed = false;
    int64_t emit_gz_bytes[2] = {0, 0};
    int64_t emit_n = 0;
    int64_t last_bytes = 0;
    bool slots16 = false;               // this batch's read offsets are multiples of 16 (checked: host batches, device ingest)
    int n_adapters = 0;
    uint8_t* d_adapters = nullptr;
    int* d_alen = nullptr;
    uint4* d_peq = nullptr;
    uint32_t* d_peq16 = nullptr;
    uint32_t* d_acode = nullptr;
    unsigned long long* d_peq_long = nullptr;
    int* d_pf_order = nullptr;
    // accumulators
    int64_t C = 0;
    unsigned long long* d_stats[2] = {nullptr, nullptr};
    unsigned long long* d_counters = nullptr;
    int64_t counter_words = 0;
    // per-read work buffers
    int64_t cap_reads = 0;
    ReadState* d_state = nullptr;
    fpl_read_result* d_results = nullptr;
    CycleWs cycle_ws;
    StatSeg* d_preseg = nullptr;
    StatSeg* d_postseg = nullptr;
    int64_t last_n = 0;
    fpl_read_result* last_results = nullptr;  // where the last call's records live (device)
    // staging for host batches
    int64_t cap_bytes = 0;
    uint8_t* d_seq = nullptr;
    uint8_t* d_qual = nullptr;
    int64_t cap_idx = 0;
    int64_t* d_offsets = nullptr;
    int32_t* d_lens = nullptr;
    std::vector<int32_t> h_lens;
    // tiling + measurement
    int64_t tile_bases = 0;
    // fpl_process_host: the upload runs on its own stream, piece by piece, and the kernels of a piece start as soon
    // as its bytes have arrived (copy/compute overlap inside one call)
    cudaStream_t copy_stream = nullptr;
    int* d_minmax = nullptr;            // fpl_process_device: min / max read length of the batch
    int* h_minmax = nullptr;
    std::vector<cudaEvent_t> piece_events;
    int64_t piece_bytes = 16ll << 20;
    bool timing = false;
    float kernel_ms[K_NKERNELS];
    int64_t kernel_n[K_NKERNELS];
    int64_t launches = 0;
    // multi-GPU merge (fpl_comm_init / fpl_allreduce_stats): one NCCL communicator per context
    ncclComm_t comm = nullptr;
    int comm_rank = 0, comm_size = 1;
    int64_t used_cycles = 0;            // longest read accumulated since the last fpl_reset
    long long* d_agree = nullptr;       // device word for the all-reduce(max) of the cycle count
    long long* h_agree = nullptr;       // pinned
    struct Ev { int k; cudaEvent_t a, b; };
    std::vector<Ev> events;
    std::vector<cudaEvent_t> pool;
};

static int ensure_reads(fpl_ctx* c, int64_t n) {
    if (n <= c->cap_reads) return 0;
    int64_t cap = c->cap_reads ? c->cap_reads : 1024;
    while (cap < n) cap *= 2;
    cudaFree(c->d_state); cudaFree(c->d_results); cudaFree(c->d_preseg); cudaFree(c->d_postseg);
    c->d_state = nullptr; c->d_results = nullptr; c->d_preseg = nullptr; c->d_postseg = nullptr; c->cap_reads = 0;
    CK(cudaMalloc(&c->d_state, sizeof(ReadState) * cap));
    CK(cudaMalloc(&c->d_results, sizeof(fpl_read_result) * cap));
    CK(cudaMalloc(&c->d_preseg, sizeof(StatSeg) * cap));
    CK(cudaMalloc(&c->d_postseg, sizeof(StatSeg) * 2 * cap));
    c->cap_reads = cap;
    return 0;
}

static int reserve_cycles(fpl_ctx* c, int64_t need) {
    if (need <= c->C) return 0;
    int64_t nc = c->C ? c->C : 1024;
    while (nc < need) nc *= 2;
    for (int w = 0; w < 2; w++) {
        unsigned long long* nb = nullptr;
        CK(cudaMalloc(&nb, sizeof(unsigned long long) * FPL_STATS_WORDS(nc)));
        CK(cudaMemsetAsync(nb, 0, sizeof(unsigned long long) * FPL_STATS_WORDS(nc), c->stream));
        if (c->d_stats[w]) {
            // rows b*C + c move to b*nc + c; the tail moves to 16*nc
            CK(cudaMemcpy2DAsync(nb, sizeof(unsigned long long) * nc, c->d_stats[w], sizeof(unsigned long long) * c->C,
                                 sizeof(unsigned long long) * c->C, 16, cudaMemcpyDeviceToDevice, c->stream));
            CK(cudaMemcpyAsync(nb + 16 * nc, c->d_stats[w] + 16 * c->C, sizeof(unsigned long long) * FPL_STATS_TAIL,
                               cudaMemcpyDeviceToDevice, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            cudaFree(c->d_stats[w]);
        }
        c->d_stats[w] = nb;
    }
    c->C = nc;
    return 0;
}

static cudaEvent_t get_event(fpl_ctx* c) {
    if (!c->pool.empty()) { cudaEvent_t e = c->pool.back(); c->pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

struct Timed {
    fpl_ctx* c; int k; bool ours; cudaEvent_t a = nullptr, b = nullptr;
    Timed(fpl_ctx* c_, int k_, bool ours_ = true) : c(c_), k(k_), ours(ours_) {   // ours = false: a library kernel (NCCL), timed but not counted
        if (c->timing) { a = get_event(c); b = get_event(c); cudaEventRecord(a, c->stream); }
    }
    ~Timed() {
        if (ours) c->launches++;
        if (c->timing) { cudaEventRecord(b, c->stream); c->events.push_back({k, a, b}); }
    }
};

// Harvest the event pairs that have completed; pending ones stay queued (kernel_ms accumulates until
// fpl_set_timing() resets it).
static void collect_times(fpl_ctx* c) {
    size_t keep = 0;
    for (auto& e : c->events) {
        if (cudaEventQuery(e.b) != cudaSuccess) { c->events[keep++] = e; continue; }
        float ms = 0;
        if (cudaEventElapsedTime(&ms, e.a, e.b) == cudaSuccess) { c->kernel_ms[e.k] += ms; c->kernel_n[e.k]++; }
        c->pool.push_back(e.a); c->pool.push_back(e.b);
    }
    c->events.resize(keep);
}

// min and max of the read lengths (fpl_process_device)
// ... and the OR of the low four bits of the slot offsets (out[2]): 0 <=> every read starts on a 16-byte boundary
__global__ void k_lens_minmax(const int32_t* __restrict__ lens, const int64_t* __restrict__ offsets, int64_t n, int* __restrict__ out) {
    int lo = INT_MAX, hi = INT_MIN;
    unsigned mis = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int v = lens[i];
        lo = min(lo, v); hi = max(hi, v);
        mis |= (unsigned)offsets[i] & 15u;
    }
    lo = __reduce_min_sync(0xffffffffu, lo); hi = __reduce_max_sync(0xffffffffu, hi); mis = __reduce_or_sync(0xffffffffu, mis);
    if ((threadIdx.x & 31) == 0) { atomicMin(&out[0], lo); atomicMax(&out[1], hi); if (mis) atomicOr(&out[2], (int)mis); }
}

// Runs every kernel over reads [0, n) of a device-resident batch whose lens are known on the host.
// cuts/arrived (optional): the batch arrives in pieces — reads [cuts[j], cuts[j+1]) are on the device once event
// arrived[j] has fired; the kernels then run piece by piece.
// h_lens may be null when the caller knows the longest read (known_max_len >= 0) and nothing below needs the individual
// lengths (no tiling, no pieces): a device-resident batch then never waits for the host to walk a million lengths.
static int run_batch(fpl_ctx* c, const DevBatch& full, const int32_t* h_lens, fpl_read_result* d_res_out, int64_t n_bytes,
                     const std::vector<int64_t>* cuts = nullptr, const cudaEvent_t* arrived = nullptr,
                     int64_t known_max_len = -1) {
    const int64_t n = full.n_reads;
    CK(cudaSetDevice(c->device));
    collect_times(c);
    c->emit_valid = false; c->emit.built = false; c->emit_gz_built = false;
    c->last_n = n;
    if (ensure_reads(c, n)) return -1;
    fpl_read_result* d_res = d_res_out ? d_res_out : c->d_results;
    c->last_results = d_res;
    int64_t max_len = 0;
    if (h_lens) {
        for (int64_t i = 0; i < n; i++) {
            if (h_lens[i] < 0) return fail("read %lld has a negative length", (long long)i);
            if (h_lens[i] > max_len) max_len = h_lens[i];
        }
    } else {
        max_len = known_max_len;
    }
    if (reserve_cycles(c, max_len > 0 ? max_len : 1)) return -1;
    if (max_len > c->used_cycles) c->used_cycles = max_len;
    // tiles of reads whose payload stays L2-resident across the kernels that revisit it
    const bool ext = c->P.opt.mask_enabled || c->P.opt.break_enabled;   // variable number of output reads: one tile
    c->ext.n_segs = 0; c->ext.n_regs = 0;
    int64_t r0 = 0;
    size_t piece = 0;
    while (r0 < n) {
        int64_t r1 = r0, bases = 0, tmax = 0;
        if (cuts) {
            if (ext) {       // one tile: wait for everything
                for (size_t j = 0; j + 1 < cuts->size(); j++) CK(cudaStreamWaitEvent(c->stream, arrived[j], 0));
                r1 = n;
            } else {
                CK(cudaStreamWaitEvent(c->stream, arrived[piece], 0));
                r1 = (*cuts)[piece + 1];
                piece++;
            }
            for (int64_t i = r0; i < r1; i++) if (h_lens[i] > tmax) tmax = h_lens[i];
        } else if (!h_lens || ext || c->tile_bases >= (1ll << 61)) {
            r1 = n; tmax = max_len;      // one tile
        } else {
            while (r1 < n && (r1 == r0 || ext || bases + h_lens[r1] <= c->tile_bases)) {
                bases += h_lens[r1];
                if (h_lens[r1] > tmax) tmax = h_lens[r1];
                r1++;
            }
        }
        DevBatch b = full;
        b.offsets = full.offsets + r0; b.lens = full.lens + r0; b.n_reads = r1 - r0;
        ReadState* st = c->d_state + r0;
        fpl_read_result* res = d_res + r0;
        StatSeg* pre = c->d_preseg + r0;
        StatSeg* post = c->d_postseg + 2 * r0;
        cudaStream_t s = c->stream;
        { Timed t(c, K_PRESEG); launch_make_preseg(b, pre, s); }
        { Timed t(c, K_TRIM); launch_trim(c->P, b, st, res, c->d_counters, s);
          if (c->P.opt.adapter_enabled && c->n_adapters > 2) c->launches++; }   // + k_trim_fasta
        { Timed t(c, K_CYCLE_PRE);
          if (launch_cycle_stats(&c->cycle_ws, full.seq, full.qual, pre, b.n_reads, tmax, c->d_stats[0], c->C, true,
                                 ext ? nullptr : c->d_stats[1] + 16 * c->C + FPL_STATS_KMER, c->slots16, s)) return fail("out of device memory (cycle stats workspace)");
          c->launches += 2; }   // + k_cs_keys and k_cs_gather around the (library) radix sort
        {
            Timed t(c, K_SCAN);
            if (c->jit.fn) { if (fpl_jit_launch_scan(&c->jit, b, st, s)) return fail("launching k_scan_jit failed"); }
            else if (c->plan.fast) launch_scan_fast(c->P, c->plan, b, st, s);
            else launch_scan(c->P, b, st, s);
        }
        { Timed t(c, K_FINAL); launch_final(c->P, b, st, res, post, s); }
        if (!ext) {
            { Timed t(c, K_COUNT); launch_count(res, b.n_reads, c->d_counters, true, s); }
            { Timed t(c, K_CYCLE_POST);
              if (launch_cycle_stats(&c->cycle_ws, full.seq, full.qual, post, 2 * b.n_reads, tmax, c->d_stats[1], c->C, false, nullptr, false, s))
                  return fail("out of device memory (cycle stats workspace)");
          c->launches += 2; }   // + k_cs_keys and k_cs_gather around the (library) radix sort
            { Timed t(c, K_KMER_FIX); launch_kmer_fix(b, res, c->d_stats[1] + 16 * c->C + FPL_STATS_KMER, s); }
            { Timed t(c, K_QUAL_PRE); launch_read_qual(b, c->d_stats[0], c->d_stats[1], c->C, res, false, s); }
        } else {
            // --mask / --break: k_final left the output reads of the adapter stage in the records; fpl_ext_run breaks /
            // masks / filters them (variable count) and the post-filter Stats run over its segment list
            char xerr[256] = "";
            const uint8_t* fseq = full.seq;
            { Timed t(c, K_QUAL_PRE); launch_read_qual(b, c->d_stats[0], c->d_stats[1], c->C, res, true, s); }
            { Timed t(c, K_COUNT); launch_count(res, b.n_reads, c->d_counters, false, s); }
            if (fpl_ext_run(&c->ext, c->P, b, n_bytes, res, c->d_counters, c->d_stats[1], c->C, &fseq, s, xerr, sizeof(xerr)))
                return fail("--mask/--break stage: %s", xerr);
            { Timed t(c, K_CYCLE_POST);
              if (launch_cycle_stats(&c->cycle_ws, fseq, full.qual, c->ext.d_stat, c->ext.n_segs, tmax, c->d_stats[1], c->C, true, nullptr, false, s))
                  return fail("out of device memory (cycle stats workspace)");
          c->launches += 2; }   // + k_cs_keys and k_cs_gather around the (library) radix sort
        }
        r0 = r1;
    }
    CK(cudaGetLastError());
    return 0;
}

extern "C" {

const char* fpl_last_error(void) { return g_err; }
int fpl_abi_version(void) { return FPL_ABI_VERSION; }

int fpl_create(const fpl_options* opt, const fpl_adapters* ad, fpl_ctx** out) {
    g_err[0] = 0;
    if (!opt || !ad || !out) return fail("fpl_create: null argument");
    if (opt->struct_size != (int32_t)sizeof(fpl_options))
        return fail("fpl_create: fpl_options.struct_size %d != %d (ABI mismatch)", opt->struct_size, (int)sizeof(fpl_options));
    if (opt->ed_max < 0 || opt->ed_max > 1.0) return fail("fpl_create: ed_max must be within 0..1");
    if (opt->trim_front < 0 || opt->trim_tail < 0) return fail("fpl_create: trim_front/trim_tail must be >= 0");
    if ((opt->cut_front_enabled && (opt->cut_front_window < 1 || opt->cut_front_window > FPL_MAX_WINDOW)) ||
        (opt->cut_tail_enabled && (opt->cut_tail_window < 1 || opt->cut_tail_window > FPL_MAX_WINDOW)))
        return fail("fpl_create: cut window size must be within 1..%d", FPL_MAX_WINDOW);
    const int n = 2 + (ad->n_fasta > 0 ? ad->n_fasta : 0);
    if (n > FPL_MAX_ADAPTERS) return fail("fpl_create: %d adapters exceed FPL_MAX_ADAPTERS=%d", n, FPL_MAX_ADAPTERS);
    // FPL_TIMING=1: where the start-up time goes (stderr)
    const bool tlog = getenv("FPL_TIMING") != nullptr;
    auto now = [] { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + 1e-9 * ts.tv_nsec; };
    double t_last = now();
    auto stamp = [&](const char* what) {
        if (!tlog) return;
        const double t = now();
        fprintf(stderr, "[libfplgpu] fpl_create: %-28s %7.3f s\n", what, t - t_last);
        t_last = t;
    };
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail("fpl_create: no usable CUDA device (%s); libfplgpu has no CPU fallback", cudaGetErrorString(e));
    if (opt->device < 0 || opt->device >= ndev) return fail("fpl_create: device %d out of range (%d devices)", opt->device, ndev);
    CK(cudaSetDevice(opt->device));
    CK(cudaFree(0));
    stamp("driver + device context");
    fpl_ctx* c = new fpl_ctx();
    c->device = opt->device;
    c->n_adapters = n;
    // host tables
    std::vector<uint8_t> h_ad((size_t)n * FPL_MAX_ADAPTER_LEN, 0);
    std::vector<int> h_alen(n, 0);
    std::vector<uint4> h_peq((size_t)n * 256, make_uint4(0, 0, 0, 0));
    std::vector<uint32_t> h_peq16((size_t)n * 512, 0);   // [adapter][prefix | suffix][byte]
    std::vector<uint32_t> h_acode((size_t)n * 4, 0);
    size_t maxlen = 0;
    for (int k = 0; k < n; k++) {
        const char* s = k == 0 ? ad->start : k == 1 ? ad->end : ad->fasta[k - 2];
        if (s && strlen(s) > maxlen) maxlen = strlen(s);
    }
    // adapters longer than 128 bp: multi-word match masks for myers_long (the 128-bit table below stays as it is)
    const int peq_words = maxlen > 128 ? (int)((maxlen + 63) / 64) + 1 : 0;
    std::vector<unsigned long long> h_peq_long((size_t)n * 256 * peq_words, 0ull);
    for (int k = 0; k < n; k++) {
        const char* s = k == 0 ? ad->start : k == 1 ? ad->end : ad->fasta[k - 2];
        if (!s) s = "";
        size_t len = strlen(s);
        if (len > FPL_MAX_ADAPTER_LEN) {
            delete c;
            return fail("fpl_create: adapter %d is %zu bp, longer than FPL_MAX_ADAPTER_LEN=%d", k, len, FPL_MAX_ADAPTER_LEN);
        }
        h_alen[k] = (int)len;
        memcpy(&h_ad[(size_t)k * FPL_MAX_ADAPTER_LEN], s, len);
        const int plen = (int)len < FPL_PATTERN_LEN ? (int)len : FPL_PATTERN_LEN;
        {   // packed 2-bit form for the windowed Hamming search (k_trim), only for ACGT-only adapters of <= 32 bp
            bool ok = len >= 1 && len <= 32;
            unsigned long long code = 0, mask = 0;
            for (size_t j = 0; j < len && ok; j++) {
                const char ch = s[j];
                if (ch != 'A' && ch != 'C' && ch != 'G' && ch != 'T') ok = false;
                code |= (unsigned long long)((ch >> 1) & 3) << (2 * j);
                mask |= 1ull << (2 * j);
            }
            if (ok) {
                h_acode[(size_t)k * 4 + 0] = (uint32_t)code; h_acode[(size_t)k * 4 + 1] = (uint32_t)(code >> 32);
                h_acode[(size_t)k * 4 + 2] = (uint32_t)mask; h_acode[(size_t)k * 4 + 3] = (uint32_t)(mask >> 32);
            }
        }
        for (size_t j = 0; j < len; j++) {
            uint8_t ch = (uint8_t)s[j];
            uint32_t* w = reinterpret_cast<uint32_t*>(&h_peq[(size_t)k * 256 + ch]);
            if (j < 128) w[j >> 5] |= 1u << (j & 31);
            if (peq_words) h_peq_long[((size_t)k * 256 + ch) * peq_words + (j >> 6)] |= 1ull << (j & 63);
            if ((int)j < plen) h_peq16[(size_t)k * 512 + ch] |= 1u << j;                            // first plen chars
            if ((int)j >= (int)len - plen) h_peq16[(size_t)k * 512 + 256 + ch] |= 1u << (j - (len - plen));  // last plen chars
        }
    }
    memset(&c->P, 0, sizeof(c->P));
    c->P.opt = *opt;
    c->P.one = 1u;
    {
        auto cls = [](int a) { return a <= 32 ? 0 : a <= 64 ? 1 : 2; };
        c->P.small_adapters = std::max(cls(h_alen[0]), cls(h_alen[1]));
        int fc = 0;
        for (int k = 2; k < n; k++) fc = std::max(fc, cls(h_alen[k]));
        c->P.fasta_class = fc;
    }
    c->P.n_adapters = n;
    // plan for the bit-sliced middle-adapter scan (k_scan_fast); anything it cannot express uses k_scan
    memset(&c->plan, 0, sizeof(c->plan));
    {
        bool fast = getenv("FPL_FORCE_GENERIC_SCAN") == nullptr;
        int maxa = 1;
        for (int k = 0; k < 2 && fast && opt->adapter_enabled; k++) {
            const char* s = k == 0 ? ad->start : ad->end;
            const int len = h_alen[k];
            if (len < 1 || len > 128) { fast = false; break; }   // bit-sliced counters: up to 8 planes, 4 halo words
            if (len > maxa) maxa = len;
            for (int i = 0; i < len; i++) {
                const char ch = s[i];
                if (ch != 'A' && ch != 'C' && ch != 'G' && ch != 'T') { fast = false; break; }
                c->plan.hm[k][i] = (ch & 2) ? 0xFFFFFFFFu : 0u;   // code bit HI = byte bit 1
                c->plan.lm[k][i] = (ch & 4) ? 0xFFFFFFFFu : 0u;   // code bit LO = byte bit 2
                c->plan.vm[k][i] = 0xFFFFFFFFu;
            }
        }
        c->plan.fast = fast ? 1 : 0;
        c->plan.npl = maxa <= 31 ? 5 : maxa <= 63 ? 6 : maxa <= 127 ? 7 : 8;
        c->plan.halo_words = ((maxa - 1) >> 5) + 1;
    }
    for (int i = 0; i <= FPL_MAX_ADAPTER_LEN; i++) c->P.thr[i] = (short)(int)round(opt->ed_max * i);  // src/adaptertrimmer.cpp:73
#define CKC(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { fail("%s failed: %s", #call, cudaGetErrorString(e_)); fpl_destroy(c); return -1; } } while (0)
    CKC(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CKC(cudaMalloc(&c->d_adapters, h_ad.size()));
    CKC(cudaMalloc(&c->d_alen, sizeof(int) * n));
    CKC(cudaMalloc(&c->d_peq, sizeof(uint4) * h_peq.size()));
    CKC(cudaMalloc(&c->d_peq16, sizeof(uint32_t) * h_peq16.size()));
    CKC(cudaMalloc(&c->d_acode, sizeof(uint32_t) * h_acode.size()));
    CKC(cudaMemcpy(c->d_acode, h_acode.data(), sizeof(uint32_t) * h_acode.size(), cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(c->d_adapters, h_ad.data(), h_ad.size(), cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(c->d_alen, h_alen.data(), sizeof(int) * n, cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(c->d_peq, h_peq.data(), sizeof(uint4) * h_peq.size(), cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(c->d_peq16, h_peq16.data(), sizeof(uint32_t) * h_peq16.size(), cudaMemcpyHostToDevice));
    if (peq_words) {
        CKC(cudaMalloc(&c->d_peq_long, sizeof(unsigned long long) * h_peq_long.size()));
        CKC(cudaMemcpy(c->d_peq_long, h_peq_long.data(), sizeof(unsigned long long) * h_peq_long.size(), cudaMemcpyHostToDevice));
    }
    c->P.peq_long = c->d_peq_long; c->P.peq_words = peq_words;
    if (n > 2) {
        // k_trim's many-adapter pre-filter works on 32 (adapter, side) pairs at a time and uses 64-bit bit-vectors for a
        // round as soon as one of its adapters is longer than 32 bp: group the adapters by width class
        std::vector<int> order;
        for (int cls = 0; cls < 3; cls++)
            for (int k = 2; k < n; k++) {
                const int kc = h_alen[k] <= 32 ? 0 : h_alen[k] <= 64 ? 1 : 2;
                if (kc == cls) order.push_back(k);
            }
        CKC(cudaMalloc(&c->d_pf_order, sizeof(int) * order.size()));
        CKC(cudaMemcpy(c->d_pf_order, order.data(), sizeof(int) * order.size(), cudaMemcpyHostToDevice));
    }
    c->P.pf_order = c->d_pf_order;
    c->P.adapters = c->d_adapters; c->P.alen = c->d_alen; c->P.peq = c->d_peq; c->P.peq16 = c->d_peq16; c->P.acode = c->d_acode;
    c->counter_words = FPL_COUNTER_WORDS(n);
    CKC(cudaMalloc(&c->d_counters, sizeof(unsigned long long) * c->counter_words));
    CKC(cudaMemset(c->d_counters, 0, sizeof(unsigned long long) * c->counter_words));
    stamp("tables");
    // specialise the scan kernel on the adapters (NVRTC); FPL_NO_JIT=1 keeps the precompiled k_scan_fast
    if (c->plan.fast && getenv("FPL_NO_JIT") == nullptr) {
        char jerr[512] = "";
        const bool doCounts = opt->qual_filter_enabled || opt->length_filter_enabled;
        if (fpl_jit_build_scan(c->device, ad->start ? ad->start : "", ad->end ? ad->end : "", opt->adapter_enabled != 0,
                               doCounts, opt->complexity_enabled != 0, opt->qualified_qual, &c->jit, jerr, sizeof(jerr))) {
            fprintf(stderr, "libfplgpu: run-time specialisation unavailable (%s); using the precompiled k_scan_fast\n", jerr);
            c->jit.fn = nullptr;
        }
    }
    stamp("scan kernel specialisation");
    const char* tb = getenv("FPL_TILE_MBASES");
    // 0 (default) = no tiling: every kernel streams the whole batch from HBM (measured faster than L2-sized tiles,
    // whose launches are too small to fill the GPU: profiles/README.md)
    c->tile_bases = (tb && atoll(tb) > 0) ? atoll(tb) * 1000000ll : (1ll << 62);
    // fpl_process_host uploads in pieces of this many MiB per buffer and overlaps them with the kernels (0 = one piece)
    const char* pm = getenv("FPL_PIECE_MB");
    if (pm) c->piece_bytes = atoll(pm) > 0 ? atoll(pm) << 20 : 0;
    for (int k = 0; k < K_NKERNELS; k++) { c->kernel_ms[k] = 0; c->kernel_n[k] = 0; }
    if (reserve_cycles(c, 1024)) { fpl_destroy(c); return -1; }
    CKC(cudaStreamSynchronize(c->stream));
    stamp("accumulators");
#undef CKC
    *out = c;
    return 0;
}

void fpl_destroy(fpl_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    collect_times(c);
    for (auto e : c->pool) cudaEventDestroy(e);
    cudaFree(c->d_adapters); cudaFree(c->d_alen); cudaFree(c->d_peq); cudaFree(c->d_peq16); cudaFree(c->d_acode); cudaFree(c->d_peq_long); cudaFree(c->d_pf_order);
    cudaFree(c->d_stats[0]); cudaFree(c->d_stats[1]); cudaFree(c->d_counters);
    fpl_cycle_ws_free(&c->cycle_ws);
    for (auto e : c->piece_events) cudaEventDestroy(e);
    cudaFree(c->d_minmax); if (c->h_minmax) cudaFreeHost(c->h_minmax);
    fpl_comm_destroy(c);
    cudaFree(c->d_agree); if (c->h_agree) cudaFreeHost(c->h_agree);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    cudaFree(c->d_state); cudaFree(c->d_results); cudaFree(c->d_preseg); cudaFree(c->d_postseg);
    cudaFree(c->d_seq); cudaFree(c->d_qual); cudaFree(c->d_offsets); cudaFree(c->d_lens);
    fpl_ingest_free(&c->ingest);
    fpl_ext_free(&c->ext);
    fpl_emit_free(&c->emit);
    fpl_gzip_free(&c->gz);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int fpl_process_device(fpl_ctx* c, const fpl_batch* b, fpl_read_result* results_dev) {
    g_err[0] = 0;
    if (!c || !b) return fail("fpl_process_device: null argument");
    CK(cudaSetDevice(c->device));
    const int64_t n = b->n_reads;
    if (n < 0) return fail("fpl_process_device: negative n_reads");
    DevBatch d = {b->seq, b->qual, b->offsets, b->lens, n};
    if (c->tile_bases < (1ll << 61)) {       // read tiling was asked for: the tile boundaries need every length
        c->h_lens.resize((size_t)n);
        if (n) {
            CK(cudaMemcpyAsync(c->h_lens.data(), b->lens, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
        }
        c->slots16 = false;     // offsets not inspected on this path: the per-segment alignment dispatch handles anything
        return run_batch(c, d, c->h_lens.data(), results_dev, b->n_bytes);
    }
    // only the extremes of the lengths are needed on the host (Stats capacity, grid sizes): reduce them on the side
    // stream, which does not wait for the kernels of the previous batch still running on the compute stream
    if (!c->copy_stream) CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    if (!c->d_minmax) {
        CK(cudaMalloc(&c->d_minmax, 4 * sizeof(int)));
        CK(cudaMallocHost(&c->h_minmax, 4 * sizeof(int)));
    }
    c->h_minmax[0] = 0; c->h_minmax[1] = 0; c->h_minmax[2] = 0;
    if (n) {
        const int init[3] = {INT_MAX, INT_MIN, 0};
        CK(cudaMemcpyAsync(c->d_minmax, init, sizeof(init), cudaMemcpyHostToDevice, c->copy_stream));
        const unsigned blocks = (unsigned)((n + 1023) / 1024 < 1184 ? (n + 1023) / 1024 : 1184);
        k_lens_minmax<<<blocks, 256, 0, c->copy_stream>>>(b->lens, b->offsets, n, c->d_minmax);
        CK(cudaMemcpyAsync(c->h_minmax, c->d_minmax, 3 * sizeof(int), cudaMemcpyDeviceToHost, c->copy_stream));
        CK(cudaStreamSynchronize(c->copy_stream));
        if (c->h_minmax[0] < 0) return fail("fpl_process_device: a read has a negative length");
    }
    c->slots16 = c->h_minmax[2] == 0;
    return run_batch(c, d, nullptr, results_dev, b->n_bytes, nullptr, nullptr, n ? c->h_minmax[1] : 0);
}

void* fpl_stream(fpl_ctx* c) { return c ? (void*)c->stream : nullptr; }

int fpl_sync(fpl_ctx* c) {
    if (!c) return fail("fpl_sync: null context");
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->stream));
    collect_times(c);
    return 0;
}

int fpl_process_host(fpl_ctx* c, const fpl_batch* b, fpl_read_result* results) {
    g_err[0] = 0;
    if (!c || !b) return fail("fpl_process_host: null argument");
    CK(cudaSetDevice(c->device));
    const int64_t n = b->n_reads;
    if (n < 0 || b->n_bytes < 0) return fail("fpl_process_host: negative size");
    if (n > 0 && !results) return fail("fpl_process_host: results is null");
    // validate the slot layout on the host (cheap, O(reads))
    bool monotonic = true;
    for (int64_t i = 0; i < n; i++) {
        const int64_t o = b->offsets[i];
        if (i > 0 && o < b->offsets[i - 1] + b->lens[i - 1]) monotonic = false;
        if (o < 0 || (o & 15) || b->lens[i] < 0 || o + b->lens[i] > b->n_bytes)
            return fail("fpl_process_host: read %lld has a bad slot (offset %lld, len %d, n_bytes %lld; offsets must be multiples of 16)",
                        (long long)i, (long long)o, b->lens[i], (long long)b->n_bytes);
    }
    const int64_t need = b->n_bytes + 64;  // tail pad for whole-word over-reads
    if (need > c->cap_bytes) {
        cudaFree(c->d_seq); cudaFree(c->d_qual); c->d_seq = c->d_qual = nullptr; c->cap_bytes = 0;
        CK(cudaMalloc(&c->d_seq, need));
        CK(cudaMalloc(&c->d_qual, need));
        c->cap_bytes = need;
    }
    if (n > c->cap_idx) {
        cudaFree(c->d_offsets); cudaFree(c->d_lens); c->d_offsets = nullptr; c->d_lens = nullptr; c->cap_idx = 0;
        CK(cudaMalloc(&c->d_offsets, sizeof(int64_t) * n));
        CK(cudaMalloc(&c->d_lens, sizeof(int32_t) * n));
        c->cap_idx = n;
    }
    // pieces of about piece_bytes, cut at read boundaries (slots in increasing order; otherwise one piece)
    std::vector<int64_t> cuts(1, 0);
    if (monotonic && c->piece_bytes > 0) {
        int64_t start = 0;
        for (int64_t i = 1; i < n; i++)
            if (b->offsets[i] - start >= c->piece_bytes) { cuts.push_back(i); start = b->offsets[i]; }
    }
    cuts.push_back(n);
    const size_t np = cuts.size() - 1;
    if (!c->copy_stream) CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    while (c->piece_events.size() < np) {
        cudaEvent_t e;
        CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c->piece_events.push_back(e);
    }
    // every call ends with a synchronize of the compute stream, so the device buffers are free to overwrite here
    cudaStream_t cs = c->copy_stream;
    if (n) {
        CK(cudaMemcpyAsync(c->d_offsets, b->offsets, sizeof(int64_t) * n, cudaMemcpyHostToDevice, cs));
        CK(cudaMemcpyAsync(c->d_lens, b->lens, sizeof(int32_t) * n, cudaMemcpyHostToDevice, cs));
    }
    for (size_t j = 0; j < np; j++) {
        const int64_t lo = j == 0 ? 0 : b->offsets[cuts[j]];
        const int64_t hi = j + 1 == np ? b->n_bytes : b->offsets[cuts[j + 1]];
        if (hi > lo) {
            CK(cudaMemcpyAsync(c->d_seq + lo, b->seq + lo, hi - lo, cudaMemcpyHostToDevice, cs));
            CK(cudaMemcpyAsync(c->d_qual + lo, b->qual + lo, hi - lo, cudaMemcpyHostToDevice, cs));
        }
        if (j + 1 == np) {
            CK(cudaMemsetAsync(c->d_seq + b->n_bytes, 0, 64, cs));
            CK(cudaMemsetAsync(c->d_qual + b->n_bytes, 0, 64, cs));
        }
        CK(cudaEventRecord(c->piece_events[j], cs));
    }
    DevBatch d = {c->d_seq, c->d_qual, c->d_offsets, c->d_lens, n};
    c->slots16 = true;          // checked above: every offset is a multiple of 16
    if (run_batch(c, d, b->lens, nullptr, b->n_bytes, &cuts, c->piece_events.data())) return -1;
    if (n) CK(cudaMemcpyAsync(results, c->d_results, sizeof(fpl_read_result) * n, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    collect_times(c);
    return 0;
}

int fpl_process_fastq_host(fpl_ctx* c, const uint8_t* text, int64_t n_bytes, int is_last, fpl_fastq_record* records,
                           fpl_read_result* results, int64_t max_records, int64_t* n_records, int64_t* consumed) {
    g_err[0] = 0;
    if (!c || !n_records || !consumed || (n_bytes > 0 && !text)) return fail("fpl_process_fastq_host: null argument");
    if (n_bytes < 0 || n_bytes >= (1ll << 40)) return fail("fpl_process_fastq_host: bad chunk size");
    CK(cudaSetDevice(c->device));
    char err[256] = "";
    int64_t nrec = 0;
    int rc = fpl_ingest_index(&c->ingest, text, n_bytes, is_last, c->stream, &nrec, consumed, err, sizeof(err));
    if (rc < 0) return fail("fpl_process_fastq_host: %s", err);
    if (rc > 0) return 1;
    *n_records = nrec;
    c->emit_valid = false; c->emit.built = false; c->emit_gz_built = false;
    if (nrec == 0) { c->emit_valid = true; c->emit_n = 0; return 0; }
    if (nrec > max_records) return 1;
    if (!records || !results) return fail("fpl_process_fastq_host: records/results is null");
    FplIngest& g = c->ingest;
    const int64_t need = g.packed_bytes + 64;
    if (need > c->cap_bytes) {
        cudaFree(c->d_seq); cudaFree(c->d_qual); c->d_seq = c->d_qual = nullptr; c->cap_bytes = 0;
        CK(cudaMalloc(&c->d_seq, need));
        CK(cudaMalloc(&c->d_qual, need));
        c->cap_bytes = need;
    }
    // slot padding is never interpreted, but keep it defined for whole-vector reads past a read's end
    CK(cudaMemsetAsync(c->d_seq, 0, need, c->stream));
    CK(cudaMemsetAsync(c->d_qual, 0, need, c->stream));
    if (fpl_ingest_pack(&g, nrec, c->d_seq, c->d_qual, c->stream, err, sizeof(err))) return fail("fpl_process_fastq_host: %s", err);
    c->h_lens.resize((size_t)nrec);
    CK(cudaMemcpyAsync(c->h_lens.data(), g.d_lens, sizeof(int32_t) * nrec, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(records, g.d_rec, sizeof(fpl_fastq_record) * nrec, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    DevBatch d = {c->d_seq, c->d_qual, g.d_offsets, g.d_lens, nrec};
    c->slots16 = false;         // the device packer's slots are aligned, but nothing here depends on it
    if (run_batch(c, d, c->h_lens.data(), nullptr, g.packed_bytes)) return -1;
    CK(cudaMemcpyAsync(results, c->d_results, sizeof(fpl_read_result) * nrec, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    collect_times(c);
    c->emit_valid = true; c->emit_n = nrec;
    return 0;
}

// Builds the emit text of the last chunk on the device unless it is built already (for the same want_failed).
static int ensure_emit(fpl_ctx* c, int want_failed, const char* fn) {
    if (!c->emit_valid)
        return fail("%s: the last call on this context was not a successful fpl_process_fastq_host", fn);
    CK(cudaSetDevice(c->device));
    FplEmit& e = c->emit;
    if (!e.built || e.with_failed != (want_failed != 0)) {
        const bool ext = c->P.opt.mask_enabled || c->P.opt.break_enabled;
        EmitSource src;
        src.text = c->ingest.d_text; src.rec = c->ingest.d_rec; src.res = c->last_results; src.n_reads = c->emit_n;
        src.segs = ext ? c->ext.d_segs : nullptr;
        src.seg_off = ext ? c->ext.d_off : nullptr;
        src.mseq = (c->P.opt.mask_enabled && c->ext.n_segs > 0) ? c->ext.d_mseq : nullptr;   // fpl_ext_run made the masked copy
        src.offsets = c->ingest.d_offsets;
        char err[256] = "";
        c->emit_gz_built = false;
        if (fpl_emit_build(&e, src, want_failed != 0, c->stream, err, sizeof(err))) return fail("%s: %s", fn, err);
        if (c->emit_n) c->launches += 2;
    }
    return 0;
}

int fpl_emit_fastq_host(fpl_ctx* c, int want_failed, uint8_t* out, int64_t out_cap, int64_t* out_bytes, uint8_t* failed,
                        int64_t failed_cap, int64_t* failed_bytes) {
    g_err[0] = 0;
    if (!c || !out_bytes || !failed_bytes) return fail("fpl_emit_fastq_host: null argument");
    *out_bytes = *failed_bytes = 0;
    if (ensure_emit(c, want_failed, "fpl_emit_fastq_host")) return -1;
    FplEmit& e = c->emit;
    *out_bytes = e.out_bytes;
    *failed_bytes = e.failed_bytes;
    if (e.out_bytes > out_cap || e.failed_bytes > failed_cap) return 1;     // the text stays built: call again with room
    if ((e.out_bytes && !out) || (e.failed_bytes && !failed)) return fail("fpl_emit_fastq_host: null output buffer");
    if (e.out_bytes) CK(cudaMemcpyAsync(out, e.d_out, (size_t)e.out_bytes, cudaMemcpyDeviceToHost, c->stream));
    if (e.failed_bytes) CK(cudaMemcpyAsync(failed, e.d_failed, (size_t)e.failed_bytes, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

// Compresses device-resident pieces into c->gz.d_out (back to back); piece_out[i] = compressed bytes of piece i.
static int gzip_pieces(fpl_ctx* c, const uint8_t* const* piece, const int64_t* bytes, int n_pieces, int64_t* piece_out,
                       const char* fn) {
    char err[256] = "";
    collect_times(c);
    if (fpl_gzip_plan(&c->gz, piece, bytes, n_pieces, c->stream, err, sizeof(err))) return fail("%s: %s", fn, err);
    if (c->gz.n_segs) {
        { Timed t(c, K_GZ_DEFLATE); fpl_gzip_deflate(&c->gz, c->stream); }
        CK(cudaGetLastError());
        if (fpl_gzip_offsets(&c->gz, c->stream, err, sizeof(err))) return fail("%s: %s", fn, err);
        { Timed t(c, K_GZ_COMPACT); fpl_gzip_compact(&c->gz, c->stream); }
        CK(cudaGetLastError());
    }
    if (fpl_gzip_piece_sizes(&c->gz, piece_out, c->stream, err, sizeof(err))) return fail("%s: %s", fn, err);
    collect_times(c);
    return 0;
}

int fpl_gzip_host(fpl_ctx* c, const uint8_t* text, const int64_t* piece_bytes, int32_t n_pieces, uint8_t* out, int64_t out_cap,
                  int64_t* out_piece_bytes) {
    g_err[0] = 0;
    if (!c || n_pieces < 0 || (n_pieces > 0 && (!piece_bytes || !out_piece_bytes))) return fail("fpl_gzip_host: bad argument");
    int64_t total = 0;
    for (int i = 0; i < n_pieces; i++) {
        if (piece_bytes[i] < 0) return fail("fpl_gzip_host: piece %d has a negative size", i);
        total += piece_bytes[i];
    }
    if ((total && !text) || out_cap < FPL_GZIP_BOUND(total, n_pieces) || (FPL_GZIP_BOUND(total, n_pieces) > 0 && !out))
        return fail("fpl_gzip_host: the output buffer holds %lld bytes, FPL_GZIP_BOUND(%lld, %d) = %lld", (long long)out_cap,
                    (long long)total, n_pieces, (long long)FPL_GZIP_BOUND(total, n_pieces));
    CK(cudaSetDevice(c->device));
    c->emit_gz_built = false;                           // gz.d_out is about to be overwritten
    char err[256] = "";
    if (fpl_gzip_grow((void**)&c->gz.d_in, &c->gz.cap_in, total + 16, err, sizeof(err))) return fail("fpl_gzip_host: %s", err);
    if (total) CK(cudaMemcpyAsync(c->gz.d_in, text, (size_t)total, cudaMemcpyHostToDevice, c->stream));
    std::vector<const uint8_t*> ptr((size_t)n_pieces);
    for (int64_t i = 0, o = 0; i < n_pieces; o += piece_bytes[i], i++) ptr[(size_t)i] = c->gz.d_in + o;
    if (gzip_pieces(c, ptr.data(), piece_bytes, n_pieces, out_piece_bytes, "fpl_gzip_host")) return -1;
    int64_t n_out = 0;
    for (int i = 0; i < n_pieces; i++) n_out += out_piece_bytes[i];
    if (n_out) CK(cudaMemcpyAsync(out, c->gz.d_out, (size_t)n_out, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int fpl_emit_fastq_gzip_host(fpl_ctx* c, int want_failed, uint8_t* out, int64_t out_cap, int64_t* out_bytes, uint8_t* failed,
                             int64_t failed_cap, int64_t* failed_bytes) {
    g_err[0] = 0;
    if (!c || !out_bytes || !failed_bytes) return fail("fpl_emit_fastq_gzip_host: null argument");
    *out_bytes = *failed_bytes = 0;
    if (ensure_emit(c, want_failed, "fpl_emit_fastq_gzip_host")) return -1;
    FplEmit& e = c->emit;
    if (!c->emit_gz_built || c->emit_gz_failed != (want_failed != 0)) {
        const uint8_t* piece[2] = {e.d_out, e.d_failed};
        const int64_t bytes[2] = {e.out_bytes, e.failed_bytes};
        if (gzip_pieces(c, piece, bytes, 2, c->emit_gz_bytes, "fpl_emit_fastq_gzip_host")) return -1;
        c->emit_gz_built = true;
        c->emit_gz_failed = want_failed != 0;
    }
    *out_bytes = c->emit_gz_bytes[0];
    *failed_bytes = c->emit_gz_bytes[1];
    if (*out_bytes > out_cap || *failed_bytes > failed_cap) return 1;      // stays compressed on the device: call again with room
    if ((*out_bytes && !out) || (*failed_bytes && !failed)) return fail("fpl_emit_fastq_gzip_host: null output buffer");
    if (*out_bytes) CK(cudaMemcpyAsync(out, c->gz.d_out, (size_t)*out_bytes, cudaMemcpyDeviceToHost, c->stream));
    if (*failed_bytes)
        CK(cudaMemcpyAsync(failed, c->gz.d_out + *out_bytes, (size_t)*failed_bytes, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int fpl_last_segments(fpl_ctx* c, fpl_segment* out, int64_t cap, int64_t* n) {
    if (!c || !n) return fail("fpl_last_segments: null argument");
    *n = c->ext.n_segs;
    if (*n == 0) return 0;
    if (!out || cap < *n) return fail("fpl_last_segments: %lld entries, capacity %lld", (long long)*n, (long long)cap);
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpyAsync(out, c->ext.d_segs, sizeof(fpl_segment) * *n, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int fpl_last_mask_regions(fpl_ctx* c, fpl_region* out, int64_t cap, int64_t* n) {
    if (!c || !n) return fail("fpl_last_mask_regions: null argument");
    *n = c->ext.n_regs;
    if (*n == 0) return 0;
    if (!out || cap < *n) return fail("fpl_last_mask_regions: %lld entries, capacity %lld", (long long)*n, (long long)cap);
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpyAsync(out, c->ext.d_regs, sizeof(fpl_region) * *n, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int fpl_fetch_results(fpl_ctx* c, fpl_read_result* results, int64_t n) {
    if (!c || !results) return fail("fpl_fetch_results: null argument");
    if (n > c->last_n) return fail("fpl_fetch_results: only %lld records available", (long long)c->last_n);
    CK(cudaSetDevice(c->device));
    if (n) CK(cudaMemcpyAsync(results, c->last_results, sizeof(fpl_read_result) * n, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    collect_times(c);
    return 0;
}

int64_t fpl_stats_cycles(fpl_ctx* c) { return c ? c->C : 0; }

int fpl_stats_reserve(fpl_ctx* c, int64_t cycles) {
    if (!c) return fail("fpl_stats_reserve: null context");
    CK(cudaSetDevice(c->device));
    if (reserve_cycles(c, cycles)) return -1;
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int fpl_stats_download(fpl_ctx* c, int which, int64_t* out, int64_t n_words) {
    if (!c || !out || which < 0 || which > 1) return fail("fpl_stats_download: bad argument");
    if (n_words != FPL_STATS_WORDS(c->C)) return fail("fpl_stats_download: n_words %lld != FPL_STATS_WORDS(%lld)", (long long)n_words, (long long)c->C);
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpyAsync(out, c->d_stats[which], sizeof(int64_t) * n_words, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int fpl_stats_device_ptr(fpl_ctx* c, int which, void** dptr, int64_t* n_words) {
    if (!c || !dptr || !n_words || which < 0 || which > 1) return fail("fpl_stats_device_ptr: bad argument");
    *dptr = c->d_stats[which];
    *n_words = FPL_STATS_WORDS(c->C);
    return 0;
}

int64_t fpl_counter_words(fpl_ctx* c) { return c ? c->counter_words : 0; }

int fpl_counters_download(fpl_ctx* c, int64_t* out, int64_t n_words) {
    if (!c || !out) return fail("fpl_counters_download: bad argument");
    if (n_words != c->counter_words) return fail("fpl_counters_download: n_words %lld != %lld", (long long)n_words, (long long)c->counter_words);
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpyAsync(out, c->d_counters, sizeof(int64_t) * n_words, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int fpl_counters_device_ptr(fpl_ctx* c, void** dptr, int64_t* n_words) {
    if (!c || !dptr || !n_words) return fail("fpl_counters_device_ptr: bad argument");
    *dptr = c->d_counters;
    *n_words = c->counter_words;
    return 0;
}

int fpl_reset(fpl_ctx* c) {
    if (!c) return fail("fpl_reset: null context");
    CK(cudaSetDevice(c->device));
    for (int w = 0; w < 2; w++)
        CK(cudaMemsetAsync(c->d_stats[w], 0, sizeof(unsigned long long) * FPL_STATS_WORDS(c->C), c->stream));
    CK(cudaMemsetAsync(c->d_counters, 0, sizeof(unsigned long long) * c->counter_words, c->stream));
    c->used_cycles = 0;
    return 0;
}

int fpl_last_kernel_times(fpl_ctx* c, const char** names, float* ms, int64_t* launches, int cap) {
    if (!c) return 0;
    collect_times(c);
    for (int k = 0; k < K_NKERNELS && k < cap; k++) {
        if (names) names[k] = kKernelNames[k];
        if (ms) ms[k] = c->kernel_ms[k];
        if (launches) launches[k] = c->kernel_n[k];
    }
    return K_NKERNELS;
}

int64_t fpl_launch_count(fpl_ctx* c) { return c ? c->launches : 0; }

int fpl_set_timing(fpl_ctx* c, int enabled) {
    if (!c) return fail("fpl_set_timing: null context");
    c->timing = enabled != 0;
    collect_times(c);
    for (int k = 0; k < K_NKERNELS; k++) { c->kernel_ms[k] = 0; c->kernel_n[k] = 0; }
    return 0;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------------------------
// Multi-GPU merge: the replacement of Stats::merge (src/stats.cpp:1013-1082) and FilterResult::merge
// (src/filterresult.cpp:28-61) for one process per GPU.  NCCL is resolved at run time (dlopen of libnccl.so.2: inside
// a torch process that is the copy torch already loaded), so the library stays loadable without it; the collectives
// run on the context's own stream, after the kernels that fill the blocks, with no host synchronisation.
// ------------------------------------------------------------------------------------------------------------------
namespace {
struct Nccl {
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
    Nccl() {
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return;
        GetUniqueId = (decltype(GetUniqueId))dlsym(h, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(h, "ncclCommInitRank");
        CommDestroy = (decltype(CommDestroy))dlsym(h, "ncclCommDestroy");
        AllReduce = (decltype(AllReduce))dlsym(h, "ncclAllReduce");
        GroupStart = (decltype(GroupStart))dlsym(h, "ncclGroupStart");
        GroupEnd = (decltype(GroupEnd))dlsym(h, "ncclGroupEnd");
        GetErrorString = (decltype(GetErrorString))dlsym(h, "ncclGetErrorString");
        ok = GetUniqueId && CommInitRank && CommDestroy && AllReduce && GroupStart && GroupEnd && GetErrorString;
    }
};
Nccl& nccl() { static Nccl n; return n; }
}  // namespace

#define CKN(call)                                                                                        \
    do {                                                                                                 \
        ncclResult_t r_ = (call);                                                                        \
        if (r_ != ncclSuccess) return fail("%s failed: %s", #call, nccl().GetErrorString(r_));          \
    } while (0)

static_assert(sizeof(ncclUniqueId) == FPL_COMM_ID_BYTES, "FPL_COMM_ID_BYTES must be sizeof(ncclUniqueId)");

extern "C" {

int fpl_comm_unique_id(uint8_t* id) {
    g_err[0] = 0;
    if (!id) return fail("fpl_comm_unique_id: null argument");
    if (!nccl().ok) return fail("fpl_comm_unique_id: libnccl.so.2 is not loadable");
    ncclUniqueId u;
    CKN(nccl().GetUniqueId(&u));
    memcpy(id, &u, sizeof(u));
    return 0;
}

int fpl_comm_init(fpl_ctx* c, const uint8_t* id, int rank, int n_ranks) {
    g_err[0] = 0;
    if (!c || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail("fpl_comm_init: bad argument");
    if (!nccl().ok) return fail("fpl_comm_init: libnccl.so.2 is not loadable");
    if (c->comm) return fail("fpl_comm_init: the context already has a communicator");
    CK(cudaSetDevice(c->device));
    ncclUniqueId u;
    memcpy(&u, id, sizeof(u));
    CKN(nccl().CommInitRank(&c->comm, n_ranks, u, rank));
    c->comm_rank = rank; c->comm_size = n_ranks;
    if (!c->d_agree) {
        CK(cudaMalloc(&c->d_agree, sizeof(long long)));
        CK(cudaMallocHost(&c->h_agree, sizeof(long long)));
    }
    return 0;
}

int fpl_comm_destroy(fpl_ctx* c) {
    if (!c || !c->comm) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    nccl().CommDestroy(c->comm);
    c->comm = nullptr; c->comm_size = 1; c->comm_rank = 0;
    return 0;
}

int fpl_comm_size(fpl_ctx* c) { return c ? c->comm_size : 0; }

int fpl_comm_agree_cycles(fpl_ctx* c, int64_t* cycles) {
    g_err[0] = 0;
    if (!c || !c->comm) return fail("fpl_comm_agree_cycles: no communicator (fpl_comm_init first)");
    CK(cudaSetDevice(c->device));
    *c->h_agree = (long long)c->used_cycles;
    CK(cudaMemcpyAsync(c->d_agree, c->h_agree, sizeof(long long), cudaMemcpyHostToDevice, c->stream));
    CKN(nccl().AllReduce(c->d_agree, c->d_agree, 1, ncclInt64, ncclMax, c->comm, c->stream));
    CK(cudaMemcpyAsync(c->h_agree, c->d_agree, sizeof(long long), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    const int64_t agreed = (int64_t)*c->h_agree;
    if (reserve_cycles(c, agreed > 0 ? agreed : 1)) return -1;      // every rank now holds at least `agreed` columns
    CK(cudaStreamSynchronize(c->stream));
    if (cycles) *cycles = agreed;
    return 0;
}

int fpl_allreduce_stats(fpl_ctx* c, int64_t cycles) {
    g_err[0] = 0;
    if (!c || !c->comm) return fail("fpl_allreduce_stats: no communicator (fpl_comm_init first)");
    CK(cudaSetDevice(c->device));
    if (cycles <= 0 && fpl_comm_agree_cycles(c, &cycles)) return -1;
    if (cycles > c->C) return fail("fpl_allreduce_stats: %lld cycles exceed this rank's capacity %lld (fpl_stats_reserve first)",
                                   (long long)cycles, (long long)c->C);
    if (cycles < c->used_cycles) return fail("fpl_allreduce_stats: %lld cycles do not cover this rank's longest read (%lld)",
                                             (long long)cycles, (long long)c->used_cycles);
    // rows [b*C, b*C + cycles) of the 16 per-cycle arrays, then the tail; the row pointers depend on this rank's C, the
    // counts do not, so ranks need not share a capacity.  One group = one fused launch.
    Timed t(c, K_ALLREDUCE, false);
    CKN(nccl().GroupStart());
    for (int w = 0; w < 2; w++) {
        unsigned long long* blk = c->d_stats[w];
        if (cycles > 0)
            for (int b = 0; b < 16; b++)
                CKN(nccl().AllReduce(blk + (int64_t)b * c->C, blk + (int64_t)b * c->C, (size_t)cycles, ncclInt64, ncclSum, c->comm, c->stream));
        CKN(nccl().AllReduce(blk + 16 * c->C, blk + 16 * c->C, FPL_STATS_TAIL, ncclInt64, ncclSum, c->comm, c->stream));
    }
    CKN(nccl().AllReduce(c->d_counters, c->d_counters, (size_t)c->counter_words, ncclInt64, ncclSum, c->comm, c->stream));
    CKN(nccl().GroupEnd());
    return 0;
}

}  // extern "C"
