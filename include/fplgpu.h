/*
 * fplgpu.h — C ABI of libfplgpu.so: the per-read hot loop of fastplong
 * (SingleEndProcessor::processSingleEnd, reference src/seprocessor.cpp:180-329) as sm_100a CUDA kernels.
 *
 * The reference has no FFI for this path; the seam is the C++ class SingleEndProcessor
 * (src/seprocessor.h:23-50).  A host that implements that class (fastplong_b200/host/seprocessor_gpu.cpp)
 * or any other binding (ctypes: fastplong_b200/binding.py) talks to the kernels through exactly the
 * entry points below: plain pointers and sizes, no C++ or torch types, int status (0 = ok), message via
 * fpl_last_error().  All buffers are caller-owned.  A context is bound to one CUDA device and one stream;
 * calls on one context must be serialised by the caller, distinct contexts are independent
 * (the reference's worker threads each own a ThreadConfig the same way, src/threadconfig.cpp:4-17).
 *
 * Every entry point names the reference interface it replaces.
 */
#ifndef FPLGPU_H
#define FPLGPU_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FPL_ABI_VERSION 6

/* Filter result codes — identical to src/common.h:43-50 (they index FilterResult::mFilterReadStats[32]). */
enum {
    FPL_PASS_FILTER = 0,
    FPL_FAIL_POLY_X = 4,
    FPL_FAIL_OVERLAP = 8,
    FPL_FAIL_N_BASE = 12,
    FPL_FAIL_LENGTH = 16,
    FPL_FAIL_TOO_LONG = 17,
    FPL_FAIL_QUALITY = 20,
    FPL_FAIL_COMPLEXITY = 24,
    FPL_FILTER_RESULT_TYPES = 32
};

/* Limits of this implementation (the reference has none; exceeding them is a loud error, not a fallback). */
#define FPL_MAX_ADAPTER_LEN 1024 /* longest adapter (start/end/FASTA entry) accepted by fpl_create; adapters of up to
                                    128 bp take the register-resident bit-vector paths, longer ones a multi-word one */
#define FPL_MAX_ADAPTERS 1024    /* start + end + FASTA entries */
#define FPL_MAX_WINDOW 1000      /* cut_front/cut_tail window size, reference range 1..1000 (src/options.cpp) */
#define FPL_INLINE_EVENTS 4

/*
 * Flat POD copy of the Options fields the hot loop reads (src/options.h:20-268, filled at src/main.cpp:115-250).
 * Booleans are int32 0/1.
 */
typedef struct fpl_options {
    int32_t struct_size;              /* = sizeof(fpl_options), ABI check */
    int32_t device;                   /* CUDA device ordinal */
    /* Filter::trimAndCut — TrimmingOptions, QualityCutOptions (src/filter.cpp:130-232) */
    int32_t trim_front;               /* opt.trim.front */
    int32_t trim_tail;                /* opt.trim.tail */
    int32_t cut_front_enabled;        /* opt.qualityCut.enabledFront */
    int32_t cut_front_window;         /* windowSizeFront */
    int32_t cut_front_quality;        /* qualityFront (phred, not char) */
    int32_t cut_tail_enabled;
    int32_t cut_tail_window;
    int32_t cut_tail_quality;
    /* PolyX::trimPolyX (src/polyx.cpp:11-78) */
    int32_t polyx_enabled;            /* opt.polyXTrim.enabled */
    int32_t polyx_min_len;            /* opt.polyXTrim.minLen */
    /* AdapterTrimmer (src/adaptertrimmer.cpp) */
    int32_t adapter_enabled;          /* opt.adapter.enabled */
    int32_t trimming_extension;       /* opt.adapter.trimmingExtension */
    double ed_max;                    /* opt.adapter.edMax; thr(n) = (int)round(ed_max*n) is tabulated on the host */
    /* Filter::passFilter (src/filter.cpp:12-65) */
    int32_t qual_filter_enabled;      /* opt.qualfilter.enabled */
    int32_t qualified_qual;           /* opt.qualfilter.qualifiedQual: the phred+33 CHAR value */
    int32_t unqualified_percent_limit;
    int32_t avg_qual_req;
    int32_t n_base_percent_limit;
    int32_t n_base_limit;             /* 1000000 means "off" (src/filter.cpp:48) */
    int32_t length_filter_enabled;    /* opt.lengthFilter.enabled */
    int32_t length_required;
    int32_t length_max;               /* 0 = no limit */
    int32_t complexity_enabled;       /* opt.complexityFilter.enabled */
    int32_t complexity_threshold_pct; /* opt.complexityFilter.threshold * 100 (src/main.cpp:205) */
    /* --mask / --break: Filter::detectLowQualityRegions + Read::maskRegionWithN / breakByRegions
       (src/seprocessor.cpp:235-262, src/filter.cpp:83-128, src/read.cpp:217-262) */
    int32_t mask_enabled;             /* opt.mask.enabled */
    int32_t mask_window;              /* opt.mask.windowSize */
    int32_t mask_quality;             /* opt.mask.quality (phred) */
    int32_t break_enabled;            /* opt.breakOpt.enabled */
    int32_t break_window;
    int32_t break_quality;
    int32_t reserved[3];
} fpl_options;

/*
 * The adapter strings the kernels receive, in the order the reference applies them:
 * index 0 = opt.adapter.sequenceStart, 1 = opt.adapter.sequenceEnd (either may be empty, or the literal
 * "auto" when detection failed — SURVEY A.10/1), 2.. = opt.adapter.seqsInFasta in std::map header order
 * (src/options.cpp:50-59).  n_fasta == 0 <=> !opt.adapter.hasFasta.
 */
typedef struct fpl_adapters {
    const char* start;                /* NUL-terminated */
    const char* end;                  /* NUL-terminated */
    int32_t n_fasta;
    const char* const* fasta;         /* n_fasta NUL-terminated strings */
} fpl_adapters;

/*
 * A packed batch of reads: sequence bytes and quality bytes in two buffers with identical layout;
 * read i occupies [offsets[i], offsets[i]+lens[i]) in both.  Offsets must be multiples of 16 and the
 * buffers 16-byte aligned (vector loads / TMA bulk copies); bytes between slots are ignored.
 * Replaces ReadPack{Read** data; int count} (src/read.h:63-66) — many 16-read packs per submission.
 */
typedef struct fpl_batch {
    const uint8_t* seq;
    const uint8_t* qual;
    const int64_t* offsets;
    const int32_t* lens;
    int64_t n_reads;
    int64_t n_bytes;                  /* size of seq (== size of qual) in bytes, including slot padding */
} fpl_batch;

/*
 * Adapter trim event (FilterResult::addAdapterTrimmed argument, src/adaptertrimmer.cpp:189,226,260,295),
 * packed: bits 0..15 adapter index (fpl_adapters order), bit 16 side (0 = trimBySequenceStart,
 * 1 = trimBySequenceEnd), bits 17..31 cmplen.  The counted string is
 *   side 0: adapter.substr(alen - cmplen, cmplen)      side 1: adapter.substr(0, cmplen)
 * (cmplen == alen for a full-adapter hit).
 */
#define FPL_EVENT(idx, side, cmplen) ((uint32_t)(idx) | ((uint32_t)(side) << 16) | ((uint32_t)(cmplen) << 17))
#define FPL_EVENT_ADAPTER(e) ((int)((e) & 0xFFFFu))
#define FPL_EVENT_SIDE(e) ((int)(((e) >> 16) & 1u))
#define FPL_EVENT_CMPLEN(e) ((int)((e) >> 17))

/* fpl_read_result.flags */
#define FPL_FLAG_DROPPED_BY_CUT 1u   /* Filter::trimAndCut returned NULL: no filter record, no output (SURVEY A.2) */
#define FPL_FLAG_POLYX 2u            /* PolyX::trimPolyX fired */
#define FPL_FLAG_MIDDLE_ADAPTER 4u   /* AdapterTrimmer::findMiddleAdapters returned true -> Read::breakByGap */
#define FPL_FLAG_SEG0_IS_RIGHT 8u    /* the only segment is the "split-by-adapter-right-" one (left was empty) */

/*
 * Everything processSingleEnd decides about one input read (64 bytes).  All windows are [lo, lo+len) on the
 * ORIGINAL read's bytes (trimming only erases a prefix / resizes, src/read.cpp:62-73).
 */
typedef struct fpl_read_result {
    uint32_t flags;
    int32_t n_segments;               /* outReads.size(): 0, 1 or 2 (src/seprocessor.cpp:222-232) */
    int32_t trim_lo, trim_len;        /* r1 after trimAndCut/polyX/adapter trims (what --failed_out prints, :278-280) */
    int32_t seg_lo[2], seg_len[2];    /* outReads windows; with one segment after a split see FPL_FLAG_SEG0_IS_RIGHT */
    uint8_t seg_result[2];            /* Filter::passFilter code per segment (src/filter.cpp:12-65) */
    uint8_t seg_median_qual[2];       /* Stats::statRead median char of a PASSING segment (src/stats.cpp:351-361), else 0 */
    uint8_t pre_median_qual;          /* median char of the input read (pre-filter Stats); 0 for an empty read */
    uint8_t polyx_base;               /* index into ATCG_BASES (src/common.h:29) when FPL_FLAG_POLYX */
    uint16_t n_events;                /* adapter trim events of this read (all of them are in the count table) */
    int32_t polyx_len;                /* FilterResult::addPolyXTrimmed length */
    int32_t adapter_trimmed_bases;    /* 'trimmed' at src/seprocessor.cpp:206-216; >0 => addReadTrimmed(trimmed) */
    uint32_t events[FPL_INLINE_EVENTS]; /* first FPL_INLINE_EVENTS events in application order */
} fpl_read_result;

/*
 * With --break a read can end up in any number of output reads, and with --mask their bases change: in those modes
 * (only) the full list of output reads and of masked regions of the last fpl_process_* call is available through
 * fpl_last_segments / fpl_last_mask_regions; fpl_read_result.n_segments counts a read's entries, which are contiguous
 * and in read order; the record's inline seg_* fields hold the first two.
 */
typedef struct fpl_segment {          /* one element of outReads (src/seprocessor.cpp:222-262) */
    int32_t read;                     /* index of the input read in the batch */
    int32_t lo, len;                  /* window on the ORIGINAL read's bytes */
    uint8_t result;                   /* Filter::passFilter code */
    uint8_t median_qual;              /* post-filter Stats median char of a passing segment, else 0 */
    uint8_t split_side;               /* 0 none, 1 "split-by-adapter-left-", 2 "split-by-adapter-right-" (Read::breakByGap) */
    uint8_t is_r1;                    /* 1 if this output read IS r1 (not a copy): --failed_out then shows its masked bases */
    int32_t break_index;              /* 0: not made by Read::breakByRegions; k > 0: name prefix "r<k>-" (src/read.cpp:240,255) */
} fpl_segment;

typedef struct fpl_region {           /* Read::maskRegionWithN: bases [lo, lo+len) of the ORIGINAL read become 'N' */
    int32_t read;
    int32_t lo, len;
} fpl_region;

/* Which of the two Stats objects (ThreadConfig::getPreStats1 / getPostStats1, src/threadconfig.h:20-23). */
enum { FPL_STATS_PRE = 0, FPL_STATS_POST = 1 };

/*
 * Layout of one Stats accumulator block, a single int64 vector (so that one allreduce merges it,
 * replacing Stats::merge src/stats.cpp:1013-1082).  C = cycles (capacity, >= longest read seen):
 *   [0, 8C)            mCycleBaseContents[b][c] at b*C + c              (src/stats.cpp:303)
 *   [8C, 16C)          mCycleBaseQual[b][c] at 8C + b*C + c (sum of qual-33)     (:304)
 *   then FPL_STATS_TAIL int64:
 *     +0    .. +1023   mKmer[0..1023]                                    (:282-347)
 *     +1024 .. +1151   mBaseQualHistogram[128]                           (:293)
 *     +1152 .. +1279   mMedianReadQualHistogram[128]                     (:362)
 *     +1280 .. +1407   mMedianReadQualBases[128]                         (:363)
 *     +1408            mReads    +1409  mLengthSum                       (:269,374)
 * mCycleTotalBase/mCycleTotalQual are the sums over b (SURVEY A.1); the Q20/Q30 per-cycle arrays are dead state.
 */
#define FPL_STATS_KMER 0
#define FPL_STATS_QUALHIST 1024
#define FPL_STATS_MEDHIST 1152
#define FPL_STATS_MEDBASES 1280
#define FPL_STATS_READS 1408
#define FPL_STATS_LENSUM 1409
#define FPL_STATS_TAIL 1536
#define FPL_STATS_WORDS(C) ((int64_t)16 * (C) + FPL_STATS_TAIL)

/*
 * FilterResult accumulator block (src/filterresult.h:58-64), int64 vector of FPL_COUNTER_WORDS:
 *   +0..31  mFilterReadStats[32]   +32 mTrimmedAdapterRead   +33 mTrimmedAdapterBases
 *   +34..37 mTrimmedPolyXReads[4]  +38..41 mTrimmedPolyXBases[4]
 *   +42     reads dropped by trimAndCut (no counter in the reference; bookkeeping)
 *   +43     reads split by a middle adapter (bookkeeping)
 * followed by the adapter event count table: count[(adapter*2 + side) * (FPL_MAX_ADAPTER_LEN+1) + cmplen].
 */
#define FPL_CNT_FILTER 0
#define FPL_CNT_ADAPTER_READS 32
#define FPL_CNT_ADAPTER_BASES 33
#define FPL_CNT_POLYX_READS 34
#define FPL_CNT_POLYX_BASES 38
#define FPL_CNT_DROPPED 42
#define FPL_CNT_SPLIT 43
#define FPL_CNT_FIXED 64
#define FPL_COUNTER_WORDS(n_adapters) (FPL_CNT_FIXED + (int64_t)(n_adapters) * 2 * (FPL_MAX_ADAPTER_LEN + 1))

typedef struct fpl_ctx fpl_ctx;

/* Last error message of the calling thread ("" if none). Replaces error_exit(msg) (src/util.h:270-273): the host decides. */
const char* fpl_last_error(void);
int fpl_abi_version(void);

/*
 * Create / destroy a context.  Replaces the per-worker state built in SingleEndProcessor::process
 * (src/seprocessor.cpp:69-77: ThreadConfig = 2 Stats + FilterResult) plus the read-only Options* the
 * operators consult.  Fails if no CUDA device is usable — there is no CPU fallback.
 */
int fpl_create(const fpl_options* opt, const fpl_adapters* adapters, fpl_ctx** out);
void fpl_destroy(fpl_ctx* ctx);

/*
 * processSingleEnd over a packed batch held in HOST memory (src/seprocessor.cpp:180-329):
 * copies the batch to the device, runs every kernel, accumulates pre/post Stats and FilterResult on the
 * device, and copies the per-read results back into results[n_reads] (host).  Synchronous.
 */
int fpl_process_host(fpl_ctx* ctx, const fpl_batch* host_batch, fpl_read_result* results);

/*
 * Same, for a batch already resident in DEVICE memory (all four pointers are device pointers);
 * results_dev is a device array of n_reads records or NULL to keep results in the context's own buffer.
 * Asynchronous on the context's stream; fpl_sync() waits.
 */
int fpl_process_device(fpl_ctx* ctx, const fpl_batch* dev_batch, fpl_read_result* results_dev);
int fpl_sync(fpl_ctx* ctx);
/* The context's CUDA stream (a cudaStream_t), so a caller can order its own work / events against the kernels. */
void* fpl_stream(fpl_ctx* ctx);

/*
 * One FASTQ record located in a chunk of plain FASTQ text (byte offsets from the start of the chunk).
 * The quality line has seq_len bytes.
 */
typedef struct fpl_fastq_record {
    int64_t name_off;                 /* the '@' of the name line */
    int64_t seq_off;
    int64_t plus_off;                 /* the '+' line (kept verbatim in the output, src/read.cpp:119-143) */
    int64_t qual_off;
    int32_t name_len, seq_len, plus_len, reserved;
} fpl_fastq_record;

/*
 * SURVEY §8f rows 1: FastqReader::getLine / FastqReader::read (src/fastqreader.cpp:219-347) + the pack->batch staging
 * + processSingleEnd, for one chunk of plain-text FASTQ held in HOST memory: the text is copied to the device, the
 * newline index, the record table and the packed batch are built there, every kernel of fpl_process_host runs, and
 * the record table (records[]) and the per-read results (results[]) come back.  *n_records = complete records found,
 * *bytes_consumed = bytes of the chunk they span (the caller prepends the rest to its next chunk); is_last_chunk != 0
 * lets an unterminated last line count.
 * Returns 0 on success; 1 if the chunk is not in the strict layout this path handles (LF line ends, exactly four lines
 * per record, '@' / '+' in place, |sequence| == |quality|, or more than max_records records) — nothing has been
 * accumulated then and the caller must parse this input with the reference reader instead; < 0 on error.
 */
int fpl_process_fastq_host(fpl_ctx* ctx, const uint8_t* text, int64_t n_bytes, int is_last_chunk,
                           fpl_fastq_record* records, fpl_read_result* results, int64_t max_records,
                           int64_t* n_records, int64_t* bytes_consumed);

/*
 * SURVEY §8f row 2, device half: Read::appendToString / appendToStringWithTag (src/read.cpp:119-173) as the per-pack loop
 * of processSingleEnd applies them (src/seprocessor.cpp:264-288), for the chunk the LAST call on this context — a
 * successful fpl_process_fastq_host — has just processed.  The chunk, its record table and the results are still in
 * device memory; this call compacts them into the text the two writer threads receive and copies it to host memory:
 *   out     every passing output read, in input order: name line (with the "r<k>-" / "split-by-adapter-left-/right-"
 *           tags of Read::breakByRegions / breakByGap after the '@'), the window of the bases (masked with --mask), the
 *           '+' line as it was, the window of the qualities
 *   failed  (want_failed != 0, i.e. --failed_out is open) every read whose only output read failed a filter: r1 after
 *           the trims, name + ' ' + FAILED_TYPES[code] (src/common.h:55-64)
 * *out_bytes / *failed_bytes are always set.  Returns 0 on success; 1 if a buffer is too small — nothing was copied, the
 * text stays built on the device and a second call with room only copies; < 0 on error (e.g. the last call was not a
 * successful fpl_process_fastq_host).  A split read appears twice, so the text can be longer than the chunk:
 * 2 * n_bytes + 64 * n_records always suffices.
 */
int fpl_emit_fastq_host(fpl_ctx* ctx, int want_failed, uint8_t* out, int64_t out_cap, int64_t* out_bytes,
                        uint8_t* failed, int64_t failed_cap, int64_t* failed_bytes);

/*
 * Gzip output — the compression step of Writer::writeInternal / libdeflate_gzip_compress (src/writer.cpp:110-126), which the
 * reference runs once per buffer flush on the writer thread.  Each piece is cut into segments of FPL_GZIP_SEGMENT bytes (the
 * last one shorter) and each segment becomes one complete RFC 1952 gzip member (header 1f 8b 08, FLG 0, MTIME 0, XFL 0,
 * OS 255; one dynamic-Huffman deflate block, or stored blocks when those are not larger; CRC-32; ISIZE).  The members of a
 * piece follow each other in input order, an empty piece gives 0 bytes, and any concatenation of them is a valid
 * multi-member gzip stream (zlib, isa-l and gzip read it).  Matches never reach outside their segment.  The bytes are a pure
 * function of the input.  FPL_GZIP_BOUND(n_bytes, n_pieces) bounds the output of n_bytes in n_pieces pieces.
 */
#define FPL_GZIP_SEGMENT 65536
#define FPL_GZIP_BOUND(n_bytes, n_pieces) \
    ((int64_t)(n_bytes) + 28 * ((int64_t)(n_bytes) / FPL_GZIP_SEGMENT + (int64_t)(n_pieces)))

/*
 * Compresses n_pieces pieces held back to back in HOST memory (text; piece_bytes[i] bytes each) on the context's device and
 * stream: the compressed pieces go to out back to back, their sizes to out_piece_bytes[n_pieces].  Fails (< 0) if
 * out_cap < FPL_GZIP_BOUND(total bytes, n_pieces).  Synchronous; uses the context's grow-only scratch and leaves the
 * state of the last fpl_process_fastq_host call alone.  Pieces exist because a writer receives one string per 16-read
 * pack (WriterThread, src/writerthread.cpp:37-48) and each must stay a whole gzip stream.
 */
int fpl_gzip_host(fpl_ctx* ctx, const uint8_t* text, const int64_t* piece_bytes, int32_t n_pieces, uint8_t* out,
                  int64_t out_cap, int64_t* out_piece_bytes);

/*
 * fpl_emit_fastq_host with both texts compressed in HBM (two pieces of one fpl_gzip_host-style launch) before the copy, so
 * only the gzip members cross PCIe: the replacement of Writer::writeInternal's libdeflate_gzip_compress (src/writer.cpp:110-126)
 * for the raw-text path.  Same precondition and the same two-call protocol: *out_bytes / *failed_bytes are always set; 1 = a
 * buffer is too small and nothing was copied (the compressed text stays on the device for a second call); < 0 on error.
 * fpl_emit_fastq_host on the same chunk keeps working and returns the uncompressed text.
 */
int fpl_emit_fastq_gzip_host(fpl_ctx* ctx, int want_failed, uint8_t* out, int64_t out_cap, int64_t* out_bytes,
                             uint8_t* failed, int64_t failed_cap, int64_t* failed_bytes);

/* Output reads / masked regions of the last fpl_process_* call (--mask / --break only; *n = 0 otherwise). */
int fpl_last_segments(fpl_ctx* ctx, fpl_segment* out, int64_t cap, int64_t* n);
int fpl_last_mask_regions(fpl_ctx* ctx, fpl_region* out, int64_t cap, int64_t* n);

/* Copy the context's last device results (n records) to host memory. */
int fpl_fetch_results(fpl_ctx* ctx, fpl_read_result* results, int64_t n_reads);

/*
 * Stats access (replaces reading the private arrays of Stats, src/stats.h:56-113).
 * fpl_stats_cycles: current capacity C.  fpl_stats_reserve grows C (all ranks must agree before an allreduce).
 * fpl_stats_download copies the FPL_STATS_WORDS(C) int64 block to host.
 * fpl_stats_device_ptr exposes the device block so the caller's collective library (NCCL via
 * torch.distributed) can all-reduce it in place — the multi-GPU replacement of Stats::merge.
 */
int64_t fpl_stats_cycles(fpl_ctx* ctx);
int fpl_stats_reserve(fpl_ctx* ctx, int64_t cycles);
int fpl_stats_download(fpl_ctx* ctx, int which, int64_t* out, int64_t n_words);
int fpl_stats_device_ptr(fpl_ctx* ctx, int which, void** dptr, int64_t* n_words);

/* FilterResult counters + adapter event table (replaces FilterResult::merge, src/filterresult.cpp:28-61). */
int64_t fpl_counter_words(fpl_ctx* ctx);
int fpl_counters_download(fpl_ctx* ctx, int64_t* out, int64_t n_words);
int fpl_counters_device_ptr(fpl_ctx* ctx, void** dptr, int64_t* n_words);

/*
 * Multi-GPU merge, one process (or thread) per GPU — the replacement of Stats::merge (src/stats.cpp:1013-1082) and
 * FilterResult::merge (src/filterresult.cpp:28-61), which SingleEndProcessor::process calls on the per-worker
 * ThreadConfigs (src/seprocessor.cpp:108-121).  Reads shard by read, so this is the path's only exchange.
 *   fpl_comm_unique_id   rank 0 creates the rendezvous id (ncclGetUniqueId) and hands its FPL_COMM_ID_BYTES bytes to
 *                        the other ranks by whatever channel the host has (file, socket, torch.distributed broadcast);
 *   fpl_comm_init        every rank joins (ncclCommInitRank, collective); one communicator per context;
 *   fpl_comm_agree_cycles  all-reduce(max) of the longest read accumulated since fpl_reset; grows this rank's Stats
 *                        capacity to it; synchronous (one int64 comes back to the host);
 *   fpl_allreduce_stats  ncclAllReduce(sum, int64) of [0, cycles) of the 16 per-cycle rows, the tail and the counter
 *                        block of both Stats objects + FilterResult, in place, as ONE group on the context's stream:
 *                        stream-ordered behind the kernels, no host synchronisation.  cycles must be the same on every
 *                        rank and cover every rank's longest read; cycles <= 0 = agree first (fpl_comm_agree_cycles).
 * NCCL (libnccl.so.2) is resolved at run time; without it these calls fail loudly and nothing else is affected.
 */
#define FPL_COMM_ID_BYTES 128
int fpl_comm_unique_id(uint8_t* id);
int fpl_comm_init(fpl_ctx* ctx, const uint8_t* id, int rank, int n_ranks);
int fpl_comm_destroy(fpl_ctx* ctx);
int fpl_comm_size(fpl_ctx* ctx);
int fpl_comm_agree_cycles(fpl_ctx* ctx, int64_t* cycles);
int fpl_allreduce_stats(fpl_ctx* ctx, int64_t cycles);

/*
 * SURVEY §8f row 4 — the counting half of Evaluator::evalAdapterAndReadNum (src/evaluator.cpp:105-265), context-free
 * because it runs before the adapters (and so the context) exist: over the reads of a HOST batch (the caller passes what
 * the reference would load: the first <= 64 Ki reads / 512 Mbases of the input) count the ten-mers of the first
 * (side 0: pos in [0, min(len - 10 - shift_tail, 127)]) or last (side 1: pos in [max(0, len - 10 - shift_tail - 128),
 * len - 10 - shift_tail]) positions: counts[key]++, position_acc[key] += pos (side 0) or len - pos (side 1),
 * *total = valid ten-mers seen; key = Evaluator::seq2int's packing (A 0, T/U 1, C 2, G 3, first base most significant;
 * a window holding any other byte is skipped).  counts and position_acc have 1 << 20 entries.  shift_tail is the
 * reference's max(1, opt.trim.tail).  Picking the top key and extending it (getTopKey / extendKeyToAdapter) is O(4^10)
 * table work and stays with the host (fastplong_b200/evaluator.py).  Returns 0, or < 0 on a CUDA error.
 */
int fpl_eval_adapter_kmers(int device, const fpl_batch* host_batch, int32_t shift_tail, int32_t side, uint32_t* counts,
                           uint64_t* position_acc, int64_t* total);

/*
 * SURVEY §8f row 4 — the table half of Evaluator::evalAdapterAndReadNum for one side, host only (no CUDA call; works
 * without a device): from the two ten-mer tables fpl_eval_adapter_kmers filled to the adapter string, by the
 * reference's rules — the number of non-empty keys is taken, counts[AAAAAAAAAA] is ignored, Evaluator::getTopKey
 * (src/evaluator.cpp:266-322) picks the most frequent ten-mer that is not low-complexity (including its quirk of reading
 * the "different neighbours" test off the COUNT's bits), the key is accepted when count > 10 and count * keys > total * 100
 * (:199-201, :241-243), and Evaluator::extendKeyToAdapter (:324-407) grows it base by base, left first, up to 64 bases;
 * a result of <= 16 bases counts as not detected (:203, :245).  is_rna writes U for T (the reference passes isRNA for the
 * read-end adapter only).  counts / position_acc: 1 << 20 entries, not modified.  Writes the NUL-terminated adapter into
 * `adapter` (cap >= 65) and returns its length; 0 = nothing detected (the option stays "auto"); < 0 = bad argument.
 * The same rules as fastplong_b200/evaluator.py:detect_one (tests/test_evaluator.py holds the two to each other and to the
 * reference binary's own detection).
 */
int fpl_eval_pick_adapter(const uint32_t* counts, const uint64_t* position_acc, int64_t total, int32_t is_rna, char* adapter,
                          int32_t cap);

/* Zero all accumulators (a fresh ThreadConfig); stream-ordered, asynchronous. */
int fpl_reset(fpl_ctx* ctx);

/*
 * Measurement hooks.  fpl_set_timing(ctx, 1) brackets every kernel launch with CUDA events on the context's
 * stream and zeroes the per-kernel totals; fpl_last_kernel_times returns, per kernel, the device time (ms) and
 * the number of timed launches accumulated since then (call after fpl_sync).  names/ms/launches hold up to cap
 * entries; returns the number of kernels.  fpl_launch_count = kernel launches made by the context so far.
 */
int fpl_last_kernel_times(fpl_ctx* ctx, const char** names, float* ms, int64_t* launches, int cap);
int64_t fpl_launch_count(fpl_ctx* ctx);
int fpl_set_timing(fpl_ctx* ctx, int enabled);

#ifdef __cplusplus
}
#endif
#endif /* FPLGPU_H */
