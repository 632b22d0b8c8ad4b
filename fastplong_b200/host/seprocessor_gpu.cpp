// Drop-in definition of the reference's class SingleEndProcessor (declared in /root/reference/src/seprocessor.h:23-50)
// whose per-pack hot loop runs on the GPU through the C ABI of include/fplgpu.h.
//
// Built by fastplong_b200/host/Makefile together with the UNMODIFIED reference translation units (everything in
// /root/reference/src except seprocessor.cpp, compiled where they lie) into build/fastplong_gpu: same CLI, same
// FastqReader / ReadPool / WriterThread / Options / JsonReporter / HtmlReporter, this file in the middle.
//
// What stays host-side here is bookkeeping only (SURVEY §8b):
//   * reader thread -> per-worker pack lists -> worker threads -> writer threads, with the writer's
//     one-string-per-pack, round-robin-over-workers contract (src/writerthread.cpp:37-48);
//   * each worker gathers the packs it is dealt into one packed batch (pinned host buffers), calls
//     fpl_process_host() on its own fpl_ctx, then walks the per-read records in pack order to assemble the output
//     strings (Read::appendToString, Read::breakByGap names) and to feed FilterResult / Stats exactly what
//     processSingleEnd would have fed them;
//   * at the end the device-accumulated Stats blocks and the adapter event table are added into each worker's
//     Stats / FilterResult objects so that Stats::merge, summarize and the reporters run unchanged.
// No per-base decision is taken on the host.
#include <algorithm>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <deque>
#include <functional>
#include <mutex>
#include <map>
#include <memory>
#include <string>
#include <thread>
#include <vector>
#include <time.h>
#include <unistd.h>
#include <cuda_runtime_api.h>

// Stats / FilterResult keep their accumulators private and offer no setters (src/stats.h:56-113,
// src/filterresult.h:58-64); this adapter TU is compiled with the class keys opened so that it can ADD the
// device-accumulated arrays into them.  The reference's own TUs are compiled untouched.  Writer / WriterThread are opened
// the same way so that FPL_DEVICE_GZIP can switch a writer's own compression off (see switchWriterToDeviceGzip).
#define private public
#include "stats.h"
#include "filterresult.h"
#include "writer.h"
#include "writerthread.h"
#undef private
#include "seprocessor.h"
#include "fastqreader.h"
#include "jsonreporter.h"
#include "htmlreporter.h"
#include "util.h"
#include "fplgpu.h"

namespace {

// ---- pinned, growable host buffer ----
template <typename T>
struct Pinned {
    T* p = nullptr;
    size_t cap = 0;
    // page-locking is slow (tens of ms per call): grow rarely, never shrink
    void reserve(size_t n, size_t at_least = 0) {
        if (n <= cap) return;
        size_t want = cap ? cap : (at_least ? at_least : 1024);
        while (want < n) want *= 2;
        T* q = nullptr;
        if (cudaMallocHost((void**)&q, want * sizeof(T)) != cudaSuccess) error_exit("fastplong_gpu: cudaMallocHost failed");
        if (p) cudaFreeHost(p);
        p = q; cap = want;
    }
    ~Pinned() { if (p) cudaFreeHost(p); }
};

struct GpuWorker {
    fpl_ctx* ctx = nullptr;
    Pinned<uint8_t> seq, qual;
    Pinned<int64_t> offsets;
    Pinned<int32_t> lens;
    Pinned<fpl_read_result> results;
    std::vector<ReadPack*> packs;
};

// how many bases a worker gathers before it submits (bounded so that host memory stays bounded like the reference's
// PACK_IN_MEM_LIMIT does, src/common.h:38)
const int64_t kBatchBases = 48ll << 20;
const size_t kSlotAlign = 128;

fpl_options makeAbiOptions(Options* o, int device) {
    fpl_options a;
    memset(&a, 0, sizeof(a));
    a.struct_size = sizeof(a);
    a.device = device;
    a.trim_front = o->trim.front;
    a.trim_tail = o->trim.tail;
    a.cut_front_enabled = o->qualityCut.enabledFront;
    a.cut_front_window = o->qualityCut.windowSizeFront;
    a.cut_front_quality = o->qualityCut.qualityFront;
    a.cut_tail_enabled = o->qualityCut.enabledTail;
    a.cut_tail_window = o->qualityCut.windowSizeTail;
    a.cut_tail_quality = o->qualityCut.qualityTail;
    a.polyx_enabled = o->polyXTrim.enabled;
    a.polyx_min_len = o->polyXTrim.minLen;
    a.adapter_enabled = o->adapter.enabled;
    a.trimming_extension = o->adapter.trimmingExtension;
    a.ed_max = o->adapter.edMax;
    a.qual_filter_enabled = o->qualfilter.enabled;
    a.qualified_qual = o->qualfilter.qualifiedQual;
    a.unqualified_percent_limit = o->qualfilter.unqualifiedPercentLimit;
    a.avg_qual_req = o->qualfilter.avgQualReq;
    a.n_base_percent_limit = o->qualfilter.nBasePercentLimit;
    a.n_base_limit = o->qualfilter.nBaseLimit;
    a.length_filter_enabled = o->lengthFilter.enabled;
    a.length_required = o->lengthFilter.requiredLength;
    a.length_max = o->lengthFilter.maxLength;
    a.complexity_enabled = o->complexityFilter.enabled;
    a.complexity_threshold_pct = (int)(o->complexityFilter.threshold * 100.0 + 0.5);  // src/main.cpp:205 divided an int by 100.0
    a.mask_enabled = o->mask.enabled; a.mask_window = o->mask.windowSize; a.mask_quality = o->mask.quality;
    a.break_enabled = o->breakOpt.enabled; a.break_window = o->breakOpt.windowSize; a.break_quality = o->breakOpt.quality;
    return a;
}

void check(int rc, const char* what) {
    if (rc != 0) error_exit(std::string("fastplong_gpu: ") + what + ": " + fpl_last_error());
}

// "@name" -> "@split-by-adapter-left-name" (Read::breakByGap, src/read.cpp:199-200, 208-209)
void appendRecord(std::string& out, const std::string& name, const char* tagAfterAt, const char* nameSuffix,
                  const char* seq, const char* qual, int n, const std::string& strand) {
    if (tagAfterAt && !name.empty()) {
        out.append(name, 0, 1);
        out.append(tagAfterAt);
        out.append(name, 1, std::string::npos);
    } else {
        out.append(name);
    }
    if (nameSuffix) { out.push_back(' '); out.append(nameSuffix); }
    out.push_back('\n');
    out.append(seq, n);
    out.push_back('\n');
    out.append(strand);
    out.push_back('\n');
    out.append(qual, n);
    out.push_back('\n');
}

// One input read as the host sees it (Read object or extents in a raw FASTQ chunk).
struct ReadView {
    const char* name; size_t name_len;
    const char* seq; const char* qual; int len;
    const char* strand; size_t strand_len;
};

void appendView(std::string& out, const ReadView& v, const char* seq, const std::string& prefixAfterAt, const char* nameSuffix,
                int lo, int n) {
    if (!prefixAfterAt.empty() && v.name_len > 0) {
        out.append(v.name, 1);
        out.append(prefixAfterAt);
        out.append(v.name + 1, v.name_len - 1);
    } else {
        out.append(v.name, v.name_len);
    }
    if (nameSuffix) { out.push_back(' '); out.append(nameSuffix); }
    out.push_back('\n');
    out.append(seq + lo, n);
    out.push_back('\n');
    out.append(v.strand, v.strand_len);
    out.push_back('\n');
    out.append(v.qual + lo, n);
    out.push_back('\n');
}

// Everything processSingleEnd does with one read AFTER the per-base work (src/seprocessor.cpp:264-288 and the
// FilterResult / Stats side effects), driven by the device's record.  segs/regs: this read's entries of the
// --mask/--break lists (nullptr in the plain mode, where the record's inline segments are used).
bool scatterRead(const ReadView& v, const fpl_read_result& rr, const fpl_segment* segs, const fpl_region* regs, int nregs,
                 ThreadConfig* config, bool haveFailedWriter, std::string& outstr, std::string& failedOut, std::string& scratch,
                 bool text = true) {      // text == false: the output text comes from fpl_emit_fastq_host, only the side effects here
    Stats* pre = config->getPreStats1();
    Stats* post = config->getPostStats1();
    FilterResult* fr = config->getFilterResult();
    const int L = v.len;
    pre->mLengthVec.push_back(L);
    pre->mNeedCalcLength = true;
    if (L > 0) pre->mQualLength[(char)rr.pre_median_qual].push_back(L);
    if (rr.flags & FPL_FLAG_POLYX) fr->addPolyXTrimmed(rr.polyx_base, rr.polyx_len);
    if (rr.adapter_trimmed_bases > 0) fr->addReadTrimmed(rr.adapter_trimmed_bases);
    const char* mseq = v.seq;          // masked view of the bases (Read::maskRegionWithN), only materialised if needed
    if (nregs > 0 && text) {
        scratch.assign(v.seq, (size_t)L);
        for (int k = 0; k < nregs; k++) memset(&scratch[regs[k].lo], 'N', (size_t)regs[k].len);
        mseq = scratch.data();
    }
    bool passed = false;
    for (int k = 0; k < rr.n_segments; k++) {
        int lo, ln, code, median, side, bidx, isR1;
        if (segs) {
            lo = segs[k].lo; ln = segs[k].len; code = segs[k].result; median = segs[k].median_qual;
            side = segs[k].split_side; bidx = segs[k].break_index; isR1 = segs[k].is_r1;
        } else {
            lo = rr.seg_lo[k]; ln = rr.seg_len[k]; code = rr.seg_result[k]; median = rr.seg_median_qual[k];
            side = (rr.flags & FPL_FLAG_MIDDLE_ADAPTER) ? ((k == 1 || (rr.flags & FPL_FLAG_SEG0_IS_RIGHT)) ? 2 : 1) : 0;
            bidx = 0; isR1 = side == 0;
        }
        config->addFilterResult(code, 1);
        if (code == PASS_FILTER) {
            std::string prefix;          // "r<k>-" (Read::breakByRegions) goes in front of the breakByGap tag
            if (bidx && text) prefix = "r" + std::to_string(bidx) + "-";
            if (side && text) prefix += side == 2 ? "split-by-adapter-right-" : "split-by-adapter-left-";
            if (text) appendView(outstr, v, mseq, prefix, NULL, lo, ln);
            passed = true;
            post->mLengthVec.push_back(ln);
            post->mNeedCalcLength = true;
            if (ln > 0) post->mQualLength[(char)median].push_back(ln);
        } else if (haveFailedWriter && rr.n_segments == 1 && text) {
            // the reference prints or1, trimmed in place — and masked in place only if the output read IS r1 (:278-280)
            appendView(failedOut, v, isR1 ? mseq : v.seq, std::string(), FAILED_TYPES[code], rr.trim_lo, rr.trim_len);
        }
    }
    return passed;
}

// the --mask/--break lists of the last call on this context, grouped per read while walking the records in order
struct ExtLists {
    std::vector<fpl_segment> segs;
    std::vector<fpl_region> regs;
    size_t sp = 0, rp = 0;
    bool on = false;
    void fetch(fpl_ctx* ctx, bool enabled) {
        on = enabled; sp = rp = 0;
        if (!on) return;
        int64_t n = 0;
        fpl_last_segments(ctx, NULL, 0, &n);
        segs.resize((size_t)n);
        if (n) check(fpl_last_segments(ctx, segs.data(), n, &n), "fpl_last_segments");
        fpl_last_mask_regions(ctx, NULL, 0, &n);
        regs.resize((size_t)n);
        if (n) check(fpl_last_mask_regions(ctx, regs.data(), n, &n), "fpl_last_mask_regions");
    }
    // entries of read i (records are walked in order, the lists are in read order)
    const fpl_segment* segsOf(int nseg) { const fpl_segment* p = on ? segs.data() + sp : NULL; if (on) sp += (size_t)nseg; return p; }
    const fpl_region* regsOf(int64_t read, int& n) {
        n = 0;
        if (!on) return NULL;
        const fpl_region* p = regs.data() + rp;
        while (rp < regs.size() && regs[rp].read == read) { rp++; n++; }
        return p;
    }
};

void addStatsBlock(Stats* s, const std::vector<int64_t>& blk, int64_t C) {
    int64_t used = 0;
    for (int64_t c = 0; c < C; c++)
        for (int b = 0; b < 8; b++)
            if (blk[b * C + c]) used = c + 1;
    if (used > s->mBufLen) s->extendBuffer((int)used);
    for (int b = 0; b < 8; b++)
        for (int64_t c = 0; c < used; c++) {
            const long n = blk[b * C + c], q = blk[8 * C + b * C + c];
            s->mCycleBaseContents[b][c] += n;
            s->mCycleBaseQual[b][c] += q;
            s->mCycleTotalBase[c] += n;      // the two row-sum arrays of src/stats.cpp:306-307
            s->mCycleTotalQual[c] += q;
        }
    const int64_t* t = blk.data() + 16 * C;
    for (int k = 0; k < 1024; k++) s->mKmer[k] += t[FPL_STATS_KMER + k];
    for (int k = 0; k < 128; k++) {
        s->mBaseQualHistogram[k] += t[FPL_STATS_QUALHIST + k];
        s->mMedianReadQualHistogram[k] += t[FPL_STATS_MEDHIST + k];
        s->mMedianReadQualBases[k] += t[FPL_STATS_MEDBASES + k];
    }
    s->mReads += t[FPL_STATS_READS];
    s->mLengthSum += t[FPL_STATS_LENSUM];
}

// ---------------------------------------------------------------------------------------------------------------
// Raw-text path (SURVEY §8f rows 1-2): for a plain (not gzipped) FASTQ file the device finds the records itself
// (fpl_process_fastq_host) and the output strings are cut straight out of the file chunk; the reference's
// FastqReader / ReadPool are not involved.  Chunks are cut on the host at record boundaries so that they are
// independent; chunk k goes to worker k % T and its output string to writer list k % T, which is exactly the order the
// writer threads consume (src/writerthread.cpp:37-48).
// ---------------------------------------------------------------------------------------------------------------
struct TextChunk {
    uint8_t* p = nullptr;      // pinned
    size_t cap = 0, n = 0;
    bool last = false;
};

struct ChunkQueue {
    std::mutex mu;
    std::condition_variable cv;
    std::deque<TextChunk*> q;
    bool done = false;
    void push(TextChunk* c) { { std::lock_guard<std::mutex> l(mu); q.push_back(c); } cv.notify_all(); }
    void finish() { { std::lock_guard<std::mutex> l(mu); done = true; } cv.notify_all(); }
    TextChunk* pop() {   // nullptr when finished
        std::unique_lock<std::mutex> l(mu);
        cv.wait(l, [&] { return !q.empty() || done; });
        if (q.empty()) return nullptr;
        TextChunk* c = q.front(); q.pop_front();
        return c;
    }
};

TextChunk* newChunk(size_t cap) {
    TextChunk* c = new TextChunk();
    if (cudaMallocHost((void**)&c->p, cap) != cudaSuccess) error_exit("fastplong_gpu: cudaMallocHost failed");
    c->cap = cap;
    return c;
}
void growChunk(TextChunk* c, size_t cap) {
    uint8_t* q = nullptr;
    if (cudaMallocHost((void**)&q, cap) != cudaSuccess) error_exit("fastplong_gpu: cudaMallocHost failed");
    memcpy(q, c->p, c->n);
    cudaFreeHost(c->p);
    c->p = q; c->cap = cap;
}

// Largest prefix of buf[0..n) that ends at a record boundary: a newline followed by an '@' line whose line-after-next
// starts with '+' (a quality line may start with '@', but then the line two below it is a sequence, not a '+' line).
size_t recordBoundary(const uint8_t* buf, size_t n) {
    size_t end = n;
    while (end > 0) {
        const uint8_t* nl = (const uint8_t*)memrchr(buf, '\n', end);
        if (!nl) return 0;
        const size_t p = (size_t)(nl - buf) + 1;                 // candidate: a record starts at p
        if (p < n && buf[p] == '@') {
            const uint8_t* l1 = (const uint8_t*)memchr(buf + p, '\n', n - p);
            const uint8_t* l2 = l1 ? (const uint8_t*)memchr(l1 + 1, '\n', n - (size_t)(l1 + 1 - buf)) : nullptr;
            if (l2 && (size_t)(l2 + 1 - buf) < n && l2[1] == '+') return p;
        }
        end = (size_t)(nl - buf);
    }
    return 0;
}

// The device parser takes the strict layout only (LF line ends, four lines per record); everything else the reference
// accepts — CR or CRLF line ends, blank or stray lines between records, a truncated last record
// (FastqReader::getLine / read, src/fastqreader.cpp:219-347) — goes through the reference's own reader.  This looks at
// the head and the tail of the file so that such a file is routed there before any work is done; a deviation in the
// middle of a file is caught later (the raw-text run is then abandoned and restarted, see process()).
bool looksStrict(const std::string& path) {
    FILE* fp = fopen(path.c_str(), "rb");
    if (!fp) return false;
    const size_t kHead = 1u << 20, kTail = 1u << 16;
    std::vector<unsigned char> buf(kHead);
    size_t n = fread(buf.data(), 1, kHead, fp);
    bool ok = true;
    if (n > 0 && buf[0] != '@') ok = false;
    if (memchr(buf.data(), '\r', n)) ok = false;
    for (size_t i = 1; ok && i < n; i++)
        if (buf[i] == '\n' && buf[i - 1] == '\n') ok = false;                  // a blank line
    if (ok && n == kHead && fseek(fp, -(long)kTail, SEEK_END) == 0) {
        n = fread(buf.data(), 1, kTail, fp);
        if (memchr(buf.data(), '\r', n)) ok = false;
        for (size_t i = 1; ok && i < n; i++)
            if (buf[i] == '\n' && buf[i - 1] == '\n') ok = false;
    }
    fclose(fp);
    return ok;
}

bool rawTextEligible(Options* o) {
    if (getenv("FPL_HOST_PARSE")) return false;
    if (o->inputFromSTDIN || o->in == "/dev/stdin" || ends_with(o->in, ".gz")) return false;
    if (o->readsToProcess > 0 || o->split.enabled) return false;
    if (o->outputToSTDOUT) return false;      // an abandoned raw-text run cannot take back what it wrote to a pipe
    return looksStrict(o->in);
}

}  // namespace

// -------------------------------------------------------------------------------------------------------------------
// The per-worker GPU state lives outside the class (its layout is fixed by the reference header).
static std::vector<std::unique_ptr<GpuWorker>> g_workers;
static std::vector<std::string> g_adapters;   // fpl_adapters order

SingleEndProcessor::SingleEndProcessor(Options* opt) {
    mOptions = opt;
    mReaderFinished = false;
    mFinishedThreads = 0;
    mFilter = new Filter(opt);
    mLeftWriter = NULL;
    mFailedWriter = NULL;
    mInputLists = NULL;
    mPackReadCounter = 0;
    mPackProcessedCounter = 0;
    mReadPool = new ReadPool(mOptions);
}

SingleEndProcessor::~SingleEndProcessor() {
    delete mFilter;
    delete mReadPool;
    delete[] mInputLists;
}

// FPL_DEVICE_GZIP=1: a writer whose file name ends in ".gz" no longer compresses (Writer::writeInternal's
// libdeflate_gzip_compress, src/writer.cpp:110-126, on the single writer thread); the workers hand it strings that are
// already whole gzip members, compressed on the device, and it only writes them.  Members may be concatenated at any
// buffer boundary, so the file stays one valid multi-member gzip stream.  --split and --stdout ignore the knob.
static bool g_gzLeft = false, g_gzFailed = false;   // the workers compress the --out / --failed_out strings

static bool switchWriterToDeviceGzip(WriterThread* wt, Options* opt) {
    if (!wt || !getenv("FPL_DEVICE_GZIP") || opt->split.enabled || wt->mWriter1 == NULL || wt->mWriter1->mSTDOUT ||
        !ends_with(wt->mFilename, ".gz"))
        return false;
    Writer* w = wt->mWriter1;
    if (w->mZipped) {
        libdeflate_free_compressor(w->mCompressor);
        w->mCompressor = NULL;
        w->mZipped = false;
    }
    return true;
}

// Compresses the non-null strings in place on the device, each into whole gzip members: one fpl_gzip_host call for all.
static void gzipStrings(fpl_ctx* ctx, const std::vector<std::string*>& strs) {
    thread_local Pinned<uint8_t> in, out;
    thread_local std::vector<int64_t> sizes, outSizes;
    sizes.clear();
    size_t total = 0;
    for (std::string* s : strs) if (s) { sizes.push_back((int64_t)s->size()); total += s->size(); }
    if (sizes.empty()) return;
    const int64_t bound = FPL_GZIP_BOUND((int64_t)total, (int64_t)sizes.size());
    in.reserve(total + 1, 1u << 20);
    out.reserve((size_t)bound + 1, 1u << 20);
    size_t o = 0;
    for (std::string* s : strs) if (s) { memcpy(in.p + o, s->data(), s->size()); o += s->size(); }
    outSizes.assign(sizes.size(), 0);
    check(fpl_gzip_host(ctx, in.p, sizes.data(), (int32_t)sizes.size(), out.p, bound, outSizes.data()), "fpl_gzip_host");
    size_t k = 0;
    o = 0;
    for (std::string* s : strs)
        if (s) { s->assign((const char*)out.p + o, (size_t)outSizes[k]); o += (size_t)outSizes[k]; k++; }
}

void SingleEndProcessor::initOutput() {
    if (!mOptions->failedOut.empty()) mFailedWriter = new WriterThread(mOptions, mOptions->failedOut);
    g_gzFailed = switchWriterToDeviceGzip(mFailedWriter, mOptions);
    g_gzLeft = false;
    if (mOptions->out.empty() && !mOptions->outputToSTDOUT) return;
    mLeftWriter = new WriterThread(mOptions, mOptions->out, mOptions->outputToSTDOUT);
    g_gzLeft = switchWriterToDeviceGzip(mLeftWriter, mOptions);
}

void SingleEndProcessor::closeOutput() {
    delete mLeftWriter; mLeftWriter = NULL;
    delete mFailedWriter; mFailedWriter = NULL;
}

void SingleEndProcessor::initConfig(ThreadConfig* config) {
    if (mOptions->out.empty()) return;
    if (mOptions->split.enabled) config->initWriterForSplit();
}

void SingleEndProcessor::recycleToPool(int tid, Read* r) {
    if (!mReadPool->input(tid, r)) delete r;
}

void SingleEndProcessor::writerTask(WriterThread* w) {
    while (true) {
        if (w->isCompleted()) { w->output(); break; }   // drain what is left, as the reference's loop does
        w->output();
    }
    if (mOptions->verbose) loginfo(w->getFilename() + " writer finished");
}

// Reader: identical contract to the reference's (16-read packs dealt round-robin, src/seprocessor.cpp:331-429).
void SingleEndProcessor::readerTask() {
    if (mOptions->verbose) loginfo("start to load data");
    FastqReader reader(mOptions->in, true);
    reader.setReadPool(mReadPool);
    const int T = mOptions->thread;
    long total = 0, reported = 0;
    bool stop = false;
    // Back-pressure by BYTES, not packs (the reference bounds packs because it works pack by pack; a GPU worker gathers
    // kBatchBases before it submits): the reader stays at most about three batches per worker — capped at 1.5 Gbases in
    // all — ahead of what the workers have taken, and the writer's backlog is held to the same number of packs.
    long packBasesSum = 0;
    const long aheadBases = std::min<long>(3L * kBatchBases * T, 1536L << 20);
    while (!stop) {
        ReadPack* pack = new ReadPack;
        pack->data = new Read*[PACK_SIZE];
        pack->count = 0;
        while (pack->count < PACK_SIZE) {
            Read* r = reader.read();
            if (!r) { stop = true; break; }
            pack->data[pack->count++] = r;
            total++;
            if (mOptions->readsToProcess > 0 && total >= mOptions->readsToProcess) { stop = true; break; }
        }
        // the reference always emits a final (possibly empty) pack when the input ends on a pack boundary
        if (pack->count == 0 && !stop) { delete[] pack->data; delete pack; continue; }
        for (int i = 0; i < pack->count; i++) packBasesSum += (long)pack->data[i]->mSeq->length();
        mInputLists[mPackReadCounter % T]->produce(pack);
        mPackReadCounter++;
        if (mOptions->verbose && total >= reported + 1000000) {
            reported = total;
            loginfo("loaded " + to_string(reported / 1000000) + "M reads");
        }
        const long avgPack = std::max<long>(1, packBasesSum / (long)mPackReadCounter);
        const long aheadPacks = std::max<long>(2L * T, aheadBases / avgPack);
        while (!stop && (long)mPackReadCounter - mPackProcessedCounter > aheadPacks) usleep(200);
        if (mLeftWriter)
            while (!stop && mLeftWriter->bufferLength() > aheadPacks) usleep(1000);
    }
    for (int t = 0; t < T; t++) mInputLists[t]->setProducerFinished();
    mReaderFinished = true;
    if (mOptions->verbose) loginfo("Loading completed with " + to_string(mPackReadCounter) + " packs");
}

// processSingleEnd for a whole batch of packs at once; `pack` == NULL flushes config's pending packs.
// (The reference calls it once per pack; the GPU path gathers packs, see processorTask.)
bool SingleEndProcessor::processSingleEnd(ReadPack* pack, ThreadConfig* config) {
    const int tid = config->getThreadId();
    GpuWorker& w = *g_workers[tid];
    if (pack) { w.packs.push_back(pack); return true; }
    if (w.packs.empty()) return true;

    // ---- gather: packed batch in pinned memory ----
    size_t nreads = 0, nbytes = 0;
    for (ReadPack* p : w.packs)
        for (int i = 0; i < p->count; i++) {
            nreads++;
            nbytes += (p->data[i]->mSeq->length() + kSlotAlign - 1) / kSlotAlign * kSlotAlign;
        }
    // pinned buffers grow to what the batches need (doubling: a small input pins little, a large one re-pins a few times)
    w.seq.reserve(nbytes + 256, 1u << 20); w.qual.reserve(nbytes + 256, 1u << 20);
    w.offsets.reserve(nreads + 1, 1u << 12); w.lens.reserve(nreads + 1, 1u << 12); w.results.reserve(nreads + 1, 1u << 12);
    size_t k = 0, off = 0;
    for (ReadPack* p : w.packs)
        for (int i = 0; i < p->count; i++) {
            Read* r = p->data[i];
            const size_t n = r->mSeq->length();
            if (r->mQuality->length() != n) error_exit("sequence and quality have different lengths: " + *r->mName);
            memcpy(w.seq.p + off, r->mSeq->data(), n);
            memcpy(w.qual.p + off, r->mQuality->data(), n);
            w.offsets.p[k] = (int64_t)off;
            w.lens.p[k] = (int32_t)n;
            off += (n + kSlotAlign - 1) / kSlotAlign * kSlotAlign;
            k++;
        }
    fpl_batch b;
    b.seq = w.seq.p; b.qual = w.qual.p; b.offsets = w.offsets.p; b.lens = w.lens.p;
    b.n_reads = (int64_t)nreads; b.n_bytes = (int64_t)off;
    check(fpl_process_host(w.ctx, &b, w.results.p), "fpl_process_host");

    // ---- scatter: walk the records in pack order (src/seprocessor.cpp:186-326) ----
    ExtLists ext;
    ext.fetch(w.ctx, mOptions->mask.enabled || mOptions->breakOpt.enabled);
    std::string scratch;
    k = 0;
    // FPL_DEVICE_GZIP: the batch's strings are compressed together (one device call) and then handed on in pack order
    const bool gz = (mLeftWriter && g_gzLeft) || (mFailedWriter && g_gzFailed);
    std::vector<std::pair<string*, string*>> held;
    for (ReadPack* p : w.packs) {
        string* outstr = new string();
        string* failedOut = new string();
        int readPassed = 0;
        for (int i = 0; i < p->count; i++, k++) {
            Read* or1 = p->data[i];
            const fpl_read_result& rr = w.results.p[k];
            ReadView v = {or1->mName->data(), or1->mName->length(), or1->mSeq->data(), or1->mQuality->data(),
                          (int)or1->mSeq->length(), or1->mStrand->data(), or1->mStrand->length()};
            int nregs = 0;
            const fpl_segment* sg = ext.segsOf(rr.n_segments);
            const fpl_region* rg = ext.regsOf((int64_t)k, nregs);
            if (scatterRead(v, rr, sg, rg, nregs, config, mFailedWriter != NULL, *outstr, *failedOut, scratch)) readPassed++;
            recycleToPool(tid, or1);
        }
        if (mOptions->split.enabled) {
            if (!mOptions->out.empty()) config->getWriter1()->writeString(outstr);
        }
        if (gz) {
            held.emplace_back(mLeftWriter ? outstr : NULL, mFailedWriter ? failedOut : NULL);
            if (mLeftWriter) outstr = NULL;
            if (mFailedWriter) failedOut = NULL;
        }
        if (mLeftWriter && outstr) { mLeftWriter->input(tid, outstr); outstr = NULL; }
        if (mFailedWriter && failedOut) { mFailedWriter->input(tid, failedOut); failedOut = NULL; }
        if (mOptions->split.byFileLines) config->markProcessed(readPassed);
        else config->markProcessed(p->count);
        delete outstr;
        delete failedOut;
        delete[] p->data;
        delete p;
    }
    w.packs.clear();
    if (gz) {
        std::vector<std::string*> strs;
        for (auto& h : held) {
            strs.push_back(g_gzLeft ? h.first : NULL);
            strs.push_back(g_gzFailed ? h.second : NULL);
        }
        gzipStrings(w.ctx, strs);
        for (auto& h : held) {
            if (h.first) mLeftWriter->input(tid, h.first);
            if (h.second) mFailedWriter->input(tid, h.second);
        }
    }
    return true;
}

void SingleEndProcessor::processorTask(ThreadConfig* config) {
    SingleProducerSingleConsumerList<ReadPack*>* input = config->getInput();
    int64_t pending = 0;
    while (true) {
        if (config->canBeStopped()) break;
        bool idle = true;
        while (input->canBeConsumed()) {
            ReadPack* pack = input->consume();
            for (int i = 0; i < pack->count; i++) pending += (int64_t)pack->data[i]->mSeq->length();
            processSingleEnd(pack, config);   // gathers
            mPackProcessedCounter++;           // "taken": lets the reader run ahead by a bounded number of packs
            idle = false;
            if (pending >= kBatchBases) break;
        }
        if (pending >= kBatchBases || (idle && pending > 0) || (input->isProducerFinished() && !input->canBeConsumed())) {
            processSingleEnd(NULL, config);   // submit + scatter
            pending = 0;
        }
        if (input->isProducerFinished() && !input->canBeConsumed()) {
            if (mOptions->verbose) loginfo("thread " + to_string(config->getThreadId() + 1) + " data processing completed");
            break;
        }
        if (idle) usleep(100);
    }
    input->setConsumerFinished();
    mFinishedThreads++;
    if (mFinishedThreads == mOptions->thread) {
        if (mLeftWriter) mLeftWriter->setInputCompleted();
        if (mFailedWriter) mFailedWriter->setInputCompleted();
    }
    if (mOptions->verbose) loginfo("thread " + to_string(config->getThreadId() + 1) + " finished");
}

static double nowSec();
// The CUDA driver takes about 1.5 s to come up on an 8-GPU box.  Start it when the program is loaded, so that it
// overlaps main()'s option parsing and evaluator pre-pass (reference code, src/main.cpp:255-285); process() waits for
// it.  Only when the command line names an input file (not for --help / --version); FPL_NO_WARMUP=1 disables it.
struct CudaWarmup {
    std::thread th;
    double t0;
    CudaWarmup() : t0(nowSec()) {
        if (getenv("FPL_NO_WARMUP")) return;
        bool hasInput = false;
        if (FILE* f = fopen("/proc/self/cmdline", "rb")) {
            std::vector<char> buf(1 << 16);
            const size_t n = fread(buf.data(), 1, buf.size() - 1, f);
            fclose(f);
            for (size_t i = 0; i < n;) {
                const char* a = buf.data() + i;
                if (!strcmp(a, "-i") || !strcmp(a, "--in") || !strncmp(a, "--in=", 5)) hasInput = true;
                i += strlen(a) + 1;
            }
        }
        if (hasInput) th = std::thread([] { cudaFree(0); });
    }
    void wait() { if (th.joinable()) th.join(); }
    ~CudaWarmup() { wait(); }
};
static CudaWarmup g_warm;

static double nowSec() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec + ts.tv_nsec * 1e-9;
}
#define FPL_STAMP(what) do { if (timing) { double t_ = nowSec(); fprintf(stderr, "[fastplong_gpu] %-34s %8.3f s\n", what, t_ - t_last); t_last = t_; } } while (0)

bool SingleEndProcessor::process() {
    const bool timing = getenv("FPL_TIMING") != nullptr;
    double t_last = g_warm.t0;
    FPL_STAMP("program start -> process()");
    // opening --out truncates whatever the path held before (about 1 s for a multi-GB file on tmpfs): do it while the
    // driver is still starting
    if (!mOptions->split.enabled) initOutput();
    FPL_STAMP("writers (initOutput)");
    g_warm.wait();
    FPL_STAMP("wait for the CUDA driver");
    const int T = mOptions->thread;

    // one GPU context per worker thread; workers are spread over the visible devices
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        error_exit("fastplong_gpu: no CUDA device available (this build has no CPU fallback for the hot path)");
    FPL_STAMP("cudaGetDeviceCount");
    g_adapters.clear();
    g_adapters.push_back(mOptions->adapter.sequenceStart);
    g_adapters.push_back(mOptions->adapter.sequenceEnd);
    if (mOptions->adapter.hasFasta)
        for (auto& s : mOptions->adapter.seqsInFasta) g_adapters.push_back(s);
    std::vector<const char*> fasta;
    for (size_t i = 2; i < g_adapters.size(); i++) fasta.push_back(g_adapters[i].c_str());
    fpl_adapters ad;
    ad.start = g_adapters[0].c_str(); ad.end = g_adapters[1].c_str();
    ad.n_fasta = (int)fasta.size(); ad.fasta = fasta.empty() ? NULL : fasta.data();
    g_workers.clear();
    for (int t = 0; t < T; t++) g_workers.emplace_back(new GpuWorker());
    {
        // the contexts are independent: create them side by side (the first one pays the driver start-up and the
        // kernel specialisation, the others find both cached)
        std::vector<int> rc(T, 0);
        std::vector<std::string> msg(T);
        std::vector<std::thread> mk;
        for (int t = 0; t < T; t++) mk.emplace_back([&, t] {
            fpl_options o = makeAbiOptions(mOptions, t % ndev);
            rc[t] = fpl_create(&o, &ad, &g_workers[t]->ctx);
            if (rc[t]) msg[t] = fpl_last_error();
        });
        for (auto& th : mk) th.join();
        for (int t = 0; t < T; t++)
            if (rc[t]) error_exit("fastplong_gpu: fpl_create: " + msg[t]);
    }

    FPL_STAMP("CUDA init + contexts + JIT");
    mInputLists = new SingleProducerSingleConsumerList<ReadPack*>*[T];
    std::vector<ThreadConfig*> configs(T);
    for (int t = 0; t < T; t++) {
        mInputLists[t] = new SingleProducerSingleConsumerList<ReadPack*>();
        configs[t] = new ThreadConfig(mOptions, t, false);
        configs[t]->setInputList(mInputLists[t]);
        initConfig(configs[t]);
    }

    std::unique_ptr<std::thread> leftWriter, failedWriter;
    if (mLeftWriter) leftWriter.reset(new std::thread(std::bind(&SingleEndProcessor::writerTask, this, mLeftWriter)));
    if (mFailedWriter) failedWriter.reset(new std::thread(std::bind(&SingleEndProcessor::writerTask, this, mFailedWriter)));

    FPL_STAMP("thread configs (Stats objects)");
    bool rawText = rawTextEligible(mOptions);
    if (rawText) {
        // ---- raw-text path: chunk reader -> T workers (device ingest + processSingleEnd + output assembly) ----
        // 32 MB of text per chunk (FPL_CHUNK_KB: smaller chunks, for tests of the chunk plumbing on small inputs)
        const size_t kChunk = getenv("FPL_CHUNK_KB") ? (size_t)std::max(1L, atol(getenv("FPL_CHUNK_KB"))) << 10 : (size_t)32 << 20;
        std::vector<ChunkQueue> queues(T);
        ChunkQueue freeList;
        for (int i = 0; i < T + 2; i++) freeList.push(newChunk(kChunk + (8u << 20)));
        FILE* fp = fopen(mOptions->in.c_str(), "rb");
        if (!fp) error_exit("Failed to open file: " + mOptions->in);
        WriterThread* left = mLeftWriter;
        WriterThread* failedW = mFailedWriter;
        Options* opt = mOptions;
        std::atomic<int> notStrict(0);
        // finished chunks the writer may hold before the workers wait (FPL_WRITER_BACKLOG: chunks per worker, default 2)
        const long backlog = (getenv("FPL_WRITER_BACKLOG") ? std::max(1L, atol(getenv("FPL_WRITER_BACKLOG"))) : 2L) * T;
        std::atomic<long> delivered(0);                         // chunks handed to the writers so far (all workers)
        const bool deviceEmit = getenv("FPL_DEVICE_EMIT") != nullptr;
        if (mOptions->verbose) loginfo("start to load data");
        std::thread reader([&] {
            TextChunk* cur = freeList.pop();
            cur->n = 0;
            long k = 0;
            bool eof = false;
            while (!eof && !notStrict) {
                if (cur->cap - cur->n < kChunk) growChunk(cur, cur->cap * 2);
                const size_t got = fread(cur->p + cur->n, 1, kChunk, fp);
                cur->n += got;
                eof = got < kChunk;
                size_t cut = eof ? cur->n : recordBoundary(cur->p, cur->n);
                if (!eof && cut == 0) continue;                       // one record larger than the chunk: keep reading
                TextChunk* next = nullptr;
                if (!eof) {
                    next = freeList.pop();
                    if (next->cap < cur->n - cut + kChunk) growChunk(next, cur->n - cut + kChunk + (8u << 20));
                    next->n = cur->n - cut;
                    memcpy(next->p, cur->p + cut, next->n);
                }
                cur->n = cut; cur->last = eof;
                queues[k % T].push(cur);
                k++;
                cur = next;
            }
            for (int t = 0; t < T; t++) queues[t].finish();
        });
        std::vector<std::thread> workers;
        for (int t = 0; t < T; t++) workers.emplace_back([&, t] {
            GpuWorker& w = *g_workers[t];
            ThreadConfig* config = configs[t];
            Stats* pre = config->getPreStats1();
            Stats* post = config->getPostStats1();
            FilterResult* fr = config->getFilterResult();
            std::vector<fpl_fastq_record> recs;
            std::vector<fpl_read_result> res;
            long mine = 0;
            while (TextChunk* c = queues[t].pop()) {
                const long k = (mine++) * T + t;                // this chunk's place in the writer's round-robin walk
                auto deliver = [&](string* l, string* f) {
                    delivered++;                                // counted first: `written` below never under-counts
                    if (left) left->input(t, l); else delete l;
                    if (failedW) failedW->input(t, f); else delete f;
                };
                // abandoned run: every chunk dealt out still hands the writers one (empty) string, because WriterThread::output
                // walks the worker lists strictly round-robin (src/writerthread.cpp:37-48) and would wait for a gap for ever
                auto skipChunk = [&] {
                    deliver(new string(), new string());
                    freeList.push(c);
                };
                if (notStrict) { skipChunk(); continue; }
                // writer back-pressure (the reference's reader waits the same way, src/seprocessor.cpp:391-395): chunk k
                // starts only once the single writer thread (which also compresses) is within `backlog` chunks of it.
                // The writer takes chunks in order of k, so the worker holding the chunk it needs next (k == written)
                // never waits: no cycle between the workers' waits and the writer's.
                auto written = [&](WriterThread* w) { return delivered.load() - (long)w->bufferLength(); };
                while (left && k - written(left) > backlog && !notStrict) usleep(200);
                while (failedW && k - written(failedW) > backlog && !notStrict) usleep(200);
                // four newlines per record: count them to size the record tables
                size_t nl = 0;
                for (const uint8_t* q = c->p, *e = c->p + c->n; (q = (const uint8_t*)memchr(q, '\n', (size_t)(e - q))) != nullptr; q++) nl++;
                const size_t cap = nl / 4 + 16;
                if (recs.size() < cap) { recs.resize(cap); res.resize(cap); }
                int64_t n = 0, used = 0;
                const int rc = fpl_process_fastq_host(w.ctx, c->p, (int64_t)c->n, c->last ? 1 : 0, recs.data(), res.data(),
                                                      (int64_t)cap, &n, &used);
                if (rc < 0) check(rc, "fpl_process_fastq_host");
                if (rc == 1 || (size_t)used != c->n) { notStrict = 1; skipChunk(); continue; }
                string* outstr = new string();
                string* failedOut = new string();
                const char* text = (const char*)c->p;
                // FPL_DEVICE_EMIT=1: the two output strings are assembled on the device from the chunk it still holds
                // (fpl_emit_fastq_host: first call builds and reports the sizes, second call copies); the loop below then
                // only applies the per-read side effects
                // With FPL_DEVICE_GZIP for every open writer, fpl_emit_fastq_gzip_host compresses both texts before the copy.
                const bool gzLeft = left && g_gzLeft, gzFailed = failedW && g_gzFailed;
                const bool gzEmit = deviceEmit && (gzLeft || gzFailed) && (!left || gzLeft) && (!failedW || gzFailed);
                auto emit = gzEmit ? fpl_emit_fastq_gzip_host : fpl_emit_fastq_host;
                const char* emitName = gzEmit ? "fpl_emit_fastq_gzip_host" : "fpl_emit_fastq_host";
                if (deviceEmit && n > 0) {
                    int64_t nOut = 0, nFailed = 0;
                    int erc = emit(w.ctx, failedW != NULL, NULL, 0, &nOut, NULL, 0, &nFailed);
                    if (erc < 0) check(erc, emitName);
                    outstr->resize((size_t)nOut);
                    failedOut->resize((size_t)nFailed);
                    if (nOut + nFailed > 0)
                        check(emit(w.ctx, failedW != NULL, nOut ? (uint8_t*)&(*outstr)[0] : NULL, nOut, &nOut,
                                   nFailed ? (uint8_t*)&(*failedOut)[0] : NULL, nFailed, &nFailed),
                              emitName);
                } else {
                    outstr->reserve(c->n);
                }
                ExtLists ext;
                ext.fetch(w.ctx, n > 0 && (opt->mask.enabled || opt->breakOpt.enabled));
                std::string scratch;
                for (int64_t i = 0; i < n; i++) {
                    const fpl_fastq_record& fq = recs[i];
                    ReadView v = {text + fq.name_off, (size_t)fq.name_len, text + fq.seq_off, text + fq.qual_off, fq.seq_len,
                                  text + fq.plus_off, (size_t)fq.plus_len};
                    int nregs = 0;
                    const fpl_segment* sg = ext.segsOf(res[i].n_segments);
                    const fpl_region* rg = ext.regsOf(i, nregs);
                    scatterRead(v, res[i], sg, rg, nregs, config, failedW != NULL, *outstr, *failedOut, scratch, !deviceEmit);
                }
                if ((gzLeft || gzFailed) && !(gzEmit && n > 0))
                    gzipStrings(w.ctx, {gzLeft ? outstr : NULL, gzFailed ? failedOut : NULL});
                deliver(outstr, failedOut);
                freeList.push(c);
            }
            (void)opt;
        });
        reader.join();
        for (auto& th : workers) th.join();
        fclose(fp);
        while (getenv("FPL_TIDY")) {
            // drain the free list (otherwise left to process teardown, see the note at the end of process())
            std::unique_lock<std::mutex> l(freeList.mu);
            if (freeList.q.empty()) break;
            TextChunk* c = freeList.q.front(); freeList.q.pop_front();
            l.unlock();
            cudaFreeHost(c->p);
            delete c;
        }
        if (notStrict) {
            // Somewhere inside the file the text left the strict layout (a CR, a blank line, a malformed or truncated
            // record).  What the reference does with such input depends on its reader's own buffer logic, so the whole
            // file goes through that reader: take back everything this run produced — stop the writers, truncate the
            // outputs, zero the accumulators on the devices and on the host — and start over.
            if (mOptions->verbose) loginfo("the input is not in the strict FASTQ layout: restarting with the reference reader");
            if (mLeftWriter) mLeftWriter->setInputCompleted();
            if (mFailedWriter) mFailedWriter->setInputCompleted();
            if (leftWriter) leftWriter->join();
            if (failedWriter) failedWriter->join();
            leftWriter.reset(); failedWriter.reset();
            closeOutput();
            initOutput();                                   // reopens (truncates) --out / --failed_out
            if (mLeftWriter) leftWriter.reset(new std::thread(std::bind(&SingleEndProcessor::writerTask, this, mLeftWriter)));
            if (mFailedWriter) failedWriter.reset(new std::thread(std::bind(&SingleEndProcessor::writerTask, this, mFailedWriter)));
            for (int t = 0; t < T; t++) {
                check(fpl_reset(g_workers[t]->ctx), "fpl_reset");
                check(fpl_sync(g_workers[t]->ctx), "fpl_sync");
                delete configs[t];                          // (frees its input list as well: ThreadConfig::cleanup)
                mInputLists[t] = new SingleProducerSingleConsumerList<ReadPack*>();
                configs[t] = new ThreadConfig(mOptions, t, false);
                configs[t]->setInputList(mInputLists[t]);
                initConfig(configs[t]);
            }
            rawText = false;
        }
        if (rawText) {
            if (mLeftWriter) mLeftWriter->setInputCompleted();
            if (mFailedWriter) mFailedWriter->setInputCompleted();
        }
    }
    if (!rawText) {
        std::thread reader(std::bind(&SingleEndProcessor::readerTask, this));
        std::vector<std::thread> workers;
        for (int t = 0; t < T; t++) workers.emplace_back(std::bind(&SingleEndProcessor::processorTask, this, configs[t]));
        reader.join();
        for (auto& th : workers) th.join();
    }
    if (!mOptions->split.enabled) {
        if (leftWriter) leftWriter->join();
        if (failedWriter) failedWriter->join();
    }
    FPL_STAMP("read + GPU + write");
    if (mOptions->verbose) loginfo("start to generate reports\n");

    // ---- device accumulators -> the workers' Stats / FilterResult objects (replaces what statRead / the trimmers
    //      would have added), then the reference's own merge + reporters ----
    std::vector<Stats*> preStats, postStats;
    std::vector<FilterResult*> filterResults;
    for (int t = 0; t < T; t++) {
        GpuWorker& w = *g_workers[t];
        const int64_t C = fpl_stats_cycles(w.ctx);
        std::vector<int64_t> blk((size_t)FPL_STATS_WORDS(C));
        check(fpl_stats_download(w.ctx, FPL_STATS_PRE, blk.data(), (int64_t)blk.size()), "fpl_stats_download");
        addStatsBlock(configs[t]->getPreStats1(), blk, C);
        check(fpl_stats_download(w.ctx, FPL_STATS_POST, blk.data(), (int64_t)blk.size()), "fpl_stats_download");
        addStatsBlock(configs[t]->getPostStats1(), blk, C);
        // adapter (sub)string counts: FilterResult::addAdapterTrimmed (src/filterresult.cpp:69-77)
        std::vector<int64_t> cnt((size_t)fpl_counter_words(w.ctx));
        check(fpl_counters_download(w.ctx, cnt.data(), (int64_t)cnt.size()), "fpl_counters_download");
        FilterResult* fr = configs[t]->getFilterResult();
        for (size_t a = 0; a < g_adapters.size(); a++)
            for (int side = 0; side < 2; side++)
                for (int c = 1; c <= FPL_MAX_ADAPTER_LEN && c <= (int)g_adapters[a].length(); c++) {
                    const int64_t n = cnt[FPL_CNT_FIXED + (a * 2 + side) * (FPL_MAX_ADAPTER_LEN + 1) + c];
                    if (!n) continue;
                    const std::string& ad_ = g_adapters[a];
                    fr->mAdapter[side == 0 ? ad_.substr(ad_.length() - c, c) : ad_.substr(0, c)] += n;
                }
        preStats.push_back(configs[t]->getPreStats1());
        postStats.push_back(configs[t]->getPostStats1());
        filterResults.push_back(fr);
    }
    FPL_STAMP("device accumulators -> Stats");
    Stats* finalPreStats = Stats::merge(preStats);
    finalPreStats->calcLengthHistogram();
    Stats* finalPostStats = Stats::merge(postStats);
    finalPostStats->calcLengthHistogram();
    FilterResult* finalFilterResult = FilterResult::merge(filterResults);

    cerr << "Before filtering:" << endl;
    finalPreStats->print();
    cerr << endl << "After filtering:" << endl;
    finalPostStats->print();
    cerr << endl << "Filtering result:" << endl;
    finalFilterResult->print();

    FPL_STAMP("merge + summary");
    JsonReporter jr(mOptions);
    jr.report(finalFilterResult, finalPreStats, finalPostStats);
    HtmlReporter hr(mOptions);
    hr.report(finalFilterResult, finalPreStats, finalPostStats);

    FPL_STAMP("JSON + HTML reports");
    // The process ends right after process() returns (src/main.cpp:295-305): device buffers, pinned memory and contexts
    // are left to process teardown instead of being released one by one (cudaFree / cudaFreeHost of hundreds of MB each
    // cost more than processing a small input).  FPL_TIDY=1 releases everything (leak checkers, embedding in a library).
    const bool tidy = getenv("FPL_TIDY") != nullptr;
    for (int t = 0; t < T; t++) {
        if (tidy) { fpl_destroy(g_workers[t]->ctx); g_workers[t]->ctx = nullptr; }
        delete configs[t];
    }
    FPL_STAMP("contexts + thread configs released");
    if (tidy) g_workers.clear();
    else for (auto& w : g_workers) w.release();
    delete finalPreStats;
    delete finalPostStats;
    delete finalFilterResult;
    FPL_STAMP("final Stats released");
    if (!mOptions->split.enabled) closeOutput();
    FPL_STAMP("outputs closed");
    if (timing) fprintf(stderr, "[fastplong_gpu] %-34s %8.3f s\n", "program start -> end of process()", nowSec() - g_warm.t0);
    return true;
}
