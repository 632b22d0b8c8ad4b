#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <vector>
#include "fplgpu.h"

// Device gzip encoder (fpl_gzip_host / fpl_emit_fastq_gzip_host): every FPL_GZIP_SEGMENT-byte segment of a piece becomes one
// gzip member, compressed by one CTA into a fixed-size slot; the members are then compacted back to back.
#define FPL_GZIP_SLOT (FPL_GZIP_SEGMENT + 64)   // >= the largest member of one segment (stored form: 10 + 2 * 5 + 65536 + 8)

struct GzSeg {
    const uint8_t* src;                         // device pointer to the segment's bytes
    int32_t len;                                // 1 .. FPL_GZIP_SEGMENT
    int32_t reserved;
};

struct FplGzip {
    uint8_t* d_in = nullptr; int64_t cap_in = 0;      // fpl_gzip_host: the uploaded pieces
    GzSeg* d_segs = nullptr; int64_t cap_segs = 0;
    uint8_t* d_slots = nullptr; int64_t cap_slots = 0;
    int64_t* d_size = nullptr; int64_t cap_size = 0;  // member bytes per segment (+ one 0: the total after the scan)
    int64_t* d_off = nullptr; int64_t cap_off = 0;
    void* d_tmp = nullptr; int64_t cap_tmp = 0;
    uint8_t* d_out = nullptr; int64_t cap_out = 0;    // the members of all pieces, back to back
    std::vector<GzSeg> h_segs;
    std::vector<int64_t> h_first;                     // first segment of each piece (+ the end)
    std::vector<int64_t> h_off;
    int64_t n_segs = 0;
};

// Cuts the pieces (device pointers) into segments and uploads the table; sizes the buffers.
int fpl_gzip_plan(FplGzip* g, const uint8_t* const* piece, const int64_t* piece_bytes, int n_pieces, cudaStream_t s, char* err,
                  size_t errlen);
void fpl_gzip_deflate(FplGzip* g, cudaStream_t s);                                          // k_gzip_deflate
int fpl_gzip_offsets(FplGzip* g, cudaStream_t s, char* err, size_t errlen);                  // cub exclusive sum of the sizes
void fpl_gzip_compact(FplGzip* g, cudaStream_t s);                                          // k_gzip_compact
// Waits for the stream; out_piece_bytes[i] = compressed bytes of piece i (they sit back to back in g->d_out).
int fpl_gzip_piece_sizes(FplGzip* g, int64_t* out_piece_bytes, cudaStream_t s, char* err, size_t errlen);
int fpl_gzip_grow(void** p, int64_t* cap, int64_t need, char* err, size_t errlen);
void fpl_gzip_free(FplGzip* g);
