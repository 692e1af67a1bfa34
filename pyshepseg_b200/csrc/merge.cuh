// merge.cuh -- interface between eliminate.cu (which prepares spectra, buckets and pixel lists) and
// merge.cu (the passes themselves).
#pragma once
#include "common.cuh"

struct SmallBarrier {
    unsigned arrive;
    unsigned pad[31];
};

// words of one segment record.  Up to 16 bands: {float means[NBMAX]; uint size; uint listOffset; pad},
// 32 / 64 / 128 bytes.  17 to 64 bands (NBMAX = 64): {uint size; uint listOffset}, 8 bytes, and the
// means sit in an array of their own (MergeState::means)
template <int NBMAX>
struct MergeRecWords { static constexpr int value = NBMAX <= 4 ? 8 : (NBMAX <= 8 ? 16 : (NBMAX <= 16 ? 32 : 2)); };
// word of the size in a record (the list offset follows it)
template <int NBMAX>
struct MergeRecSizeAt { static constexpr int value = NBMAX <= 16 ? NBMAX : 0; };

struct MergeState {
    unsigned *seg;
    unsigned *segSize;                 // kept in step for the relabel that follows (0 = dead)
    unsigned *rec;                     // len records {float32 band means, size, list (first slice) offset}
    float *fsum;                       // len x nB float32 band sums (touched by merges only)
    unsigned long long colMagic;       // floor(2^40 / nCols) + 1: row of a pixel index without a division
    unsigned *pix;                     // per-segment list regions of minSegSize-1 entries, or packed lists + arena
    unsigned *mergeTo;                 // len, zeroed
    unsigned long long *pendHead;      // len, zeroed: (pass stamp << 32) | last pushed source
    unsigned *pendNext;                // len
    const unsigned *bucketStart;       // minSegSize + 1
    const unsigned *bucketList;        // initially small segments grouped by size
    unsigned *grownList;               // per size: targets that grew to exactly that size
    const unsigned long long *grownStart;   // minSegSize + 1 offsets into grownList
    unsigned *grownCount;              // minSegSize + 1, zeroed
    unsigned long long *ctr;           // counters (2 x MC_COUNT), then the SmallBarrier
    SmallBarrier *bar;                 // one per launch of the chain
    unsigned stage;                    // which launch of the chain this is (0 wide grid, 1 lean grid, 2 cluster)
    unsigned long long exitSlots;      // stop at the first size >= 2 whose candidates x lanes fit this (0: run to the end)
    int nB;
    unsigned nRows, nCols;
    int four;
    int minSegSize;
    double thr;
    // packed lists only: the list of a segment is a chain of slices; slice ch is
    // pix[rec[ch].off, + sliceLen[ch]) and is followed by slice nextChunk[ch] (SSG_NIL: the end)
    unsigned *sliceLen;                // len
    unsigned *nextChunk;               // len
    unsigned *tailChunk;               // len: last slice of a live segment's chain
    unsigned long long *arenaUsed;     // zeroed: arena entries handed out (or asked for, past the end)
    unsigned arenaBase, arenaCap;      // the arena: pix[arenaBase, arenaBase + arenaCap)
    // 17 to 64 bands only: len x nBP float32 means, rows padded with zeros to nBP (a multiple of 4)
    float *means;
    int nBP;
};

struct MergePlan {
    const float *fsum;          // len x nB float32 band sums (buildSegmentSpectra)
    const unsigned *sliceOff;   // len: list offset (region or first slice) of every segment
    int64_t len;
    bool packed;                // lists are packed slices rather than regions
};

size_t ssgk_merge_rec_bytes(int nB, int64_t len);
size_t ssgk_merge_ctr_bytes(void);
int ssgk_merge(ssg_ctx *ctx, MergeState &st, const MergePlan &plan, uint32_t *numPasses, int64_t *numElim);
