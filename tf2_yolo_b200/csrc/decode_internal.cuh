// Internal (not part of the C ABI): pieces of the decode pipeline shared with the fused
// loss+decode launch in loss.cu.
#pragma once
#include "common.cuh"
#include "head_transform.cuh"

namespace yb {

struct DecodeLaunch {
    const void* preds[YB_MAX_SCALES];
    int gh[YB_MAX_SCALES], gw[YB_MAX_SCALES], B[YB_MAX_SCALES];
    int pcf[YB_MAX_SCALES];            // values per cell
    long long cells[YB_MAX_SCALES];    // gh*gw
    long long cell_base[YB_MAX_SCALES + 1];  // prefix of cells over scales (per image)
    long long scale_base[YB_MAX_SCALES + 1]; // prefix of n_img*cells over scales
    int n_scales, C, version;
    long long n_img;
    double thr;
    // K1 tiling
    int tile_cells[YB_MAX_SCALES];
    int tile_base[YB_MAX_SCALES + 1];
    int bulk_ok[YB_MAX_SCALES];
    int stage_bytes;
};

// Work-list entry for a BOX with hits: everything the emit pass needs, no 64-bit divisions.
struct __align__(16) HotBox {
    long long out_idx;     // the cell's position in OUTPUT order (image, scale, y, x): index into offsets
    unsigned int mem_idx;  // the cell's position inside its scale tensor: img * cells + cell
    unsigned int packed;   // bits 0..3 scale, 4..9 box, 10..31 rows of the cell's earlier boxes
};
__host__ __device__ inline HotBox make_hot(long long o, unsigned mem_idx, int scale, int box, unsigned rows_before) {
    HotBox h;
    h.out_idx = o;
    h.mem_idx = mem_idx;
    h.packed = (unsigned)scale | ((unsigned)box << 4) | (rows_before << 10);
    return h;
}

// Per-image row buckets for the one-CTA-per-image decode + NMS kernel (decode_nms.cu): the
// counting pass files every (box, class) hit of image i - the values it has in registers and
// shared memory anyway - at row[i*cap + slot], slots handed out by an atomic on n[i], so the
// per-image kernel reads a few KB of compact rows instead of gathering the hot cells back from
// the head tensors.  n[i] > cap = overflow.  key orders the rows like the reference's decode:
// ((cell position in output order (scale, y, x)) * 32 + box) * 256 + class.
struct __align__(16) FusedRow {
    unsigned int key;
    float x, y, w, h, c, p;    // the head's values for the box (cell-relative x, y) and the class score
    unsigned int cell;         // scale << 28 | cell index inside the scale (y * grid_w + x)
};
struct HotBuckets {
    unsigned int* n = nullptr;   // [n_img], zero before the counting pass; nullptr = not collected
    FusedRow* row = nullptr;     // [n_img][cap]
    int cap = 0;
};
__device__ __forceinline__ unsigned fused_key(unsigned cellpos, int box, int cls) {
    return ((cellpos * 32u + (unsigned)box) << 8) | (unsigned)cls;
}

// Destinations of a counting pass (decode_count_kernel, or the fused loss kernel) and the geometry it
// needs to place a cell in decode OUTPUT order (image, scale, y, x).
struct DecodeSink {
    unsigned int* counts;                // hits per cell, OUTPUT order; may be null
    unsigned int* n_hot;
    HotBox* hot;                         // boxes with hits, the emit pass's work list; may be null
    HotBuckets buckets;                  // per-image rows for the one-CTA-per-image kernel, or off
    long long per_img;                   // cells per image over all scales
    long long cell_base[YB_MAX_SCALES];  // first cell of a scale inside an image
    long long cells[YB_MAX_SCALES];      // grid_h * grid_w
    float thr;                           // the threshold rounded to float32 (the loss kernel's heads)
};

// c * p with one rounding: the decode files are built with -fmad=false and loss.cu is not, and both
// must compare the same product against the threshold
template <typename T>
__device__ __forceinline__ T mul_rn(T a, T b);
template <>
__device__ __forceinline__ float mul_rn<float>(float a, float b) { return __fmul_rn(a, b); }
template <>
__device__ __forceinline__ double mul_rn<double>(double a, double b) { return __dmul_rn(a, b); }

// What a lane of the counting pass keeps to file its box's rows later.
struct LaneHits {
    int n;             // hits of the lane's box
    unsigned img;      // image of the lane's cell
    unsigned cellpos;  // the cell's position inside its image, OUTPUT order
    unsigned cis;      // scale << 28 | cell index inside the scale (y * grid_w + x)
    unsigned base;     // first of the n slots reserved in the image's bucket
};

// What the counting pass does with the n hits of one lane = one box (lane = cell*B + box, B lanes per
// cell) of cell g of scale s: the cell's count (by shuffle, lane of box 0) and the box's work-list entry
// where those sinks are set, and the reservation of the box's rows in its image's bucket.  Called by
// whole warps; `valid` = the lane holds a box.
__device__ __forceinline__ LaneHits decode_place_lane(const DecodeSink& K, bool valid, int n, int B, int lc, int lb,
                                                      int s, long long g) {
    LaneHits h = {n, 0u, 0u, 0u, 0u};
    int tot = 0, before = 0;
    for (int q = 0; q < B; ++q) {
        const int nq = __shfl_sync(0xffffffffu, h.n, lc * B + q);
        tot += nq;
        before += (q < lb) ? nq : 0;
    }
    if (valid) {
        const long long img = g / K.cells[s];
        const long long o = img * K.per_img + K.cell_base[s] + (g - img * K.cells[s]);
        if (lb == 0 && K.counts != nullptr) K.counts[o] = (unsigned)tot;
        if (h.n > 0 && K.hot != nullptr)
            K.hot[atomicAdd(K.n_hot, 1u)] = make_hot(o, (unsigned)g, s, lb, (unsigned)before);
        h.img = (unsigned)img;
        h.cellpos = (unsigned)(o - img * K.per_img);
        h.cis = ((unsigned)s << 28) | (unsigned)(g - img * K.cells[s]);
        // every hot lane reserves its rows now, before the caller files them: the atomics' round trips
        // overlap each other and whatever the caller does in between
        if (K.buckets.n != nullptr && h.n > 0) h.base = atomicAdd(&K.buckets.n[h.img], (unsigned)h.n);
    }
    return h;
}

// Counting pass of one lane: hits of c*p_k >= thr over the box's C class scores `prob`, then
// decode_place_lane.
template <typename T>
__device__ __forceinline__ LaneHits decode_count_lane(const DecodeSink& K, bool valid, const T* prob, T c, T thr,
                                                      int C, int B, int lc, int lb, int s, long long g) {
    int n = 0;
    if (valid) {
#pragma unroll 16
        for (int k = 0; k < C; ++k) n += (mul_rn<T>(c, prob[k]) >= thr) ? 1 : 0;
    }
    return decode_place_lane(K, valid, n, B, lc, lb, s, g);
}

// Hits of c*sigmoidf_(p_k) >= thr of the warp's boxes whose class scores are RAW logits (the from-logits
// loss kernel; c is already activated).  A box with c < thr has none, exactly: sigmoidf_ <= 1, so
// c*sigmoidf_(p) rounds to at most c, and a NaN product fails the >= test.  The few other boxes are
// served by the whole WARP, one at a time, 32 scores per step: a lane walking its own C scores would
// stall the other 31.  Returns the hits of the lane's own box; `prob_at` = offset of its scores in `tile`.
__device__ __forceinline__ int decode_hits_logits(bool valid, const float* tile, int prob_at, float c, float thr,
                                                  int C, int lane) {
    int n = 0;
    unsigned cand = __ballot_sync(0xffffffffu, valid && !(c < thr));
    while (cand) {
        const int src = __ffs(cand) - 1;
        cand &= cand - 1;
        const float* hprob = tile + __shfl_sync(0xffffffffu, prob_at, src);
        const float hc = __shfl_sync(0xffffffffu, c, src);
        int hits = 0;
        for (int k0 = 0; k0 < C; k0 += 32) {
            const int k = k0 + lane;
            const bool hit = (k < C) && (mul_rn<float>(hc, sigmoidf_(hprob[k])) >= thr);
            hits += __popc(__ballot_sync(0xffffffffu, hit));
        }
        if (lane == src) n = hits;
    }
    return n;
}

// The rows of the warp's boxes with hits into their images' buckets, the WARP serving one hot box at a
// time (32 class scores per step, ballot, lane-parallel row writes): a lane walking its own C scores
// again would stall the other 31 for C steps.  Each lane passes its box's values and the offset of its
// class scores in `tile`; only the hot lanes' are read.  kLogits: the scores are raw logits, the rows
// get sigmoidf_(p_k) - the value decode_hits_logits counted.
template <typename T, bool kLogits = false>
__device__ __forceinline__ void decode_file_rows(const HotBuckets& K, const LaneHits& h, const T* tile, int prob_at,
                                                 int lb, T x, T y, T w, T hgt, T c, T thr, int C, int lane) {
    unsigned hot = __ballot_sync(0xffffffffu, h.n > 0);
    while (hot) {
        const int src = __ffs(hot) - 1;
        hot &= hot - 1;
        const int hlb = __shfl_sync(0xffffffffu, lb, src);
        const T* hprob = tile + __shfl_sync(0xffffffffu, prob_at, src);
        const T hc = __shfl_sync(0xffffffffu, c, src);
        const T hx = __shfl_sync(0xffffffffu, x, src), hy = __shfl_sync(0xffffffffu, y, src);
        const T hw = __shfl_sync(0xffffffffu, w, src), hh = __shfl_sync(0xffffffffu, hgt, src);
        const unsigned himg = __shfl_sync(0xffffffffu, h.img, src);
        const unsigned hpos = __shfl_sync(0xffffffffu, h.cellpos, src);
        const unsigned hcis = __shfl_sync(0xffffffffu, h.cis, src);
        unsigned u = __shfl_sync(0xffffffffu, h.base, src);
        FusedRow* dst = K.row + (size_t)himg * K.cap;
        for (int k0 = 0; k0 < C; k0 += 32) {
            const int k = k0 + lane;
            const T p = (k < C) ? (kLogits ? sigmoidf_(hprob[k]) : hprob[k]) : (T)0;
            const bool hit = (k < C) && (mul_rn<T>(hc, p) >= thr);
            const unsigned m = __ballot_sync(0xffffffffu, hit);
            const unsigned at = u + __popc(m & ((1u << lane) - 1u));
            if (hit && at < (unsigned)K.cap) {
                FusedRow fr;
                fr.key = fused_key(hpos, hlb, k);
                fr.x = (float)hx; fr.y = (float)hy; fr.w = (float)hw; fr.h = (float)hh;
                fr.c = (float)hc; fr.p = (float)p;
                fr.cell = hcis;
                dst[at] = fr;
            }
            u += __popc(m);
        }
    }
}

struct DecodeWs {          // carved out of the caller's decode workspace
    unsigned int* n_hot;   // number of boxes with hits
    unsigned int* counts;  // hits per cell, OUTPUT order (image, scale, y, x)
    long long* offsets;    // exclusive scan of counts (+ total)
    HotBox* hot;           // work list of boxes with hits
    void* scan_ws;
    size_t zero_bytes;     // n_hot + scan status: cleared by one memset before the counting pass
    long long total_cells;
};

// fill L from the public parameter struct (no workspace); YB_OK / YB_E_*
int decode_fill(const void* const* preds, int64_t n_img, const yb_decode_params* p, DecodeLaunch& L);
// the sink of a counting pass over the heads of L: per-cell counts + flat work list (either may be
// null) and / or per-image buckets
DecodeSink decode_sink(const DecodeLaunch& L, unsigned int* counts, unsigned int* n_hot, HotBox* hot,
                       const HotBuckets& buckets);
// counting pass alone
int decode_count(DecodeLaunch& L, bool is_f64, const DecodeSink& K, cudaStream_t stream);
// validate + fill L and ws (no launches).  Returns YB_OK / YB_E_*.
int decode_setup(const void* const* preds, int64_t n_img, const yb_decode_params* p, void* workspace,
                 size_t workspace_bytes, DecodeLaunch& L, DecodeWs& ws);
// scan of the per-cell counts + emission of the rows (after counts / hot list are complete)
int decode_finish(const DecodeLaunch& L, const DecodeWs& ws, bool is_f64, double* rows, long long cap,
                  long long* row_offsets, cudaStream_t stream, bool status_zeroed = false);

// One-CTA-per-image decode + NMS (decode_nms.cu), split so that the fused loss kernel can do the
// counting pass: fused_prepare validates, carves the workspace, clears its control block (one
// memset) and returns the per-image buckets the counting pass must fill; fused_finish launches
// the per-image kernel.
int fused_prepare(const void* const* preds, int64_t n_img, const yb_decode_params* p, int row_cap, void* workspace,
                  size_t workspace_bytes, DecodeLaunch& D, HotBuckets& K, cudaStream_t stream, bool clear = true);
int fused_finish(const DecodeLaunch& D, int64_t n_img, int row_cap, void* workspace, double nms_threshold,
                 int iou_mode, double* out_rows, int64_t out_capacity, int64_t* out_offsets,
                 unsigned int* n_overflow, cudaStream_t stream);

}  // namespace yb
