// Head decode: threshold c*p_k per (cell, box, class) and emit float64 rows
// [x, y, w, h, c, class, p] in the reference's order (utils/tools.py:370-438),
// batched over images and scales.
//
//   K1 decode_count : one warp per cell reads the cell's scores once (coalesced),
//                     counts hits with warp ballots, stores the count at the
//                     cell's position in OUTPUT order (image, scale, y, x).
//   scan            : exclusive prefix of the per-cell counts -> row offset per cell.
//   K2 decode_emit  : warps skip empty cells (32 counts per load, one ballot) and
//                     re-evaluate only cells with hits, writing rows in (box, class)
//                     order at the scanned offset.
//
// The comparison runs in the INPUT dtype (fp32 product, threshold rounded to fp32
// for fp32 heads), the row arithmetic in fp64 with one rounding per operation
// (this file is compiled with -fmad=false).
#include <cstring>

#include "common.cuh"
#include "decode_internal.cuh"
#include "scan.cuh"

namespace yb {

// K1: persistent CTAs; a producer warp streams tiles of cells through a shared-memory
// ring with 1-D bulk-async copies (TMA), consumer warps own whole cells (lane = cell*B + box),
// each lane walks the C class scores of its box (lanes are an odd number of words apart ->
// conflict-free), per-cell counts by shuffle.  Cells with hits are appended to a work list.
constexpr int kDecMaxConsumerWarps = 8;
constexpr int kDecStages = 3;

template <typename T, bool kBuckets>
__global__ void __launch_bounds__((kDecMaxConsumerWarps + 1) * 32)
decode_count_kernel(const __grid_constant__ DecodeLaunch L, const __grid_constant__ DecodeSink K) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t full[kDecStages], done[kDecStages];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ncw = (int)(blockDim.x >> 5) - 1;
    if (tid == 0) {
        for (int i = 0; i < kDecStages; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&done[i], ncw * 32);
        }
        mbar_fence_init();
    }
    __syncthreads();
    const int total_tiles = L.tile_base[L.n_scales];
    const int n_my = (total_tiles > (int)blockIdx.x)
                         ? (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x
                         : 0;
    const T thr = (T)L.thr;

    if (warp == ncw) {  // ---- producer ----
        int s = 0;
        for (int t = 0; t < n_my; ++t) {
            const int tile = blockIdx.x + t * gridDim.x;
            while (tile >= L.tile_base[s + 1]) ++s;
            const long long cell0 = (long long)(tile - L.tile_base[s]) * L.tile_cells[s];
            const long long n_cells = L.n_img * L.cells[s];
            const int nc = (int)min((long long)L.tile_cells[s], n_cells - cell0);
            const int stage = t % kDecStages;
            if (t >= kDecStages) mbar_wait(&done[stage], ((t / kDecStages) - 1) & 1);
            T* dst = reinterpret_cast<T*>(smem + (size_t)stage * L.stage_bytes);
            const T* src = reinterpret_cast<const T*>(L.preds[s]) + cell0 * L.pcf[s];
            const uint32_t bytes = (uint32_t)nc * L.pcf[s] * (uint32_t)sizeof(T);
            if (L.bulk_ok[s] && (bytes & 15u) == 0u) {
                if (lane == 0) {
                    mbar_arrive_expect_tx(&full[stage], bytes);
                    bulk_g2s(dst, src, bytes, &full[stage]);
                }
            } else {
                for (int i = lane; i < nc * L.pcf[s]; i += 32) dst[i] = src[i];
                __syncwarp();
                if (lane == 0) mbar_arrive(&full[stage]);
            }
        }
    } else {            // ---- consumers ----
        int s = 0, cur = -1, cpw = 0, lc = 0, lb = 0;
        bool lane_on = false;
        for (int it = 0; it < n_my; ++it) {
            const int tile = blockIdx.x + it * gridDim.x;
            while (tile >= L.tile_base[s + 1]) ++s;
            if (s != cur) {
                cur = s;
                cpw = 32 / L.B[s];
                lc = lane / L.B[s];
                lb = lane - lc * L.B[s];
                lane_on = lc < cpw;
            }
            const int B = L.B[s], C = L.C, pcf = L.pcf[s];
            const long long cell0 = (long long)(tile - L.tile_base[s]) * L.tile_cells[s];
            const long long n_cells = L.n_img * L.cells[s];
            const int nc = (int)min((long long)L.tile_cells[s], n_cells - cell0);
            const int stage = it % kDecStages;
            const T* sp = reinterpret_cast<const T*>(smem + (size_t)stage * L.stage_bytes);
            mbar_wait(&full[stage], (it / kDecStages) & 1);
            for (int c0 = warp * cpw; c0 < nc; c0 += ncw * cpw) {
                const int cell = c0 + lc;
                const bool valid = lane_on && cell < nc;
                const int box_at = cell * pcf + lb * ((L.version == 1) ? 5 : 5 + C);
                const int prob_at = (L.version == 1) ? cell * pcf + 5 * B : box_at + 5;
                const T c = valid ? sp[box_at + 4] : (T)0;
                const LaneHits h = decode_count_lane<T>(K, valid, sp + prob_at, c, thr, C, B, lc, lb, s, cell0 + cell);
                if (kBuckets) {
                    T x = 0, y = 0, w = 0, hgt = 0;
                    if (h.n > 0) {
                        x = sp[box_at]; y = sp[box_at + 1]; w = sp[box_at + 2]; hgt = sp[box_at + 3];
                    }
                    decode_file_rows<T>(K.buckets, h, sp, prob_at, lb, x, y, w, hgt, c, thr, C, lane);
                }
            }
            mbar_arrive(&done[stage]);
        }
    }
}

// K2: eight lanes per box that has hits (work list from K1): the lanes take contiguous slices of
// the box's C class scores (one coalesced read of the box, independent loads), count their hits,
// prefix-sum across the group and write the rows, in class order, at
// offsets[cell] + rows of the cell's earlier boxes.
constexpr int kEmitGroup = 8;

template <typename T>
__global__ void __launch_bounds__(256)
decode_emit_kernel(const __grid_constant__ DecodeLaunch L, const unsigned int* __restrict__ n_hot,
                   const HotBox* __restrict__ hot_boxes, const long long* __restrict__ offsets,
                   double* __restrict__ rows, long long cap, long long* __restrict__ row_offsets) {
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n_threads = (long long)gridDim.x * blockDim.x;
    const long long per_img = L.cell_base[L.n_scales];
    const T thr = (T)L.thr;
    for (long long i = tid; i <= L.n_img; i += n_threads) row_offsets[i] = offsets[i * per_img];
    const long long n = *n_hot;
    const int sub = threadIdx.x & (kEmitGroup - 1);
    const long long n_groups = n_threads / kEmitGroup;
    // whole warps iterate together (uniform trip count) so the group shuffles stay converged
    const long long rounds = (n + n_groups - 1) / n_groups;
    for (long long it = 0; it < rounds; ++it) {
        const long long w = it * n_groups + tid / kEmitGroup;
        const bool live = w < n;
        HotBox hb = make_hot(0, 0, 0, 0, 0);
        if (live) hb = hot_boxes[w];
        const int s = (int)(hb.packed & 15u), b = (int)((hb.packed >> 4) & 63u);
        const int C = L.C, B = L.B[s];
        const T* cptr = reinterpret_cast<const T*>(L.preds[s]) + (size_t)hb.mem_idx * L.pcf[s];
        const T* box = cptr + b * ((L.version == 1) ? 5 : 5 + C);
        const T* prob = (L.version == 1) ? cptr + 5 * B : box + 5;
        const int per = (C + kEmitGroup - 1) / kEmitGroup;
        const int k0 = sub * per, k1 = min(C, k0 + per);
        T c = 0;
        long long r = 0;
        if (live) {
            c = box[4];
            r = offsets[hb.out_idx] + (long long)(hb.packed >> 10);
        }
        int cnt = 0;
        if (live)
            for (int k = k0; k < k1; ++k) cnt += (mul_rn<T>(c, prob[k]) >= thr) ? 1 : 0;
        // exclusive prefix of cnt over the lanes of the group
        int inc = cnt;
#pragma unroll
        for (int o = 1; o < kEmitGroup; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, inc, o, kEmitGroup);
            if (sub >= o) inc += v;
        }
        const int ex = inc - cnt;
        if (live && cnt > 0) {
            const unsigned cell = hb.mem_idx % (unsigned)L.cells[s];  // position inside the image
            const int yi = (int)(cell / (unsigned)L.gw[s]), xi = (int)(cell - (unsigned)yi * (unsigned)L.gw[s]);
            const double bx = ((double)xi + (double)box[0]) / (double)L.gw[s];
            const double by = ((double)yi + (double)box[1]) / (double)L.gh[s];
            const double bw = (double)box[2], bh = (double)box[3], bc = (double)c;
            r += ex;
            for (int k = k0; k < k1; ++k) {
                const T p = prob[k];
                if (mul_rn<T>(c, p) >= thr) {
                    if (r < cap) {
                        double* o = rows + r * 7;
                        o[0] = bx; o[1] = by; o[2] = bw; o[3] = bh; o[4] = bc;
                        o[5] = (double)k;
                        o[6] = (double)p;
                    }
                    ++r;
                }
            }
        }
    }
}

int decode_fill(const void* const* preds, int64_t n_img, const yb_decode_params* p, DecodeLaunch& L) {
    if (preds == nullptr || p == nullptr) return YB_E_NULL;
    if (p->version < 1 || p->version > 4) return YB_E_PARAM;
    if (p->n_scales < 1 || p->n_scales > YB_MAX_SCALES || p->class_num <= 0 || n_img < 0) return YB_E_SHAPE;
    memset(&L, 0, sizeof(L));
    L.n_scales = p->n_scales;
    L.C = p->class_num;
    L.version = p->version;
    L.n_img = n_img;
    L.thr = p->threshold;
    const size_t esz = p->is_f64 ? 8 : 4;
    for (int s = 0; s < p->n_scales; ++s) {
        if (preds[s] == nullptr) return YB_E_NULL;
        if ((uintptr_t)preds[s] & (esz - 1)) return YB_E_ALIGN;
        if (p->grid_h[s] <= 0 || p->grid_w[s] <= 0 || p->bbox_num[s] <= 0 || p->bbox_num[s] > 32)
            return YB_E_SHAPE;
        L.preds[s] = preds[s];
        L.gh[s] = p->grid_h[s];
        L.gw[s] = p->grid_w[s];
        L.B[s] = p->bbox_num[s];
        L.pcf[s] = (p->version == 1) ? 5 * p->bbox_num[s] + p->class_num
                                     : p->bbox_num[s] * (5 + p->class_num);
        L.cells[s] = (long long)p->grid_h[s] * p->grid_w[s];
        L.cell_base[s + 1] = L.cell_base[s] + L.cells[s];
        L.scale_base[s + 1] = L.scale_base[s] + n_img * L.cells[s];
    }
    return YB_OK;
}

DecodeSink decode_sink(const DecodeLaunch& L, unsigned int* counts, unsigned int* n_hot, HotBox* hot,
                       const HotBuckets& buckets) {
    DecodeSink K{counts, n_hot, hot, buckets, L.cell_base[L.n_scales], {}, {}, (float)L.thr};
    for (int s = 0; s < L.n_scales; ++s) {
        K.cell_base[s] = L.cell_base[s];
        K.cells[s] = L.cells[s];
    }
    return K;
}

// K1 geometry (3 stages of <= 24 KB, 3 CTAs per SM) + launch
int decode_count(DecodeLaunch& L, bool is_f64, const DecodeSink& K, cudaStream_t stream) {
    const size_t esz = is_f64 ? 8 : 4;
    const int stage_budget = 24 * 1024;
    int ncw = 1, stage_bytes = 0;
    for (int s = 0; s < L.n_scales; ++s) {
        const int cb = (int)(L.pcf[s] * esz);
        if (4 * cb > 72 * 1024) return YB_E_SHAPE;
        const int cpw = 32 / L.B[s];
        int t = stage_budget / cb / 4 * 4;
        t = min(t, kDecMaxConsumerWarps * cpw / 4 * 4);
        t = max(4, t);
        L.tile_cells[s] = t;
        L.tile_base[s + 1] = L.tile_base[s] + (int)((L.n_img * L.cells[s] + t - 1) / t);
        L.bulk_ok[s] = (((uintptr_t)L.preds[s] & 15) == 0) ? 1 : 0;
        stage_bytes = max(stage_bytes, (int)align_up((size_t)t * cb, 128));
        ncw = max(ncw, min(kDecMaxConsumerWarps, (t + cpw - 1) / cpw));
    }
    const int n_tiles = L.tile_base[L.n_scales];
    L.stage_bytes = stage_bytes;
    const size_t smem = (size_t)kDecStages * stage_bytes;
    const int ctas_per_sm = max(1, min(4, (int)((227 * 1024) / (smem + 2048))));
    const int grid = max(1, min(n_tiles, kNumSMs * ctas_per_sm));
    const int threads1 = (ncw + 1) * 32;
    if (is_f64) {
        if (K.buckets.n != nullptr) return YB_E_PARAM;   // row buckets hold the float32 head values
        static SmemRaised done;
        YB_CUDA_TRY(raise_dynamic_smem_once(decode_count_kernel<double, false>, (int)smem, &done));
        decode_count_kernel<double, false><<<grid, threads1, smem, stream>>>(L, K);
    } else if (K.buckets.n != nullptr) {
        static SmemRaised done;
        YB_CUDA_TRY(raise_dynamic_smem_once(decode_count_kernel<float, true>, (int)smem, &done));
        decode_count_kernel<float, true><<<grid, threads1, smem, stream>>>(L, K);
    } else {
        static SmemRaised done;
        YB_CUDA_TRY(raise_dynamic_smem_once(decode_count_kernel<float, false>, (int)smem, &done));
        decode_count_kernel<float, false><<<grid, threads1, smem, stream>>>(L, K);
    }
    YB_CUDA_TRY(cudaGetLastError());
    return YB_OK;
}

}  // namespace yb

using namespace yb;

static size_t decode_counts_bytes(long long total_cells) {
    return align_up((size_t)(total_cells + 1) * sizeof(unsigned int), 256);
}
static size_t decode_offsets_bytes(long long total_cells) {
    return align_up((size_t)(total_cells + 2) * sizeof(long long), 256);
}
static size_t decode_hot_bytes(long long total_boxes) {
    return align_up((size_t)(total_boxes + 1) * sizeof(HotBox), 256);
}

extern "C" size_t yb_decode_workspace_bytes(const yb_decode_params* p, int64_t n_img) {
    if (p == nullptr || n_img < 0) return 0;
    long long per_img = 0, boxes_per_img = 0;
    for (int s = 0; s < p->n_scales && s < YB_MAX_SCALES; ++s) {
        per_img += (long long)p->grid_h[s] * p->grid_w[s];
        boxes_per_img += (long long)p->grid_h[s] * p->grid_w[s] * (p->bbox_num[s] > 0 ? p->bbox_num[s] : 1);
    }
    const long long total = per_img * n_img;
    return 256 + decode_counts_bytes(total) + decode_offsets_bytes(total) + decode_hot_bytes(boxes_per_img * n_img) +
           scan_workspace_bytes(total > 0 ? total : 1);
}

namespace yb {

int decode_setup(const void* const* preds, int64_t n_img, const yb_decode_params* p, void* workspace,
                 size_t workspace_bytes, DecodeLaunch& L, DecodeWs& ws) {
    int rc = decode_fill(preds, n_img, p, L);
    if (rc != YB_OK) return rc;
    if (workspace == nullptr) return YB_E_NULL;
    if (workspace_bytes < yb_decode_workspace_bytes(p, n_img) || ((uintptr_t)workspace & 255))
        return YB_E_WORKSPACE;
    const long long total = L.n_img * L.cell_base[L.n_scales];
    for (int s = 0; s < L.n_scales; ++s)
        if (L.n_img * L.cells[s] > 0xffffffffll || L.B[s] > 32 || (long long)L.B[s] * L.C >= (1 << 22))
            return YB_E_SHAPE;  // HotBox packs the cell index in 32 bits, box in 6, row offset in 22
    ws.total_cells = total;
    // [n_hot | scan status] first: ONE memset clears both before the counting pass
    ws.n_hot = reinterpret_cast<unsigned int*>(workspace);
    ws.scan_ws = (char*)workspace + 256;
    ws.zero_bytes = 256 + scan_workspace_bytes(total > 0 ? total : 1);
    ws.counts = reinterpret_cast<unsigned int*>((char*)workspace + ws.zero_bytes);
    ws.offsets = reinterpret_cast<long long*>((char*)ws.counts + decode_counts_bytes(total));
    long long total_boxes = 0;
    for (int s = 0; s < L.n_scales; ++s) total_boxes += L.n_img * L.cells[s] * L.B[s];
    ws.hot = reinterpret_cast<HotBox*>((char*)ws.offsets + decode_offsets_bytes(total));
    (void)total_boxes;
    return YB_OK;
}

int decode_finish(const DecodeLaunch& L, const DecodeWs& ws, bool is_f64, double* rows, long long cap,
                  long long* row_offsets, cudaStream_t stream, bool status_zeroed) {
    int rc = exclusive_scan_u32(ws.counts, ws.total_cells, ws.offsets, ws.scan_ws, stream, status_zeroed);
    if (rc != 0) return rc;
    const int threads = 256;
    const int blocks2 = kNumSMs * 5;   // one wave (48 registers: 5 CTAs of 256 threads per SM)
    if (is_f64)
        decode_emit_kernel<double><<<blocks2, threads, 0, stream>>>(L, ws.n_hot, ws.hot, ws.offsets, rows, cap,
                                                                    row_offsets);
    else
        decode_emit_kernel<float><<<blocks2, threads, 0, stream>>>(L, ws.n_hot, ws.hot, ws.offsets, rows, cap,
                                                                   row_offsets);
    YB_CUDA_TRY(cudaGetLastError());
    return YB_OK;
}

}  // namespace yb

extern "C" int yb_decode(const void* const* preds, int64_t n_img, const yb_decode_params* p, double* rows,
                         int64_t row_capacity, int64_t* row_offsets, void* workspace,
                         size_t workspace_bytes, yb_stream_t stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    if (row_offsets == nullptr) return YB_E_NULL;
    if (rows == nullptr && row_capacity > 0) return YB_E_NULL;
    if (row_capacity < 0) return YB_E_CAPACITY;
    DecodeLaunch L;
    DecodeWs ws;
    int rc = decode_setup(preds, n_img, p, workspace, workspace_bytes, L, ws);
    if (rc != YB_OK) return rc;
    if (ws.total_cells == 0) {
        YB_CUDA_TRY(cudaMemsetAsync(row_offsets, 0, sizeof(int64_t) * (n_img + 1), stream));
        return YB_OK;
    }
    YB_CUDA_TRY(cudaMemsetAsync(ws.n_hot, 0, ws.zero_bytes, stream));
    rc = decode_count(L, p->is_f64 != 0, decode_sink(L, ws.counts, ws.n_hot, ws.hot, HotBuckets{}), stream);
    if (rc != YB_OK) return rc;
    return decode_finish(L, ws, p->is_f64 != 0, rows, row_capacity, reinterpret_cast<long long*>(row_offsets), stream, true);
}

// Second half of a split decode: the per-cell counts and the hot-cell list are already in
// `workspace` (left there by yb_loss_decode_fused called with row_offsets == NULL).
extern "C" int yb_decode_finish(const void* const* preds, int64_t n_img, const yb_decode_params* p, double* rows,
                                int64_t row_capacity, int64_t* row_offsets, void* workspace,
                                size_t workspace_bytes, yb_stream_t stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    if (row_offsets == nullptr) return YB_E_NULL;
    if (rows == nullptr && row_capacity > 0) return YB_E_NULL;
    if (row_capacity < 0) return YB_E_CAPACITY;
    DecodeLaunch L;
    DecodeWs ws;
    int rc = decode_setup(preds, n_img, p, workspace, workspace_bytes, L, ws);
    if (rc != YB_OK) return rc;
    if (ws.total_cells == 0) {
        YB_CUDA_TRY(cudaMemsetAsync(row_offsets, 0, sizeof(int64_t) * (n_img + 1), stream));
        return YB_OK;
    }
    return decode_finish(L, ws, p->is_f64 != 0, rows, row_capacity, reinterpret_cast<long long*>(row_offsets), stream);
}
