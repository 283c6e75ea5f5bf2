// Fused YOLO grid loss: forward + gradient in one pass over the head tensors.
//
// Replaces the TensorFlow op chains of
//   yolov4/losses/loss.py:10-61,64-169   yolov3/losses/loss.py:9-37,40-164
//   yolov2/losses/loss.py:9-37,40-137    yolov1_5/losses/loss.py:9-37,40-118
// with one persistent, warp-specialised kernel per launch (all FPN scales):
//
//   producer warp : 1-D bulk-async (TMA) loads of a tile of cells (y_pred + y_true)
//                   into a shared-memory ring, bulk-async store of the same
//                   buffer -- by then overwritten in place with dL/dy_pred -- back
//                   to HBM.
//   consumer warps: a warp owns whole cells, one lane per (cell, box): fp32 IoU against
//                   the label box, argmax over the B boxes by shuffle -> responsible /
//                   ignore masks, box + objectness + wh terms and their 5 gradients
//                   written in place, zero-fill of the box's class-score gradients;
//                   the rare responsible boxes then get their class cross-entropy and
//                   gradient from the whole warp (fp64).  No CTA-wide barrier.
//   scheduling    : tiles are handed out by a global ticket counter (the first tile of a
//                   CTA is its block index), so SMs that stream faster take more tiles
//                   and every CTA finishes within one tile of the others.
//   reduction     : every addend is split onto two fixed binary grids (2^-12 and 2^-42)
//                   before it is accumulated, so all additions are exact and the sums do
//                   not depend on which CTA took which tile: thread -> warp -> CTA ->
//                   fp64 atomics in global memory stay bit-reproducible; the last CTA
//                   combines the two grids and emits the fp32 loss of every scale.
//
// The loss is cell-local; the only coupling is the argmax over the boxes of one
// cell and the final sum, so HBM traffic is exactly: read y_pred, read y_true,
// write dpred, once each.
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "decode_internal.cuh"

namespace yb {

constexpr int kLossMaxConsumerWarps = 8;
constexpr int kLossMaxThreads = (kLossMaxConsumerWarps + 1) * 32;
constexpr int kMaxStages = 4;
constexpr int kTerms = 10;     // 5 loss terms + 5 in-training metric sums
constexpr int kLossTerms = 5;
constexpr float kEpsF = 1e-07f;
constexpr double kEps = 1e-07;
constexpr int kCtrlWords = 4;  // [0] finished CTAs, [1] tile tickets

// Order-independent accumulation.  x is rounded onto the grid 2^-12 (adding 1.5*2^40 makes the
// ulp of the sum 2^-12), the exact remainder onto 2^-42; what is left (< 2^-43 per addend) is
// dropped.  Sums of grid points are exact while |sum| < 2^41 resp. 2^11 (more than 16 M addends
// per term), so they are associative: any schedule gives the same bits.  Beyond those bounds the
// additions round like ordinary fp64 sums.  NaN / Inf propagate.
constexpr double kBinHi = 1649267441664.0;  // 1.5 * 2^40
constexpr double kBinLo = 1536.0;           // 1.5 * 2^10
__device__ __forceinline__ void bin_add(double& hi, double& lo, double x) {
    const double h = __dsub_rn(__dadd_rn(x, kBinHi), kBinHi);
    const double r = (h == x) ? 0.0 : __dsub_rn(x, h);
    const double l = __dsub_rn(__dadd_rn(r, kBinLo), kBinLo);
    hi = __dadd_rn(hi, h);
    lo = __dadd_rn(lo, l);
}

struct LossScaleDev {
    const float* y_true;
    const float* y_pred;
    float* dpred;
    long long n_cells;
    int tile_cells;  // cells per tile (multiple of 4)
    int n_tiles;
    int tile_base;   // first tile id of this scale in the launch-wide tile list
    int pcf, tcf;    // floats per cell in y_pred / y_true
    int bulk_ok;     // all three base pointers 16-byte aligned
    int B, C;
    float gw, gh;
    float anc[2 * YB_MAX_BOXES];
    float bw;
    float lw[4];
    float whw;
    float ignore_thr, truth_thr, label_smooth, gamma;
    int use_focal, use_scale;
    float inv_n;
    float recall_thr;       // IoU threshold of the recall metric
    double term_w[kLossTerms];  // weights combining the raw terms into the loss
    double inv_n_d;
};

struct LossLaunch {
    LossScaleDev sc[YB_MAX_SCALES];
    int n_scales;
    int total_tiles;
    int stage_bytes;       // bytes of one ring stage
    int n_stages;
    double* gacc;          // [n_scales][kAcc][2] order-independent sums (zero on entry, re-zeroed on exit)
    unsigned int* ctrl;    // [kCtrlWords]
    float* loss_out;       // [n_scales]
    double* terms_out;     // [n_scales][YB_LOSS_TERMS] or null
    double* metrics_out;   // [n_scales][YB_LOSS_METRICS] or null
    int from_logits;       // all scales: y_pred holds raw head outputs
    DecodeSink dec;        // the decode counting pass riding on the kernel (kDecode)
};

// ---- box geometry ------------------------------------------------------------

// fp32 IoU with one rounding per operation, in the reference's operation order
// (loss.py:14-38) so that masks match a TensorFlow fp32 evaluation.
__device__ __forceinline__ float grid_iou_f32(float px, float py, float pw, float ph, float tx,
                                              float ty, float tw, float th, float gw, float gh) {
    const float pcx = __fdiv_rn(px, gw), pcy = __fdiv_rn(py, gh);
    const float tcx = __fdiv_rn(tx, gw), tcy = __fdiv_rn(ty, gh);
    const float phw = __fmul_rn(pw, 0.5f), phh = __fmul_rn(ph, 0.5f);
    const float thw = __fmul_rn(tw, 0.5f), thh = __fmul_rn(th, 0.5f);
    const float ix0 = fmaxf(__fsub_rn(pcx, phw), __fsub_rn(tcx, thw));
    const float iy0 = fmaxf(__fsub_rn(pcy, phh), __fsub_rn(tcy, thh));
    const float ix1 = fminf(__fadd_rn(pcx, phw), __fadd_rn(tcx, thw));
    const float iy1 = fminf(__fadd_rn(pcy, phh), __fadd_rn(tcy, thh));
    const float iw = fmaxf(__fsub_rn(ix1, ix0), 0.f);
    const float ih = fmaxf(__fsub_rn(iy1, iy0), 0.f);
    const float inter = __fmul_rn(iw, ih);
    const float uni = __fsub_rn(__fadd_rn(__fmul_rn(pw, ph), __fmul_rn(tw, th)), inter);
    return __fdiv_rn(inter, __fadd_rn(uni, kEpsF));
}

// IoU / CIoU and their derivatives w.r.t. the predicted (x, y, w, h), fp64.
// Selection rules follow TensorFlow's Maximum/Minimum gradients (first operand
// = the predicted box wins ties; max(.,0) passes the gradient at 0).
struct BoxGrad {
    double iou, ciou;
    double diou[4], dciou[4];
};

template <bool kCiou>
__device__ __forceinline__ void box_fwd_bwd(double x, double y, double w, double h, double X,
                                            double Y, double W, double H, double gw, double gh,
                                            BoxGrad& o) {
    const double pcx = x / gw, pcy = y / gh, tcx = X / gw, tcy = Y / gh;
    const double p0x = pcx - w / 2.0, p1x = pcx + w / 2.0, p0y = pcy - h / 2.0, p1y = pcy + h / 2.0;
    const double t0x = tcx - W / 2.0, t1x = tcx + W / 2.0, t0y = tcy - H / 2.0, t1y = tcy + H / 2.0;
    // intersection
    const double a0x = (p0x >= t0x) ? 1.0 : 0.0, a1x = (p1x <= t1x) ? 1.0 : 0.0;
    const double a0y = (p0y >= t0y) ? 1.0 : 0.0, a1y = (p1y <= t1y) ? 1.0 : 0.0;
    const double rx = fmin(p1x, t1x) - fmax(p0x, t0x), ry = fmin(p1y, t1y) - fmax(p0y, t0y);
    const double gx0 = (rx >= 0.0) ? 1.0 : 0.0, gy0 = (ry >= 0.0) ? 1.0 : 0.0;
    const double iw = fmax(rx, 0.0), ih = fmax(ry, 0.0);
    const double inter = iw * ih;
    const double uni = w * h + W * H - inter;
    const double den = uni + kEps;
    const double iou = inter / den;
    // d(iw)/dx, d(iw)/dw ; d(ih)/dy, d(ih)/dh
    const double diw_dx = gx0 * (a1x - a0x) / gw, diw_dw = gx0 * (a1x + a0x) * 0.5;
    const double dih_dy = gy0 * (a1y - a0y) / gh, dih_dh = gy0 * (a1y + a0y) * 0.5;
    const double dI[4] = {ih * diw_dx, iw * dih_dy, ih * diw_dw, iw * dih_dh};
    const double dU[4] = {-dI[0], -dI[1], h - dI[2], w - dI[3]};
    const double inv_den2 = 1.0 / (den * den);
#pragma unroll
    for (int k = 0; k < 4; ++k) o.diou[k] = (dI[k] * den - inter * dU[k]) * inv_den2;
    o.iou = iou;
    if (!kCiou) return;
    // enclosing box diagonal
    const double b0x = (p0x <= t0x) ? 1.0 : 0.0, b1x = (p1x >= t1x) ? 1.0 : 0.0;
    const double b0y = (p0y <= t0y) ? 1.0 : 0.0, b1y = (p1y >= t1y) ? 1.0 : 0.0;
    const double ew = fmax(p1x, t1x) - fmin(p0x, t0x), eh = fmax(p1y, t1y) - fmin(p0y, t0y);
    const double c2 = ew * ew + eh * eh;
    const double dc2[4] = {2.0 * ew * (b1x - b0x) / gw, 2.0 * eh * (b1y - b0y) / gh,
                           2.0 * ew * (b1x + b0x) * 0.5, 2.0 * eh * (b1y + b0y) * 0.5};
    const double ddx = tcx - pcx, ddy = tcy - pcy;
    const double rho2 = ddx * ddx + ddy * ddy;
    const double drho2[4] = {-2.0 * ddx / gw, -2.0 * ddy / gh, 0.0, 0.0};
    // aspect-ratio term, alpha is differentiated (loss.py:51-57)
    const double hh = h + kEps;
    const double at = atan(W / (H + kEps)), ap = atan(w / hh);
    const double kk = 4.0 / (3.14159265358979323846 * 3.14159265358979323846);
    const double da = at - ap;
    const double v = kk * da * da;
    const double r2 = hh * hh + w * w;
    const double dv[4] = {0.0, 0.0, -2.0 * kk * da * (hh / r2), 2.0 * kk * da * (w / r2)};
    const double D = 1.0 - iou + v;
    const double av = v * v / D;  // alpha * v
    o.ciou = iou - rho2 / c2 - av;
    const double inv_c4 = 1.0 / (c2 * c2), inv_D2 = 1.0 / (D * D);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const double dR = (drho2[k] * c2 - rho2 * dc2[k]) * inv_c4;
        const double dav = (2.0 * v * dv[k] * D - v * v * (dv[k] - o.diou[k])) * inv_D2;
        o.dciou[k] = o.diou[k] - dR - dav;
    }
}

// focal-style term f(e) = -e^g * log(1-e) and its derivative.
__device__ __forceinline__ void focal_term(float e, float g, float& f, float& df) {
    const float l = logf(1.f - e);
    float eg, eg1;
    if (g == 2.f) {
        eg = e * e;
        eg1 = e;
    } else if (g == 1.f) {
        eg = e;
        eg1 = 1.f;
    } else if (g == 0.f) {
        eg = 1.f;
        eg1 = 0.f;
    } else {
        eg1 = powf(e, g - 1.f);
        eg = eg1 * e;
    }
    f = -eg * l;
    df = -g * eg1 * l + eg / (1.f - e);
}

// ---- the kernel --------------------------------------------------------------
//
// Thread mapping of the consumer warps: a warp owns whole cells, lane = cell_local*B + box
// (32/B cells per warp, the last 32 % B lanes idle), so the argmax over the boxes of a cell is
// a handful of shuffles and the consumer warps never synchronise with each other - only with
// the producer, through the full/done mbarriers of the stage.

template <int V, bool kLogits>
__device__ __forceinline__ void class_row(float* q, const float* t, float m, int C, int lane, bool write,
                                          double lwc, double& part) {
    // cross-entropy over the C class scores of one responsible box (v2-v4) / object cell (v1)
    for (int k = lane; k < C; k += 32) {
        const double p = kLogits ? 1.0 / (1.0 + exp(-(double)q[k])) : (double)q[k];
        const double tk = (double)t[k];
        const double pc = fmin(fmax(p, kEps), 1.0 - kEps);
        const double band = (p >= kEps && p <= 1.0 - kEps) ? 1.0 : 0.0;
        double l, g;
        if (V == 1 || V == 2) {  // positive-only CE (yolov2/losses/loss.py:116-124, v1 :101-109)
            l = tk * log(pc);
            g = -tk / pc;
        } else {                 // BCE (yolov4/losses/loss.py:145-154)
            l = tk * log(pc) + (1.0 - tk) * log(1.0 - pc);
            g = -(tk / pc - (1.0 - tk) / (1.0 - pc));
        }
        part -= (double)m * l;
        if (write) q[k] = (float)(lwc * (double)m * g * band * (kLogits ? p * (1.0 - p) : 1.0));
    }
}

// first-index argmax of C floats by one warp (tf.argmax semantics)
__device__ __forceinline__ int warp_argmax(const float* v, int C, int lane) {
    float best = -INFINITY;
    int arg = 0x7fffffff;
    for (int k = lane; k < C; k += 32) {
        const float x = v[k];
        if (x > best || arg == 0x7fffffff) {
            best = x;
            arg = k;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
        if (oa != 0x7fffffff && (arg == 0x7fffffff || ob > best || (ob == best && oa < arg))) {
            best = ob;
            arg = oa;
        }
    }
    return arg;
}

#ifdef YB_LOSS_PROFILE
__device__ unsigned long long yb_loss_prof[1024 * 6];
__device__ __forceinline__ unsigned long long gtimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
#define YB_PROF(slot) do { yb_loss_prof[blockIdx.x * 6 + (slot)] = gtimer(); } while (0)
#else
#define YB_PROF(slot) do { } while (0)
#endif

template <int V, bool kMetrics, bool kDecode, bool kLogits = false>
__global__ void __launch_bounds__(kLossMaxThreads)
loss_fwd_bwd_kernel(const __grid_constant__ LossLaunch L) {
    constexpr int kAcc = kMetrics ? kTerms : kLossTerms;  // per-thread accumulators
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int n_stages = L.n_stages;
    const int ncw = (int)(blockDim.x >> 5) - 1;  // consumer warps; the last warp is the producer

    unsigned char* ring = smem;
    double* s_acc = reinterpret_cast<double*>(smem + (size_t)n_stages * L.stage_bytes);
    // s_acc: [ncw][n_scales][kTerms][2]
    const int n_sc = L.n_scales;
    uint64_t* full = reinterpret_cast<uint64_t*>(s_acc + ncw * n_sc * kTerms * 2);
    uint64_t* done = full + kMaxStages;
    __shared__ int s_is_last;
    __shared__ int s_tile[kMaxStages];  // tile held by each ring stage, -1 = no more work

    if (tid == 0) {
        for (int i = 0; i < kMaxStages; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&done[i], ncw * 32);
        }
        mbar_fence_init();
    }
    for (int i = tid; i < ncw * n_sc * kTerms * 2; i += blockDim.x) s_acc[i] = 0.0;
    __syncthreads();
    if (tid == 0) YB_PROF(0);

    const int total_tiles = L.total_tiles;

    if (warp == ncw) {
        // ===================== producer warp =====================
        // Iteration t fills ring stage t % n_stages with the next tile (or posts the end marker)
        // and then retires tile t-(n_stages-1): waits for the consumers, stores the stage (now
        // holding dL/dy_pred) back, and waits until the store has read shared memory, which
        // frees that stage for iteration t+1.
        int s_ld = 0, s_st = 0;
        int next = ((int)blockIdx.x < total_tiles) ? (int)blockIdx.x : -1;  // lane 0's view
        int n_loaded = 0;
        bool end_posted = false;
        for (int t = 0;; ++t) {
            const int stage = t % n_stages;
            const int tile = __shfl_sync(0xffffffffu, next, 0);
            if (tile >= 0) {
                while (tile >= L.sc[s_ld].tile_base + L.sc[s_ld].n_tiles) ++s_ld;
                const LossScaleDev& S = L.sc[s_ld];
                const long long cell0 = (long long)(tile - S.tile_base) * S.tile_cells;
                const int nc = (int)min((long long)S.tile_cells, S.n_cells - cell0);
                float* sp = reinterpret_cast<float*>(ring + (size_t)stage * L.stage_bytes);
                float* st = sp + S.tile_cells * S.pcf;
                const float* gp = S.y_pred + cell0 * S.pcf;
                const float* gt = S.y_true + cell0 * S.tcf;
                if (S.bulk_ok && (nc & 3) == 0) {
                    if (lane == 0) {
                        const uint32_t bp = (uint32_t)nc * S.pcf * 4u, bt = (uint32_t)nc * S.tcf * 4u;
                        s_tile[stage] = tile;
                        mbar_arrive_expect_tx(&full[stage], bp + bt);
                        bulk_g2s(sp, gp, bp, &full[stage]);
                        bulk_g2s(st, gt, bt, &full[stage]);
                    }
                } else {  // ragged tail / unaligned tensors: plain loads
                    for (int i = lane; i < nc * S.pcf; i += 32) sp[i] = __ldg(gp + i);
                    for (int i = lane; i < nc * S.tcf; i += 32) st[i] = __ldg(gt + i);
                    __syncwarp();
                    if (lane == 0) {
                        s_tile[stage] = tile;
                        mbar_arrive(&full[stage]);
                    }
                }
                ++n_loaded;
                // ticket for the next tile; the atomic's latency overlaps the retire step below
                if (lane == 0) {
                    const unsigned tk = atomicAdd(&L.ctrl[1], 1u) + gridDim.x;
                    next = (tk < (unsigned)total_tiles) ? (int)tk : -1;
                }
            } else if (!end_posted) {
                if (lane == 0) {
                    s_tile[stage] = -1;
                    mbar_arrive(&full[stage]);
                }
                end_posted = true;
            }
            const int j = t - (n_stages - 1);
            if (j >= 0 && j < n_loaded) {
                const int jstage = j % n_stages;
                mbar_wait(&done[jstage], (j / n_stages) & 1);
                const int jt = s_tile[jstage];
                while (jt >= L.sc[s_st].tile_base + L.sc[s_st].n_tiles) ++s_st;
                const LossScaleDev& S = L.sc[s_st];
                if (S.dpred != nullptr) {
                    const long long cell0 = (long long)(jt - S.tile_base) * S.tile_cells;
                    const int nc = (int)min((long long)S.tile_cells, S.n_cells - cell0);
                    float* sp = reinterpret_cast<float*>(ring + (size_t)jstage * L.stage_bytes);
                    float* gd = S.dpred + cell0 * S.pcf;
                    if (S.bulk_ok && (nc & 3) == 0) {
                        if (lane == 0) {
                            bulk_s2g(gd, sp, (uint32_t)nc * S.pcf * 4u);
                            bulk_commit();
                            bulk_wait_read<0>();
                        }
                    } else {
                        for (int i = lane; i < nc * S.pcf; i += 32) gd[i] = sp[i];
                    }
                    __syncwarp();
                }
            }
            if (end_posted && j >= n_loaded - 1) break;
        }
        if (lane == 0) YB_PROF(2);
        if (lane == 0) bulk_wait_all<0>();
        if (lane == 0) YB_PROF(3);
    } else {
        // ===================== consumer warps =====================
        double hi[kAcc], lo[kAcc];
#pragma unroll
        for (int k = 0; k < kAcc; ++k) hi[k] = lo[k] = 0.0;
        auto add = [&](int k, double v) { bin_add(hi[k], lo[k], v); };
        int cur = -1;
        int cpw = 0, lc = 0, lb = 0;  // cells per warp, this lane's local cell / box
        bool lane_on = false;
        float aw = 1.f, ah = 1.f;
        auto flush = [&](int s) {
#pragma unroll
            for (int k = 0; k < kAcc; ++k) {
                const double vh = warp_sum(hi[k]), vl = warp_sum(lo[k]);   // exact: grid points
                if (lane == 0) {
                    double* a = s_acc + ((warp * n_sc + s) * kTerms + k) * 2;
                    a[0] += vh;
                    a[1] += vl;
                }
                hi[k] = lo[k] = 0.0;
            }
        };

        for (int it = 0;; ++it) {
            const int stage = it % n_stages;
            mbar_wait(&full[stage], (it / n_stages) & 1);
            const int tile = s_tile[stage];
            if (tile < 0) break;
            int s = (cur < 0) ? 0 : cur;
            while (tile >= L.sc[s].tile_base + L.sc[s].n_tiles) ++s;
            if (s != cur) {
                if (cur >= 0) flush(cur);
                cur = s;
                const int Bs = L.sc[s].B;
                cpw = 32 / Bs;
                lc = lane / Bs;
                lb = lane - lc * Bs;
                lane_on = lc < cpw;
                aw = L.sc[s].anc[2 * (lane_on ? lb : 0)];
                ah = L.sc[s].anc[2 * (lane_on ? lb : 0) + 1];
            }
            const LossScaleDev& S = L.sc[s];
            const long long cell0 = (long long)(tile - S.tile_base) * S.tile_cells;
            const int nc = (int)min((long long)S.tile_cells, S.n_cells - cell0);
            float* sp = reinterpret_cast<float*>(ring + (size_t)stage * L.stage_bytes);
            const float* st = sp + S.tile_cells * S.pcf;
            const int B = S.B, C = S.C;
            const int bstride = (V == 1) ? 5 : (5 + C);
            const bool write = S.dpred != nullptr;
            const float inv_n = S.inv_n;

            for (int c0 = warp * cpw; c0 < nc; c0 += ncw * cpw) {
                const int cell = c0 + lc;
                const bool valid = lane_on && cell < nc;
                float* pc = sp + (valid ? cell : c0) * S.pcf + lb * bstride;
                const float* tc = st + (valid ? cell : c0) * S.tcf;
                float px = 0.f, py = 0.f, pw = 1.f, ph = 1.f, c = 0.5f;
                float tx = 0.f, ty = 0.f, tw = 0.f, th = 0.f, obj = 0.f;
                if (valid) {
                    px = pc[0]; py = pc[1]; pw = pc[2]; ph = pc[3]; c = pc[4];
                    tx = tc[0]; ty = tc[1]; tw = tc[2]; th = tc[3]; obj = tc[4];
                    if (kLogits) {  // head transform: sigmoid offsets / objectness, anchor * exp sizes
                        px = head_act(px, 0, aw); py = head_act(py, 1, ah); c = head_act(c, 4, aw);
                        pw = head_act(pw, 2, aw); ph = head_act(ph, 3, ah);
                    }
                }
                const float iou = grid_iou_f32(px, py, pw, ph, tx, ty, tw, th, S.gw, S.gh);
                // argmax over the boxes of the cell (first maximum, like tf.argmax)
                int amax = 0;
                float best = __shfl_sync(0xffffffffu, iou, lc * B);
                for (int q = 1; q < B; ++q) {
                    const float v = __shfl_sync(0xffffffffu, iou, lc * B + q);
                    if (v > best) {
                        best = v;
                        amax = q;
                    }
                }
                const float resp = (lb == amax) ? 1.f : 0.f;
                // head decode, counting pass (utils/tools.py:411-412), on the tile that is already in
                // shared memory.  It reserves the rows of a hot box in its image's bucket NOW; they are
                // filed after the loss arithmetic below, which hides the atomic's round trip to L2.
                // Both must precede the in-place gradient writes.
                const int prob_at = cell * S.pcf + ((V == 1) ? 5 * B : lb * bstride + 5);   // the box's class scores
                // Raw-logit heads: the scores are activated on the fly (c already is), the warp serving the
                // few boxes that pass the exact prefilter c >= thr.
                LaneHits dec = {0, 0u, 0u, 0u, 0u};
                if constexpr (kDecode && kLogits)
                    dec = decode_place_lane(L.dec, valid, decode_hits_logits(valid, sp, prob_at, c, L.dec.thr, C, lane),
                                            B, lc, lb, s, cell0 + cell);
                else if (kDecode)
                    dec = decode_count_lane<float>(L.dec, valid, sp + prob_at, c, L.dec.thr, C, B, lc, lb, s,
                                                   cell0 + cell);
                if (kMetrics) {
                    // In-training metrics of yolov*/metrics/yolo_metrics.py folded into this pass (they
                    // read the same tensors): objectness accuracy, mean best IoU, class accuracy, recall.
                    float cmax = __shfl_sync(0xffffffffu, c, lc * B);
                    for (int q = 1; q < B; ++q) cmax = fmaxf(cmax, __shfl_sync(0xffffffffu, c, lc * B + q));
                    if (valid && lb == 0) {
                        add(kAcc - 5, (obj == ((cmax > 0.5f) ? 1.f : 0.f)) ? 1.0 : 0.0);
                        add(kAcc - 4, (double)(best * obj));
                        add(kAcc - 3, (double)obj);
                    }
                    float eq = 0.f;  // argmax(class scores) agrees with the label's class
                    unsigned om = __ballot_sync(0xffffffffu, valid && obj != 0.f && (V != 1 || lb == 0));
                    while (om) {
                        const int src = __ffs(om) - 1;
                        om &= om - 1;
                        const int rc = __shfl_sync(0xffffffffu, cell, src);
                        const int rb = __shfl_sync(0xffffffffu, lb, src);
                        const float* q = (V == 1) ? sp + rc * S.pcf + 5 * B : sp + rc * S.pcf + rb * bstride + 5;
                        const int ap = warp_argmax(q, C, lane);
                        const int at = warp_argmax(st + rc * S.tcf + 5, C, lane);
                        if (lane == src) eq = (ap == at) ? 1.f : 0.f;
                    }
                    if (V == 1) eq = __shfl_sync(0xffffffffu, eq, lc * B);  // per-cell class scores
                    if (valid && (V != 1 || lb == 0)) add(kAcc - 2, (double)(eq * obj));
                    float hit = iou * (eq * obj);
                    float hmax = __shfl_sync(0xffffffffu, hit, lc * B);
                    for (int q = 1; q < B; ++q) hmax = fmaxf(hmax, __shfl_sync(0xffffffffu, hit, lc * B + q));
                    if (valid && lb == 0) add(kAcc - 1, (hmax >= S.recall_thr) ? 1.0 : 0.0);
                }
                float g0 = 0.f, g1 = 0.f, g2 = 0.f, g3 = 0.f, g4 = 0.f;
                float pos = 0.f;
                if (valid) {
                    if (V == 1) {
                        pos = obj * resp;
                        const float neg = 1.f - pos;
                        const float dx = tx - px, dy = ty - py;
                        add(0, (double)(pos * (dx * dx + dy * dy)));
                        g0 = -2.f * S.lw[0] * pos * dx * inv_n;
                        g1 = -2.f * S.lw[0] * pos * dy * inv_n;
                        const float sw = sqrtf(fmaxf(pw, kEpsF)), sh = sqrtf(fmaxf(ph, kEpsF));
                        const float dw = sqrtf(fmaxf(tw, kEpsF)) - sw, dh = sqrtf(fmaxf(th, kEpsF)) - sh;
                        add(1, (double)(pos * (dw * dw + dh * dh)));
                        g2 = (pw >= kEpsF) ? -S.lw[1] * pos * dw / sw * inv_n : 0.f;
                        g3 = (ph >= kEpsF) ? -S.lw[1] * pos * dh / sh * inv_n : 0.f;
                        if (pos != 0.f) {  // objectness regresses to the IoU, which carries gradient
                            BoxGrad bg;
                            box_fwd_bwd<false>(px, py, pw, ph, tx, ty, tw, th, S.gw, S.gh, bg);
                            const double d = bg.iou - (double)c;
                            add(2, (double)pos * d * d + (double)(S.bw * neg * c * c));
                            const double gi = 2.0 * S.lw[2] * pos * d * S.inv_n_d;
                            g0 += (float)(gi * bg.diou[0]);
                            g1 += (float)(gi * bg.diou[1]);
                            g2 += (float)(gi * bg.diou[2]);
                            g3 += (float)(gi * bg.diou[3]);
                            g4 = (float)(-gi) + 2.f * S.lw[2] * S.bw * neg * c * inv_n;
                        } else {
                            add(2, (double)(S.bw * neg * c * c));
                            g4 = 2.f * S.lw[2] * S.bw * neg * c * inv_n;
                        }
                    } else {
                        pos = obj * resp;
                        if (V == 4 && S.truth_thr < 1.f)
                            pos = pos + ((iou > S.truth_thr) ? 1.f : 0.f) * (1.f - pos);
                        const float neg = (1.f - pos) * ((iou < S.ignore_thr) ? 1.f : 0.f);
                        const float lpw = logf(pw / aw), lph = logf(ph / ah);
                        if (V == 4) {
                            // wh regulariser, every box (loss.py:156-160)
                            add(3, (double)(lpw * lpw + lph * lph));
                            g2 = 2.f * S.whw * lpw / pw * inv_n;
                            g3 = 2.f * S.whw * lph / ph * inv_n;
                            // focal objectness with label smoothing (loss.py:119-143)
                            const float cc = fminf(fmaxf(c, kEpsF), 1.f - kEpsF);
                            const float band = (c >= kEpsF && c <= 1.f - kEpsF) ? 1.f : 0.f;
                            float e_p, e_n, de_p, de_n;
                            if (S.label_smooth > 0.f) {
                                const float u = 1.f - S.label_smooth - cc, w2 = S.label_smooth - cc;
                                e_p = fabsf(u);
                                de_p = (u > 0.f) ? -1.f : ((u < 0.f) ? 1.f : 0.f);
                                e_n = fabsf(w2);
                                de_n = (w2 > 0.f) ? -1.f : ((w2 < 0.f) ? 1.f : 0.f);
                            } else {
                                e_p = 1.f - cc;
                                de_p = -1.f;
                                e_n = cc;
                                de_n = 1.f;
                            }
                            float fn, dfn;
                            focal_term(e_n, S.gamma, fn, dfn);
                            float lcf = S.bw * neg * fn;
                            float gc = S.bw * neg * dfn * de_n;
                            if (pos != 0.f) {
                                float fp, dfp;
                                focal_term(e_p, S.gamma, fp, dfp);
                                lcf += pos * fp;
                                gc += pos * dfp * de_p;
                                // CIoU box term (loss.py:113-117)
                                BoxGrad bg;
                                box_fwd_bwd<true>(px, py, pw, ph, tx, ty, tw, th, S.gw, S.gh, bg);
                                add(0, (double)pos * (1.0 - bg.ciou));
                                const double gb = -(double)S.lw[0] * pos * S.inv_n_d;
                                g0 += (float)(gb * bg.dciou[0]);
                                g1 += (float)(gb * bg.dciou[1]);
                                g2 += (float)(gb * bg.dciou[2]);
                                g3 += (float)(gb * bg.dciou[3]);
                            }
                            add(1, (double)lcf);
                            g4 = S.lw[1] * gc * band * inv_n;
                        } else {  // V == 2 or 3
                            add(4, (double)(lpw * lpw + lph * lph));
                            g2 = 2.f * S.whw * lpw / pw * inv_n;
                            g3 = 2.f * S.whw * lph / ph * inv_n;
                            if (pos != 0.f) {
                                const float sc = S.use_scale ? (2.f - tw * th) : 1.f;
                                const float dx = tx - px, dy = ty - py;
                                add(0, (double)(pos * sc * (dx * dx + dy * dy)));
                                g0 = -2.f * S.lw[0] * pos * sc * dx * inv_n;
                                g1 = -2.f * S.lw[0] * pos * sc * dy * inv_n;
                                const float dlw = logf(fmaxf(tw / aw, kEpsF)) - lpw;
                                const float dlh = logf(fmaxf(th / ah, kEpsF)) - lph;
                                add(1, (double)(pos * sc * (dlw * dlw + dlh * dlh)));
                                g2 += -2.f * S.lw[1] * pos * sc * dlw / pw * inv_n;
                                g3 += -2.f * S.lw[1] * pos * sc * dlh / ph * inv_n;
                            }
                            if (V == 3 && S.use_focal) {
                                const float cc = fminf(fmaxf(c, kEpsF), 1.f - kEpsF);
                                const float band = (c >= kEpsF && c <= 1.f - kEpsF) ? 1.f : 0.f;
                                float fn, dfn;
                                focal_term(cc, S.gamma, fn, dfn);
                                float lcf = S.bw * neg * fn, gc = S.bw * neg * dfn;
                                if (pos != 0.f) {
                                    float fp, dfp;
                                    focal_term(1.f - cc, S.gamma, fp, dfp);
                                    lcf += pos * fp;
                                    gc -= pos * dfp;
                                }
                                add(2, (double)lcf);
                                g4 = S.lw[2] * gc * band * inv_n;
                            } else {
                                const float om = 1.f - c;
                                add(2, (double)(pos * om * om + S.bw * neg * c * c));
                                g4 = S.lw[2] * (-2.f * pos * om + 2.f * S.bw * neg * c) * inv_n;
                            }
                        }
                    }
                    if (kLogits) {  // chain rule through the head transform
                        g0 *= px * (1.f - px); g1 *= py * (1.f - py); g4 *= c * (1.f - c);
                        g2 *= pw; g3 *= ph;
                    }
                }
                if (kDecode && L.dec.buckets.n != nullptr)   // before the gradients overwrite the tile
                    decode_file_rows<float, kLogits>(L.dec.buckets, dec, sp, prob_at, lb, px, py, pw, ph, c, L.dec.thr, C,
                                                     lane);
                if (valid) {
                    if (write) {
                        pc[0] = g0; pc[1] = g1; pc[2] = g2; pc[3] = g3; pc[4] = g4;
                        // class scores of a non-responsible box get exactly zero gradient;
                        // lanes are 85 (odd) floats apart -> bank-conflict-free stores
                        if (V != 1 && pos == 0.f) {
                            float* q = pc + 5;
                            for (int k = 0; k < C; ++k) q[k] = 0.f;
                        }
                        if (V == 1 && lb == 0 && obj == 0.f) {
                            float* q = sp + cell * S.pcf + 5 * B;
                            for (int k = 0; k < C; ++k) q[k] = 0.f;
                        }
                    }
                }
                // class term of the (rare) responsible boxes: the whole warp takes one row at a time
                const float rowm = (V == 1) ? ((lb == 0) ? obj : 0.f) : pos;
                unsigned pm = __ballot_sync(0xffffffffu, valid && rowm != 0.f);
                while (pm) {
                    const int src = __ffs(pm) - 1;
                    pm &= pm - 1;
                    const int rc = __shfl_sync(0xffffffffu, cell, src);
                    const int rb = __shfl_sync(0xffffffffu, lb, src);
                    const float m = __shfl_sync(0xffffffffu, rowm, src);
                    float* q = (V == 1) ? sp + rc * S.pcf + 5 * B : sp + rc * S.pcf + rb * bstride + 5;
                    const float* t = st + rc * S.tcf + 5;
                    double part = 0.0;
                    class_row<V, kLogits>(q, t, m, C, lane, write, (double)S.lw[(V == 4) ? 2 : 3] * S.inv_n_d, part);
                    add((V == 4) ? 2 : 3, part);
                }
            }
            fence_proxy_async();
            mbar_arrive(&done[stage]);
        }
        if (cur >= 0) flush(cur);
        if (tid == 0) YB_PROF(1);
    }

    // ---- CTA sums -> global (exact, order-independent adds), last CTA finishes -------
    __syncthreads();
    const int n_vals = L.n_scales * kAcc * 2;
    for (int i = tid; i < n_vals; i += (int)blockDim.x) {
        const int s = i / (kAcc * 2), r = i - s * (kAcc * 2);
        double v = 0.0;
        for (int w = 0; w < ncw; ++w) v += s_acc[(w * n_sc + s) * kTerms * 2 + r];
        if (v != 0.0) atomicAdd(&L.gacc[i], v);
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_is_last = (atomicAdd(&L.ctrl[0], 1u) == gridDim.x - 1);
    __syncthreads();
    if (tid == 0) YB_PROF(4);
    if (!s_is_last) return;
    __threadfence();
    double* s_fin = s_acc;  // reuse: [n_scales][kTerms]
    for (int i = tid; i < L.n_scales * kAcc; i += (int)blockDim.x) {
        const int s = i / kAcc, k = i - s * kAcc;
        const double vh = __ldcg(&L.gacc[2 * i]), vl = __ldcg(&L.gacc[2 * i + 1]);
        L.gacc[2 * i] = 0.0;      // leave the workspace reusable
        L.gacc[2 * i + 1] = 0.0;
        s_fin[s * kTerms + k] = vh + vl;
    }
    __syncthreads();
    if (tid < L.n_scales) {
        const LossScaleDev& S = L.sc[tid];
        double total = 0.0;
        for (int k = 0; k < kLossTerms; ++k) total += S.term_w[k] * s_fin[tid * kTerms + k];
        total *= S.inv_n_d;
        L.loss_out[tid] = (float)total;
        if (L.terms_out != nullptr) {
            double* o = L.terms_out + tid * YB_LOSS_TERMS;
            o[0] = total;
            for (int k = 0; k < kLossTerms; ++k) o[1 + k] = s_fin[tid * kTerms + k] * S.inv_n_d;
            o[6] = 0.0;
            o[7] = 0.0;
        }
        if (L.metrics_out != nullptr) {
            const double* m = s_fin + tid * kTerms + kLossTerms;  // hits, sum best-IoU, sum obj, sum equal, tp
            double* o = L.metrics_out + tid * YB_LOSS_METRICS;
            const double cells = (double)S.n_cells;
            const double eps = 1e-07;
            o[0] = cells > 0 ? m[0] / cells : 0.0;                      // obj_acc
            o[1] = m[1] / (m[2] + eps);                                // mean_iou
            o[2] = m[3] / (m[2] * ((V == 1) ? 1.0 : (double)S.B) + eps);  // class_acc
            o[3] = m[4] / (m[2] + eps);                                // recall
            for (int k = 0; k < 5; ++k) o[4 + k] = m[k];               // raw sums (for sharded batches)
            o[9] = cells;
        }
    }
    if (tid == 0) {
        L.ctrl[0] = 0u;
        L.ctrl[1] = 0u;
    }
    if (tid == 0) YB_PROF(5);
}

// ---- grid IoU (public cal_iou of the loss modules) ----------------------------
__global__ void grid_iou_kernel(const float* __restrict__ bt, int ts, const float* __restrict__ bp,
                                int ps, long long n_boxes, int B, float gw, float gh,
                                float* __restrict__ iou_out, float* __restrict__ ciou_out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_boxes) return;
    const long long cell = i / B;
    const float* t = bt + cell * ts;
    const float* p = bp + i * ps;
    const float iou = grid_iou_f32(p[0], p[1], p[2], p[3], t[0], t[1], t[2], t[3], gw, gh);
    iou_out[i] = iou;
    if (ciou_out != nullptr) {
        BoxGrad bg;
        box_fwd_bwd<true>(p[0], p[1], p[2], p[3], t[0], t[1], t[2], t[3], gw, gh, bg);
        ciou_out[i] = (float)bg.ciou;
    }
}

// ---- head transform of raw heads (yb_activate_head) ----------------------------
// Elementwise over the flattened (n_cells, B, 5+C) head, kW floats per access (4: 16-byte aligned
// tensors).  A thread keeps the (box, value) position of its first float and advances it by the
// grid stride (adv_b boxes + adv_j values) instead of dividing per element.  out may alias raw.
struct HeadAnchors {
    float a[2 * YB_MAX_BOXES];
};

template <int kW>
__global__ void __launch_bounds__(256) activate_head_kernel(const float* raw, float* out, long long n_items,
                                                            int n_tail, int bs, int B, int adv_b, int adv_j,
                                                            const __grid_constant__ HeadAnchors anc) {
    __shared__ float s_anc[2 * YB_MAX_BOXES];
    if (threadIdx.x < 2 * YB_MAX_BOXES) s_anc[threadIdx.x] = anc.a[threadIdx.x];
    __syncthreads();
    const long long cell_floats = (long long)B * bs;
    const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const int r = (int)((i0 * kW) % cell_floats);
    int b = r / bs, j = r - b * bs;
    for (long long i = i0; i < n_items; i += stride) {
        float v[kW];
        if constexpr (kW == 4) {
            const float4 q = reinterpret_cast<const float4*>(raw)[i];
            v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
        } else {
            v[0] = raw[i];
        }
#pragma unroll
        for (int t = 0; t < kW; ++t) {
            int jt = j + t, bt = b;
            if (jt >= bs) {   // bs = 5 + C > 4: at most one box boundary inside an access
                jt -= bs;
                if (++bt == B) bt = 0;
            }
            v[t] = head_act(v[t], jt, s_anc[2 * bt + (jt == 3 ? 1 : 0)]);
        }
        if constexpr (kW == 4) {
            reinterpret_cast<float4*>(out)[i] = make_float4(v[0], v[1], v[2], v[3]);
        } else {
            out[i] = v[0];
        }
        j += adv_j;
        b += adv_b;
        if (j >= bs) {
            j -= bs;
            ++b;
        }
        if (b >= B) b -= B;
    }
    // the n_tail (< kW) floats after the last full access
    if (blockIdx.x == 0 && (int)threadIdx.x < n_tail) {
        const long long e = n_items * kW + threadIdx.x;
        const int re = (int)(e % cell_floats), be = re / bs, je = re - be * bs;
        out[e] = head_act(raw[e], je, s_anc[2 * be + (je == 3 ? 1 : 0)]);
    }
}

// ---- host side ----------------------------------------------------------------

// Tuning knobs (YB_LOSS_STAGES, YB_LOSS_CTAS_PER_SM, YB_LOSS_TILE_CELLS, YB_LOSS_WARPS): read from the environment
// ONCE per process (function-local statics, thread-safe), not on every launch.
struct LossEnv {
    int stages, ctas_per_sm, tile_cells, warps;
    static int get(const char* name, int dflt) {
        const char* v = getenv(name);
        return (v && *v) ? atoi(v) : dflt;
    }
    LossEnv() : stages(get("YB_LOSS_STAGES", 2)), ctas_per_sm(get("YB_LOSS_CTAS_PER_SM", 4)),
                tile_cells(get("YB_LOSS_TILE_CELLS", 0)), warps(get("YB_LOSS_WARPS", 0)) {}
};
static const LossEnv& loss_env() {
    static const LossEnv e;
    return e;
}

static size_t loss_gacc_bytes(int n_scales) {
    return align_up((size_t)n_scales * kTerms * 2 * sizeof(double), 256);
}

static int fill_scale(const yb_loss_scale& in, LossScaleDev& d) {
    const yb_loss_params& p = in.p;
    if (in.y_true == nullptr || in.y_pred == nullptr) return YB_E_NULL;
    if (p.version < 1 || p.version > 4) return YB_E_PARAM;
    if (p.grid_h <= 0 || p.grid_w <= 0 || p.bbox_num <= 0 || p.bbox_num > YB_MAX_BOXES ||
        p.class_num <= 0 || in.n_cells < 0)
        return YB_E_SHAPE;
    if (((uintptr_t)in.y_true | (uintptr_t)in.y_pred | (uintptr_t)in.dpred) & 3) return YB_E_ALIGN;
    d.y_true = in.y_true;
    d.y_pred = in.y_pred;
    d.dpred = in.dpred;
    d.n_cells = in.n_cells;
    d.B = p.bbox_num;
    d.C = p.class_num;
    d.tcf = 5 + p.class_num;
    d.pcf = (p.version == 1) ? 5 * p.bbox_num + p.class_num : p.bbox_num * (5 + p.class_num);
    d.bulk_ok = ((((uintptr_t)in.y_true | (uintptr_t)in.y_pred | (uintptr_t)in.dpred) & 15) == 0) ? 1 : 0;
    d.gw = (float)p.grid_w;
    d.gh = (float)p.grid_h;
    for (int i = 0; i < 2 * YB_MAX_BOXES; ++i)
        d.anc[i] = (p.has_anchors && i < 2 * p.bbox_num) ? p.anchors[i] : 1.f;
    d.bw = p.binary_weight;
    for (int i = 0; i < 4; ++i) d.lw[i] = p.loss_weight[i];
    d.ignore_thr = p.ignore_thresh;
    d.truth_thr = p.truth_thresh;
    d.label_smooth = p.label_smooth;
    d.gamma = p.focal_gamma;
    d.use_focal = p.use_focal;
    d.use_scale = (p.version == 2) ? 1 : p.use_scale;
    d.inv_n = (float)p.inv_batch;
    d.inv_n_d = p.inv_batch;
    for (int k = 0; k < kLossTerms; ++k) d.term_w[k] = 0.0;
    d.recall_thr = 0.5f;
    if (p.version == 4) {
        d.whw = p.wh_reg_weight;
        d.term_w[0] = p.loss_weight[0];
        d.term_w[1] = p.loss_weight[1];
        d.term_w[2] = p.loss_weight[2];
        d.term_w[3] = p.wh_reg_weight;
    } else {
        d.whw = (p.version == 1) ? 0.f : 0.01f;
        for (int k = 0; k < 4; ++k) d.term_w[k] = p.loss_weight[k];
        d.term_w[4] = (p.version == 1) ? 0.0 : 0.01;
    }
    return YB_OK;
}

template <int V, bool kMetrics, bool kDecode>
static int launch_loss_variant(const LossLaunch& L, int grid, int threads, size_t smem, cudaStream_t stream) {
    static SmemRaised done;   // per template instance
    YB_CUDA_TRY(raise_dynamic_smem_once(loss_fwd_bwd_kernel<V, kMetrics, kDecode>, (int)smem, &done));
    loss_fwd_bwd_kernel<V, kMetrics, kDecode><<<grid, threads, smem, stream>>>(L);
    YB_CUDA_TRY(cudaGetLastError());
    return YB_OK;
}

template <int V, bool kMetrics, bool kDecode>
static int launch_loss_logits(const LossLaunch& L, int grid, int threads, size_t smem, cudaStream_t stream) {
    static SmemRaised done;
    YB_CUDA_TRY(raise_dynamic_smem_once(loss_fwd_bwd_kernel<V, kMetrics, kDecode, true>, (int)smem, &done));
    loss_fwd_bwd_kernel<V, kMetrics, kDecode, true><<<grid, threads, smem, stream>>>(L);
    YB_CUDA_TRY(cudaGetLastError());
    return YB_OK;
}

// d: the launch carries a counting pass.  From logits, that is only the per-image buckets of the
// two-launch step (step_impl): the other counting passes are followed by an emit pass that re-reads
// the head tensors (yb_loss_decode_fused rejects raw heads before it gets here), and metrics do not
// ride on the step.
template <int V>
static int launch_loss(const LossLaunch& L, bool d, int grid, int threads, size_t smem, cudaStream_t stream) {
    const bool m = L.metrics_out != nullptr;
    if (L.from_logits) {
        if (V != 3 && V != 4) return YB_E_PARAM;  // v1/v2 heads end in a softmax
        if (V == 3 || V == 4) {
            constexpr int W = (V == 3 || V == 4) ? V : 4;
            if (d) return launch_loss_logits<W, false, true>(L, grid, threads, smem, stream);
            return m ? launch_loss_logits<W, true, false>(L, grid, threads, smem, stream)
                     : launch_loss_logits<W, false, false>(L, grid, threads, smem, stream);
        }
    }
    if (m && d) return launch_loss_variant<V, true, true>(L, grid, threads, smem, stream);
    if (m) return launch_loss_variant<V, true, false>(L, grid, threads, smem, stream);
    if (d) return launch_loss_variant<V, false, true>(L, grid, threads, smem, stream);
    return launch_loss_variant<V, false, false>(L, grid, threads, smem, stream);
}

}  // namespace yb

using namespace yb;

#ifdef YB_LOSS_PROFILE
extern "C" int yb_debug_loss_profile(unsigned long long* host_out) {
    return (int)cudaMemcpyFromSymbol(host_out, yb::yb_loss_prof, sizeof(unsigned long long) * 1024 * 6);
}
#endif

extern "C" size_t yb_loss_workspace_bytes(int n_scales) {
    if (n_scales < 1) n_scales = 1;
    if (n_scales > YB_MAX_SCALES) n_scales = YB_MAX_SCALES;
    return loss_gacc_bytes(n_scales) + 256;
}

// dec: optional, count decode hits inside the loss pass
static int loss_impl(const yb_loss_scale* scales, int n_scales, float* loss_out, double* terms_out,
                     double* metrics_out, double recall_iou_threshold, void* workspace,
                     size_t workspace_bytes, yb_stream_t stream_, const DecodeSink* dec = nullptr,
                     bool workspace_is_clean = false) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    if (scales == nullptr || loss_out == nullptr || workspace == nullptr) return YB_E_NULL;
    if (n_scales < 1 || n_scales > YB_MAX_SCALES) return YB_E_SHAPE;
    if (workspace_bytes < yb_loss_workspace_bytes(n_scales) || ((uintptr_t)workspace & 255))
        return YB_E_WORKSPACE;

    LossLaunch L;
    memset(&L, 0, sizeof(L));
    L.n_scales = n_scales;
    const int version = scales[0].p.version;
    L.from_logits = scales[0].p.from_logits ? 1 : 0;
    int cell_bytes_max = 0;
    for (int s = 0; s < n_scales; ++s) {
        if (scales[s].p.version != version) return YB_E_PARAM;
        if ((scales[s].p.from_logits ? 1 : 0) != L.from_logits) return YB_E_PARAM;
        int rc = fill_scale(scales[s], L.sc[s]);
        if (rc != YB_OK) return rc;
        cell_bytes_max = max(cell_bytes_max, (L.sc[s].pcf + L.sc[s].tcf) * 4);
    }

    // Ring geometry: by default 2 stages and 4 CTAs per SM (for v3/v4 cells: 20 cells = 27.2 KB per
    // stage, two consumer warps of 10 cells); fat cells get fewer CTAs per SM.  An SM has 228 KB of
    // shared memory, every resident CTA costs its static + dynamic bytes + 1 KB.
    int n_stages = loss_env().stages;
    n_stages = max(2, min(kMaxStages, n_stages));
    int ctas_per_sm = max(1, min(8, loss_env().ctas_per_sm));
    const int tile_env = loss_env().tile_cells;
    const size_t sm_smem = 228 * 1024, static_smem = 192;
    auto acc_bytes = [&](int warps) { return sizeof(double) * warps * n_scales * kTerms * 2; };
    const size_t bar_bytes = 2 * kMaxStages * sizeof(uint64_t);
    int total_tiles = 0, stage_bytes = 0, ncw = kLossMaxConsumerWarps;
    for (int pass = 0; pass < 2; ++pass) {  // pass 0 assumes the maximum warp count, pass 1 the real one
        int stage_budget = 0;
        for (;;) {
            const size_t per_cta = sm_smem / ctas_per_sm - 1024 - static_smem - acc_bytes(ncw) - bar_bytes;
            stage_budget = (int)(per_cta / n_stages) / 128 * 128;
            if (stage_budget >= 4 * cell_bytes_max) break;
            if (ctas_per_sm > 1) {
                --ctas_per_sm;
            } else if (n_stages > 2) {
                --n_stages;
            } else {
                return YB_E_SHAPE;  // 4 cells do not fit a stage: B*(5+C) too large
            }
        }
        total_tiles = 0;
        stage_bytes = 0;
        int warps = 1;
        for (int s = 0; s < n_scales; ++s) {
            LossScaleDev& d = L.sc[s];
            const int cb = (d.pcf + d.tcf) * 4;
            const int cpw = 32 / d.B;                        // cells one consumer warp covers per pass
            int t = stage_budget / cb / 4 * 4;
            t = min(t, kLossMaxConsumerWarps * cpw / 4 * 4);  // one pass of the consumer warps
            if (tile_env > 0) t = min(t, tile_env / 4 * 4);
            t = max(4, t);
            d.tile_cells = t;
            d.n_tiles = (int)((d.n_cells + t - 1) / t);
            d.tile_base = total_tiles;
            total_tiles += d.n_tiles;
            stage_bytes = max(stage_bytes, (int)align_up((size_t)t * cb, 128));  // 128 B-aligned stages
            warps = max(warps, min(kLossMaxConsumerWarps, (t + cpw - 1) / cpw));
        }
        ncw = max(1, min(kLossMaxConsumerWarps, (loss_env().warps > 0 ? loss_env().warps : warps)));
    }
    L.total_tiles = total_tiles;
    L.stage_bytes = stage_bytes;
    L.n_stages = n_stages;
    L.gacc = reinterpret_cast<double*>(workspace);
    L.ctrl = reinterpret_cast<unsigned int*>((char*)workspace + loss_gacc_bytes(n_scales));
    L.loss_out = loss_out;
    L.terms_out = terms_out;
    L.metrics_out = metrics_out;
    for (int s = 0; s < n_scales; ++s) L.sc[s].recall_thr = (float)recall_iou_threshold;
    if (dec != nullptr) L.dec = *dec;

    const size_t smem = (size_t)n_stages * stage_bytes + acc_bytes(ncw) + bar_bytes;
    const int threads = (ncw + 1) * 32;
    int grid = min(max(total_tiles, 1), kNumSMs * ctas_per_sm);
    // sums + control words start at zero; the kernel leaves them zeroed, so a caller that zeroed the
    // workspace once and only ever hands it to this kernel may skip the per-call memset
    if (!workspace_is_clean)
        YB_CUDA_TRY(cudaMemsetAsync(workspace, 0, loss_gacc_bytes(n_scales) + kCtrlWords * sizeof(unsigned int), stream));
    switch (version) {
        case 1: return launch_loss<1>(L, dec != nullptr, grid, threads, smem, stream);
        case 2: return launch_loss<2>(L, dec != nullptr, grid, threads, smem, stream);
        case 3: return launch_loss<3>(L, dec != nullptr, grid, threads, smem, stream);
        default: return launch_loss<4>(L, dec != nullptr, grid, threads, smem, stream);
    }
}

extern "C" int yb_loss_fwd_bwd(const yb_loss_scale* scales, int n_scales, float* loss_out,
                               double* terms_out, void* workspace, size_t workspace_bytes,
                               yb_stream_t stream) {
    return loss_impl(scales, n_scales, loss_out, terms_out, nullptr, 0.5, workspace, workspace_bytes, stream);
}

extern "C" int yb_loss_fwd_bwd_metrics(const yb_loss_scale* scales, int n_scales, float* loss_out,
                                       double* terms_out, double* metrics_out, double recall_iou_threshold,
                                       void* workspace, size_t workspace_bytes, yb_stream_t stream) {
    if (metrics_out == nullptr) return YB_E_NULL;
    return loss_impl(scales, n_scales, loss_out, terms_out, metrics_out, recall_iou_threshold, workspace,
                     workspace_bytes, stream);
}

// The decode parameters and head pointers of the float32 heads the loss scales hold; every scale must
// hold the same images, of one version and class count.  YB_OK / YB_E_*.
static int loss_decode_params(const yb_loss_scale* scales, int n_scales, double threshold, yb_decode_params& dp,
                              const void** preds, int64_t& n_img) {
    memset(&dp, 0, sizeof(dp));
    dp.version = scales[0].p.version;
    dp.class_num = scales[0].p.class_num;
    dp.n_scales = n_scales;
    dp.is_f64 = 0;
    dp.threshold = threshold;
    n_img = -1;
    for (int s = 0; s < n_scales; ++s) {
        const yb_loss_params& p = scales[s].p;
        // raw heads: every scale, and only the sigmoid heads of v3/v4 (v1/v2 end in a softmax)
        if ((p.from_logits != 0) != (scales[0].p.from_logits != 0)) return YB_E_PARAM;
        if (p.from_logits && p.version != 3 && p.version != 4) return YB_E_PARAM;
        if (p.grid_h <= 0 || p.grid_w <= 0) return YB_E_SHAPE;
        const int64_t cells = (int64_t)p.grid_h * p.grid_w;
        if (scales[s].n_cells % cells != 0) return YB_E_SHAPE;
        const int64_t n = scales[s].n_cells / cells;
        if (n_img >= 0 && n != n_img) return YB_E_SHAPE;
        n_img = n;
        if (p.class_num != dp.class_num || p.version != dp.version) return YB_E_PARAM;
        dp.grid_h[s] = p.grid_h;
        dp.grid_w[s] = p.grid_w;
        dp.bbox_num[s] = p.bbox_num;
        preds[s] = scales[s].y_pred;
    }
    return YB_OK;
}

// Loss fwd+grad AND head decode of the same head outputs: y_pred is read from HBM once for both.
extern "C" int yb_loss_decode_fused(const yb_loss_scale* scales, int n_scales, float* loss_out,
                                    double* terms_out, double decode_threshold, double* rows,
                                    int64_t row_capacity, int64_t* row_offsets, void* loss_workspace,
                                    size_t loss_workspace_bytes, void* decode_workspace,
                                    size_t decode_workspace_bytes, yb_stream_t stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    if (scales == nullptr) return YB_E_NULL;
    if (n_scales < 1 || n_scales > YB_MAX_SCALES) return YB_E_SHAPE;
    if (rows == nullptr && row_capacity > 0) return YB_E_NULL;
    const bool count_only = row_offsets == nullptr;  // rows are emitted later by yb_decode_finish
    if (row_capacity < 0) return YB_E_CAPACITY;
    // the emit pass reads the rows back from the head tensors, which must hold activated values:
    // activate raw heads with yb_activate_head first
    for (int s = 0; s < n_scales; ++s)
        if (scales[s].p.from_logits) return YB_E_PARAM;
    yb_decode_params dp;
    const void* preds[YB_MAX_SCALES];
    int64_t n_img;
    int rc = loss_decode_params(scales, n_scales, decode_threshold, dp, preds, n_img);
    if (rc != YB_OK) return rc;
    DecodeLaunch DL;
    DecodeWs ws;
    rc = decode_setup(preds, n_img, &dp, decode_workspace, decode_workspace_bytes, DL, ws);
    if (rc != YB_OK) return rc;
    if (ws.total_cells == 0) {
        if (!count_only) YB_CUDA_TRY(cudaMemsetAsync(row_offsets, 0, sizeof(int64_t) * (n_img + 1), stream));
        return loss_impl(scales, n_scales, loss_out, terms_out, nullptr, 0.5, loss_workspace, loss_workspace_bytes,
                         stream_);
    }
    YB_CUDA_TRY(cudaMemsetAsync(ws.n_hot, 0, ws.zero_bytes, stream));
    const DecodeSink dec = decode_sink(DL, ws.counts, ws.n_hot, ws.hot, HotBuckets{});
    rc = loss_impl(scales, n_scales, loss_out, terms_out, nullptr, 0.5, loss_workspace, loss_workspace_bytes,
                   stream_, &dec);
    if (rc != YB_OK || count_only) return rc;
    return decode_finish(DL, ws, false, rows, row_capacity, reinterpret_cast<long long*>(row_offsets), stream, true);
}

// The whole train-and-evaluate step in TWO launches: the loss kernel (forward + gradient + the
// decode counting pass into per-image buckets) and the one-CTA-per-image decode + NMS kernel.
static int step_impl(const yb_loss_scale* scales, int n_scales, float* loss_out, double* terms_out,
                     double decode_threshold, double nms_threshold, int iou_mode, int rows_per_img_cap,
                     double* out_rows, int64_t out_capacity, int64_t* out_offsets, unsigned int* n_overflow,
                     void* loss_workspace, size_t loss_workspace_bytes, void* fused_workspace,
                     size_t fused_workspace_bytes, yb_stream_t stream_, bool clean) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    if (scales == nullptr) return YB_E_NULL;
    const bool count_only = out_offsets == nullptr;   // the per-image kernel comes later: yb_decode_nms_finish
    if (n_scales < 1 || n_scales > YB_MAX_SCALES) return YB_E_SHAPE;
    if (out_rows == nullptr && out_capacity > 0) return YB_E_NULL;
    if (out_capacity < 0) return YB_E_CAPACITY;
    if (iou_mode != 1 && iou_mode != 2) return YB_E_PARAM;
    yb_decode_params dp;
    const void* preds[YB_MAX_SCALES];
    int64_t n_img;
    int rc = loss_decode_params(scales, n_scales, decode_threshold, dp, preds, n_img);
    if (rc != YB_OK) return rc;
    if (n_img == 0) {
        if (!count_only) YB_CUDA_TRY(cudaMemsetAsync(out_offsets, 0, sizeof(int64_t), stream));
        if (n_overflow != nullptr) YB_CUDA_TRY(cudaMemsetAsync(n_overflow, 0, sizeof(unsigned int), stream));
        return loss_impl(scales, n_scales, loss_out, terms_out, nullptr, 0.5, loss_workspace, loss_workspace_bytes,
                         stream_);
    }
    DecodeLaunch DL;
    HotBuckets K;
    rc = fused_prepare(preds, n_img, &dp, rows_per_img_cap, fused_workspace, fused_workspace_bytes, DL, K, stream,
                       !clean);
    if (rc != YB_OK) return rc;
    const DecodeSink dec = decode_sink(DL, nullptr, nullptr, nullptr, K);   // only the per-image buckets are filled
    rc = loss_impl(scales, n_scales, loss_out, terms_out, nullptr, 0.5, loss_workspace, loss_workspace_bytes, stream_,
                   &dec, clean);
    if (rc != YB_OK || count_only) return rc;
    return fused_finish(DL, n_img, rows_per_img_cap, fused_workspace, nms_threshold, iou_mode, out_rows, out_capacity,
                        out_offsets, n_overflow, stream);
}

extern "C" int yb_loss_decode_nms_fused(const yb_loss_scale* scales, int n_scales, float* loss_out,
                                        double* terms_out, double decode_threshold, double nms_threshold,
                                        int iou_mode, int rows_per_img_cap, double* out_rows,
                                        int64_t out_capacity, int64_t* out_offsets, unsigned int* n_overflow,
                                        void* loss_workspace, size_t loss_workspace_bytes, void* fused_workspace,
                                        size_t fused_workspace_bytes, yb_stream_t stream) {
    return step_impl(scales, n_scales, loss_out, terms_out, decode_threshold, nms_threshold, iou_mode, rows_per_img_cap,
                     out_rows, out_capacity, out_offsets, n_overflow, loss_workspace, loss_workspace_bytes,
                     fused_workspace, fused_workspace_bytes, stream, false);
}

// The same for workspaces the caller zeroed ONCE and has handed to nothing but this entry point
// since: both kernels leave their control blocks zeroed, so the step is two launches and nothing else
// (no memsets) - what a captured CUDA graph of a training loop replays.
extern "C" int yb_loss_decode_nms_fused_clean(const yb_loss_scale* scales, int n_scales, float* loss_out,
                                              double* terms_out, double decode_threshold, double nms_threshold,
                                              int iou_mode, int rows_per_img_cap, double* out_rows,
                                              int64_t out_capacity, int64_t* out_offsets, unsigned int* n_overflow,
                                              void* loss_workspace, size_t loss_workspace_bytes,
                                              void* fused_workspace, size_t fused_workspace_bytes,
                                              yb_stream_t stream) {
    if (out_offsets == nullptr) return YB_E_NULL;   // the split form would leave the buckets filled
    return step_impl(scales, n_scales, loss_out, terms_out, decode_threshold, nms_threshold, iou_mode, rows_per_img_cap,
                     out_rows, out_capacity, out_offsets, n_overflow, loss_workspace, loss_workspace_bytes,
                     fused_workspace, fused_workspace_bytes, stream, true);
}

static int loss_single(int version, const float* y_true, const float* y_pred, int64_t n_cells,
                       float* loss_out, float* dpred, const yb_loss_params* p, void* workspace,
                       size_t workspace_bytes, yb_stream_t stream) {
    if (p == nullptr) return YB_E_NULL;
    if (p->version != version) return YB_E_PARAM;
    yb_loss_scale sc;
    sc.y_true = y_true;
    sc.y_pred = y_pred;
    sc.dpred = dpred;
    sc.n_cells = n_cells;
    sc.p = *p;
    return yb_loss_fwd_bwd(&sc, 1, loss_out, nullptr, workspace, workspace_bytes, stream);
}

#define YB_DEFINE_LOSS(V)                                                                          \
    extern "C" int yb_loss_v##V##_fwd_bwd(const float* y_true, const float* y_pred, int64_t n_cells, \
                                          float* loss_out, float* dpred, const yb_loss_params* p,   \
                                          void* workspace, size_t workspace_bytes,                  \
                                          yb_stream_t stream) {                                     \
        return loss_single(V, y_true, y_pred, n_cells, loss_out, dpred, p, workspace,               \
                           workspace_bytes, stream);                                                \
    }
YB_DEFINE_LOSS(1)
YB_DEFINE_LOSS(2)
YB_DEFINE_LOSS(3)
YB_DEFINE_LOSS(4)

extern "C" int yb_activate_head(const yb_loss_params* p, const float* raw, float* out, int64_t n_cells,
                                yb_stream_t stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    if (p == nullptr || raw == nullptr || out == nullptr) return YB_E_NULL;
    if ((p->version != 3 && p->version != 4) || !p->has_anchors) return YB_E_PARAM;
    if (p->bbox_num <= 0 || p->bbox_num > YB_MAX_BOXES || p->class_num <= 0 || n_cells < 0) return YB_E_SHAPE;
    const long long bs = 5LL + p->class_num, cell_floats = p->bbox_num * bs;
    if (n_cells > INT64_MAX / cell_floats || cell_floats > INT32_MAX) return YB_E_SHAPE;
    if (((uintptr_t)raw | (uintptr_t)out) & 3) return YB_E_ALIGN;
    const long long n = n_cells * cell_floats;
    if (n == 0) return YB_OK;
    HeadAnchors anc;
    for (int i = 0; i < 2 * YB_MAX_BOXES; ++i) anc.a[i] = (i < 2 * p->bbox_num) ? p->anchors[i] : 1.f;
    const bool vec = (((uintptr_t)raw | (uintptr_t)out) & 15) == 0;
    const int kw = vec ? 4 : 1, threads = 256;
    const long long n_items = n / kw;
    const int blocks = (int)max(1LL, min((long long)kNumSMs * 8, (n_items + threads - 1) / threads));
    const long long adv = ((long long)blocks * threads * kw) % cell_floats;
    const int adv_b = (int)(adv / bs), adv_j = (int)(adv % bs), n_tail = (int)(n - n_items * kw);
    if (vec)
        activate_head_kernel<4><<<blocks, threads, 0, stream>>>(raw, out, n_items, n_tail, (int)bs, p->bbox_num, adv_b,
                                                                 adv_j, anc);
    else
        activate_head_kernel<1><<<blocks, threads, 0, stream>>>(raw, out, n_items, n_tail, (int)bs, p->bbox_num, adv_b,
                                                                 adv_j, anc);
    YB_CUDA_TRY(cudaGetLastError());
    return YB_OK;
}

extern "C" int yb_grid_iou(const float* box_true, int true_stride, const float* box_pred,
                           int pred_stride, int64_t n_cells, int bbox_num, int grid_h, int grid_w,
                           float* iou_out, float* ciou_out, yb_stream_t stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    if (box_true == nullptr || box_pred == nullptr || iou_out == nullptr) return YB_E_NULL;
    if (n_cells < 0 || bbox_num <= 0 || grid_h <= 0 || grid_w <= 0 || true_stride < 4 || pred_stride < 4)
        return YB_E_SHAPE;
    const long long n = (long long)n_cells * bbox_num;
    if (n == 0) return YB_OK;
    const int threads = 256;
    const long long blocks = (n + threads - 1) / threads;
    grid_iou_kernel<<<(unsigned)blocks, threads, 0, stream>>>(box_true, true_stride, box_pred, pred_stride,
                                                              n, bbox_num, (float)grid_w, (float)grid_h,
                                                              iou_out, ciou_out);
    YB_CUDA_TRY(cudaGetLastError());
    return YB_OK;
}
