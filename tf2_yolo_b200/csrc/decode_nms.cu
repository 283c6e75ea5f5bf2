// Head decode + per-class NMS of a batch in ONE launch, one CTA per image.
//
// Replaces the chain  yb_decode (scan + emit)  ->  yb_nms (classify, scatter, sweep, emit)  -
// six latency-bound launches and three memsets behind the counting pass - for the regime the
// train-and-evaluate step and per-image inference live in: at most a few thousand rows per image
// (utils/tools.py:370-438 decode, :687-733 nms with the IoU of :630-684).  The decode rows of an
// image never leave the SM: the counting pass (decode_count_kernel or the fused loss kernel) files
// every hit - the head's values it holds anyway - into the image's bucket; the image's CTA orders
// them (row-major cell, box, class), builds the float64 rows [x, y, w, h, c, class, p] in shared
// memory in the reference's order, groups them by class and runs the greedy (D)IoU-NMS of every
// class (visit order = confidence descending, equal confidences -> higher original index first;
// suppression on >=; division-free pair test with the pinned exact fallback, see nms_pair.cuh).
// The pair test of two boxes does not depend on the state of the sweep, so for classes of up to
// 128 rows ALL pairs of ALL classes are tested in parallel (a flat list of pairs, contiguous runs
// per thread): the earlier-visited box of a pair gets the later one's bit in its 128-bit mask, and
// the sweep itself is one thread per class walking the visit order: dead |= mask[v] if v is alive.
// Larger classes keep one warp each.  Survivors leave class-major, original order inside a class, at
// the image's offset in the compact output - found with a decoupled look-back over the earlier
// images (tickets make every predecessor of a CTA already running, so the chain cannot stall).
// The last CTA to finish leaves the control block (bucket counters, look-back words, tickets) zeroed:
// a caller that zeroed the workspace once never has to again (yb_loss_decode_nms_fused_clean).
// Results are bit-identical to the six-launch chain.  An image with more rows than the caller's
// rows_per_img_cap is not processed: it contributes no rows and is counted in *n_overflow; the
// caller falls back to yb_decode + yb_nms (same contract as the row capacity of yb_decode).
#include <climits>
#include <cstring>

#include "common.cuh"
#include "decode_internal.cuh"
#include "nms_pair.cuh"

namespace yb {

constexpr int kFusedThreads = 1024;
constexpr int kFusedWarps = kFusedThreads / 32;

constexpr unsigned long long kStFlagAgg = 1ull << 62, kStFlagIncl = 2ull << 62, kStFlagMask = 3ull << 62;
constexpr int kStOvfShift = 40;          // payload: survivors in bits 0..39, overflowed images in 40..61

struct FusedLaunch {
    DecodeLaunch D;            // float32 heads
    HotBuckets K;
    int row_cap;               // rows (and hot boxes) per image held in shared memory
    double nms_thr;
    double* out_rows;          // compact survivors (may be mapped host memory)
    long long out_cap;
    long long* out_offsets;    // [n_img + 1]
    unsigned int* n_overflow;  // [1] or null
    unsigned long long* status;   // [n_img] look-back words, zero on entry
    unsigned int* ticket;         // [2]: ticket counter, finished-CTA counter; zero on entry, zero on exit
};

__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Classes of up to kMaskMembers rows take the mask path of the greedy sweep (every pair tested in
// parallel, then one short scan per class); larger classes keep one warp each.
constexpr int kMaskWords = 4, kMaskMembers = 32 * kMaskWords;

// shared-memory carve-up for R = row_cap rows and C classes (host and device agree through this)
struct FusedSmem {
    size_t rows, conf, key, cls, vis, vrank, rank, outsrc, mask, ccount, cstart, ckept, cpair, cdead, total;
    __host__ __device__ FusedSmem(int R, int C) {
        size_t o = 0;
        auto take = [&](size_t bytes) { const size_t at = o; o += (bytes + 15) / 16 * 16; return at; };
        rows = take(sizeof(double) * 7 * R);
        conf = take(sizeof(double) * R);
        key = take(4 * (size_t)R);
        cls = take(2 * (size_t)R);
        vis = take(2 * (size_t)R);
        vrank = take(4 * (size_t)R);
        rank = take(2 * (size_t)R);
        outsrc = take(2 * (size_t)R);
        mask = take(4 * (size_t)kMaskWords * R);
        ccount = take(4 * (size_t)C);
        cstart = take(4 * ((size_t)C + 1));
        ckept = take(4 * ((size_t)C + 1));
        cpair = take(4 * ((size_t)C + 1));
        cdead = take(4 * (size_t)kMaskWords * C);
        total = o;
    }
};

#ifdef YB_FUSED_PROF
__device__ unsigned long long g_fused_prof[4096 * 16];
__device__ __forceinline__ unsigned long long prof_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t) :: "memory");
    return t;
}
#define PROF(k) do { if (threadIdx.x == 0 && blockIdx.x < 4096) g_fused_prof[blockIdx.x * 16 + (k)] = prof_now(); } while (0)
#else
#define PROF(k) do { } while (0)
#endif

// pairs of a class that takes the mask path
__device__ __forceinline__ unsigned mask_pairs(unsigned n) {
    return (n >= 2u && n <= (unsigned)kMaskMembers) ? n * (n - 1u) / 2u : 0u;
}

template <int MODE>
__global__ void __launch_bounds__(kFusedThreads)
decode_nms_image_kernel(const __grid_constant__ FusedLaunch F) {
    extern __shared__ __align__(16) unsigned char fsm[];
    const DecodeLaunch& L = F.D;
    const int R = F.row_cap, C = L.C;
    const FusedSmem lay(R, C);
    double* s_rows = reinterpret_cast<double*>(fsm + lay.rows);
    double* s_conf = reinterpret_cast<double*>(fsm + lay.conf);
    unsigned int* s_key = reinterpret_cast<unsigned int*>(fsm + lay.key);
    unsigned short* s_cls = reinterpret_cast<unsigned short*>(fsm + lay.cls);
    unsigned short* s_vis = reinterpret_cast<unsigned short*>(fsm + lay.vis);
    unsigned int* s_vrank = reinterpret_cast<unsigned int*>(fsm + lay.vrank);
    unsigned int* s_mask = reinterpret_cast<unsigned int*>(fsm + lay.mask);
    unsigned int* s_cdead = reinterpret_cast<unsigned int*>(fsm + lay.cdead);
    unsigned int* s_cpair = reinterpret_cast<unsigned int*>(fsm + lay.cpair);
    unsigned short* s_rank = reinterpret_cast<unsigned short*>(fsm + lay.rank);
    unsigned short* s_outsrc = reinterpret_cast<unsigned short*>(fsm + lay.outsrc);
    unsigned int* s_ccount = reinterpret_cast<unsigned int*>(fsm + lay.ccount);
    unsigned int* s_cstart = reinterpret_cast<unsigned int*>(fsm + lay.cstart);
    unsigned int* s_ckept = reinterpret_cast<unsigned int*>(fsm + lay.ckept);
    __shared__ unsigned int s_img, s_kept;
    __shared__ long long s_base;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    PROF(0);
    if (tid == 0) {
        s_img = atomicAdd(F.ticket, 1u);   // images in ticket order: predecessors are running
    }
    for (int c = tid; c < C; c += kFusedThreads) {
        s_ccount[c] = 0u;
        s_ckept[c] = 0u;
    }
    __syncthreads();
    const long long img = s_img;
    PROF(1);

    // ---- 1. the image's rows, as the counting pass filed them (any order): class histogram ----------
    const unsigned n_filed = F.K.n[img];
    const bool overflow = n_filed > (unsigned)min(R, F.K.cap);
    const int n_rows = overflow ? 0 : (int)n_filed;
    const FusedRow* bucket = F.K.row + img * F.K.cap;
    for (int i = tid; i < n_rows; i += kFusedThreads) atomicAdd(&s_ccount[bucket[i].key & 255u], 1u);
    __syncthreads();
    PROF(2);
    // exclusive prefixes over the classes (C <= 256): warp 0, eight classes per lane
    if (warp == 0) {
        unsigned cnt[8], sum = 0, prs = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int c = lane * 8 + k;
            const unsigned n = c < C ? s_ccount[c] : 0u;
            cnt[k] = n;
            sum += n;
            prs += mask_pairs(n);
        }
        unsigned xs = sum, xp = prs;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned ts = __shfl_up_sync(0xffffffffu, xs, o), tp = __shfl_up_sync(0xffffffffu, xp, o);
            if (lane >= o) { xs += ts; xp += tp; }
        }
        unsigned es = xs - sum, ep = xp - prs;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int c = lane * 8 + k;
            if (c <= C) { s_cstart[c] = es; s_cpair[c] = ep; }
            es += cnt[k];
            ep += mask_pairs(cnt[k]);
        }
        if (lane == 31 && C == 256) { s_cstart[256] = es; s_cpair[256] = ep; }
    }
    __syncthreads();
    PROF(3);
#ifdef YB_FUSED_PROF
    if (tid == 0 && blockIdx.x < 4096) {
        unsigned mx = 0;
        for (int c = 0; c < C; ++c) mx = max(mx, s_ccount[c]);
        g_fused_prof[blockIdx.x * 16 + 12] = n_rows;
        g_fused_prof[blockIdx.x * 16 + 13] = mx;
        g_fused_prof[blockIdx.x * 16 + 14] = img;
    }
#endif
    // ---- 2. class-major order.  Only the survivors leave the kernel, class-major and in the
    //         reference's row order inside a class (utils/tools.py:730-732), so the rows are sorted
    //         by (class, cell, box) directly: a row takes any free slot of its class segment, then
    //         its rank among the (few) rows of that segment is its final position ---------------------
    for (int i = tid; i < n_rows; i += kFusedThreads) {
        const unsigned key = bucket[i].key;
        const unsigned cls = key & 255u;
        const unsigned slot = s_cstart[cls] + atomicAdd(&s_ckept[cls], 1u);   // s_ckept: fill counters for now
        s_key[slot] = key;
    }
    __syncthreads();
    PROF(4);
    for (int i = tid; i < n_rows; i += kFusedThreads) {
        const FusedRow fr = bucket[i];
        const unsigned key = fr.key, cls = key & 255u;
        const int start = (int)s_cstart[cls], n = (int)s_ccount[cls];
        int rank = start;
        for (int j = 0; j < n; ++j) rank += (s_key[start + j] < key) ? 1 : 0;   // keys are unique
        // the float64 row of utils/tools.py:426-436: x = (x_i + x) / grid_w, y = (y_i + y) / grid_h
        const int s = (int)(fr.cell >> 28);
        const unsigned cell = fr.cell & 0x0fffffffu;
        const int yi = (int)(cell / (unsigned)L.gw[s]), xi = (int)(cell - (unsigned)yi * (unsigned)L.gw[s]);
        double* o = s_rows + (size_t)rank * 7;
        o[0] = ((double)xi + (double)fr.x) / (double)L.gw[s];
        o[1] = ((double)yi + (double)fr.y) / (double)L.gh[s];
        o[2] = (double)fr.w; o[3] = (double)fr.h; o[4] = (double)fr.c;
        o[5] = (double)cls;
        o[6] = (double)fr.p;
        s_cls[rank] = (unsigned short)cls;
        s_vrank[rank] = 0u;
        *reinterpret_cast<uint4*>(s_mask + (size_t)rank * kMaskWords) = make_uint4(0u, 0u, 0u, 0u);
        s_conf[rank] = __dmul_rn((double)fr.c, (double)fr.p);   // conf = c * p in float64 (utils/tools.py:716)
    }
    __syncthreads();
    PROF(5);
    for (int c = tid; c < C; c += kFusedThreads) s_ckept[c] = 0u;
    const bool pos_thr = F.nms_thr > 0.0;
    const double nms_thr = F.nms_thr;
    // ---- 3. every pair of a class, in parallel, one pair per thread and turn.  Member i of a class
    //         is visited at rank #{j : j before i} (np.argsort(conf)[::-1], utils/tools.py:717); if
    //         it is visited alive it removes the later members its IoU test hits (:722-726) - that
    //         set is a mask over the class, independent of the sweep.  Pair q of the image -> class
    //         (search in the prefix of n(n-1)/2) -> members i < j (row of the triangle) ---------------
    const int n_pairs = (int)s_cpair[C];
    {
        // a thread takes a contiguous run of pairs: one search, then (i, j) -> (i, j + 1) -> next row
        // of the triangle -> next class; the box of member i is built once per row
        const int len = (n_pairs + kFusedThreads - 1) / kFusedThreads;
        int q = tid * len;
        const int q_end = min(n_pairs, q + len);
        if (q < q_end) {
            int lo = 0, hi = C;                               // largest c with s_cpair[c] <= q
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if ((int)s_cpair[mid] <= q) lo = mid; else hi = mid;
            }
            int c = lo, n = (int)s_ccount[c], start = (int)s_cstart[c];
            const int k = q - (int)s_cpair[c];
            const int m = 2 * n - 1;
            int i = (int)(((float)m - sqrtf((float)(m * m - 8 * k))) * 0.5f);
            i = max(0, min(i, n - 2));
            while (i * (m - i) / 2 > k) --i;                  // pairs before row i: i (2n - i - 1) / 2
            while ((i + 1) * (m - i - 1) / 2 <= k) ++i;
            int j = i + 1 + (k - i * (m - i) / 2);
            const double* pi = s_rows + (size_t)(start + i) * 7;
            BoxC bi = make_box(pi[0], pi[1], pi[2], pi[3]);
            double ci = s_conf[start + i];
            for (;;) {
                const int ri = start + i, rj = start + j;
                const bool i_first = visited_before(ci, i, s_conf[rj], j);
                atomicAdd(&s_vrank[i_first ? rj : ri], 1u);    // the later one is visited after one more
                const double* pj = s_rows + (size_t)rj * 7;
                const BoxC bj = make_box(pj[0], pj[1], pj[2], pj[3]);
                // the division-free test is symmetric bit for bit (min/max, commutative sums, squares);
                // the exact expression gets the boxes in the order of the sweep
                const int fast = suppresses_fast<MODE>(bi, bj, nms_thr, pos_thr);
                const int ra = i_first ? ri : rj, rb = i_first ? rj : ri;
                if (fast > 0 || (fast < 0 && suppresses_exact<MODE>(s_rows, ra, rb, nms_thr))) {
                    const int mb = rb - start;
                    atomicOr(&s_mask[(size_t)ra * kMaskWords + (mb >> 5)], 1u << (mb & 31));
                }
                if (++q >= q_end) break;
                if (++j >= n) {
                    ++i;
                    if (i >= n - 1) {                         // next class with pairs (there is one: q < n_pairs)
                        do {
                            ++c;
                            n = (int)s_ccount[c];
                        } while (n < 2 || n > kMaskMembers);
                        start = (int)s_cstart[c];
                        i = 0;
                    }
                    j = i + 1;
                    pi = s_rows + (size_t)(start + i) * 7;
                    bi = make_box(pi[0], pi[1], pi[2], pi[3]);
                    ci = s_conf[start + i];
                }
            }
        }
    }
    // rows of a class too large for a mask: only the visit rank (the warp sweep below does the rest)
    for (int r = tid; r < n_rows; r += kFusedThreads) {
        const int c = s_cls[r];
        const int n = (int)s_ccount[c];
        if (n <= kMaskMembers) continue;
        const int start = (int)s_cstart[c], i = r - start;
        const double ci = s_conf[r];
        int vis = 0;
        for (int j = 0; j < n; ++j) vis += (j != i && visited_before(s_conf[start + j], j, ci, i)) ? 1 : 0;
        s_vrank[r] = (unsigned)vis;
    }
    __syncthreads();
    PROF(6);
    for (int r = tid; r < n_rows; r += kFusedThreads) {
        const int start = (int)s_cstart[s_cls[r]];
        s_vis[start + (int)s_vrank[r]] = (unsigned short)(r - start);
    }
    __syncthreads();
    // ---- 4a. classes too large for a mask: one warp each, greedy sweep in visit order --------------
    for (int c = warp; c < C; c += kFusedWarps) {
        const int n = (int)s_ccount[c];
        if (n <= kMaskMembers) continue;
        const int start = (int)s_cstart[c];
        // lane l owns members l, l+32, ...; dead bit t of a lane = member l + 32 t
        unsigned dead = 0;
        for (int v = 0; v < n; ++v) {
            const int iv = s_vis[start + v];
            const unsigned dv = __shfl_sync(0xffffffffu, dead, iv & 31);
            if ((dv >> (iv >> 5)) & 1u) continue;            // a suppressed box suppresses nothing (:723)
            const int rv = start + iv;
            const double* a = s_rows + (size_t)rv * 7;
            const BoxC av = make_box(a[0], a[1], a[2], a[3]);
            for (int i = lane, t = 0; i < n; i += 32, ++t) {
                if ((dead >> t) & 1u) continue;
                if ((int)s_vrank[start + i] <= v) continue;   // already visited (white list, :722)
                const int ri = start + i;
                const double* b = s_rows + (size_t)ri * 7;
                const BoxC bi = make_box(b[0], b[1], b[2], b[3]);
                if (suppresses<MODE>(av, bi, nms_thr, pos_thr, s_rows, rv, ri)) dead |= 1u << t;
            }
        }
        // survivors: position inside the class, original order
        int kept_before = 0;
        for (int i0 = 0, t = 0; i0 < n; i0 += 32, ++t) {
            const int i = i0 + lane;
            const bool alive = i < n && !((dead >> t) & 1u);
            const unsigned m = __ballot_sync(0xffffffffu, alive);
            if (i < n) s_rank[start + i] = alive ? (unsigned short)(kept_before + __popc(m & lt_mask)) : 0xffffu;
            kept_before += __popc(m);
        }
        if (lane == 0) s_ckept[c] = (unsigned)kept_before;
    }
    // ---- 4b. the other classes: one thread each walks the visit order over the masks (neighbouring
    //          classes on different warps: a warp takes as long as its longest class) ----------------
    {
        const int c = lane * kFusedWarps + warp;
        const int n = c < C ? (int)s_ccount[c] : 0;
        if (c < C && n <= kMaskMembers) {
            const int start = (int)s_cstart[c];
            unsigned long long d0 = 0, d1 = 0;
#pragma unroll 4
            for (int v = 0; v < n; ++v) {        // no branch: the loads of the next turns do not wait for this one
                const int iv = s_vis[start + v];
                const uint4 m = *reinterpret_cast<const uint4*>(s_mask + (size_t)(start + iv) * kMaskWords);
                const unsigned long long w = iv < 64 ? d0 : d1;
                // a suppressed box suppresses nothing (:723)
                const unsigned long long live = ((w >> (iv & 63)) & 1ull) ? 0ull : ~0ull;
                d0 |= ((unsigned long long)m.x | ((unsigned long long)m.y << 32)) & live;
                d1 |= ((unsigned long long)m.z | ((unsigned long long)m.w << 32)) & live;
            }
            uint4 d;
            d.x = (unsigned)d0; d.y = (unsigned)(d0 >> 32); d.z = (unsigned)d1; d.w = (unsigned)(d1 >> 32);
            *reinterpret_cast<uint4*>(s_cdead + (size_t)c * kMaskWords) = d;
            s_ckept[c] = (unsigned)(n - __popcll(d0) - __popcll(d1));
        }
    }
    __syncthreads();
    // survivors of the mask classes: position inside the class, original order
    for (int r = tid; r < n_rows; r += kFusedThreads) {
        const int c = s_cls[r];
        if ((int)s_ccount[c] > kMaskMembers) continue;
        const int i = r - (int)s_cstart[c];
        const unsigned* d = s_cdead + (size_t)c * kMaskWords;
        const int wi = i >> 5;
        const unsigned dw = d[wi];
        if ((dw >> (i & 31)) & 1u) {
            s_rank[r] = 0xffffu;
        } else {
            int dead_before = __popc(dw & ((1u << (i & 31)) - 1u));
            for (int w = 0; w < wi; ++w) dead_before += __popc(d[w]);
            s_rank[r] = (unsigned short)(i - dead_before);
        }
    }
    PROF(7);      // thread 0's own classes done
    __syncthreads();
    PROF(8);
    // ---- 5. survivors of the image: class-major positions; the image's offset by look-back ---------
    if (warp == 0) {                   // exclusive prefix of the kept counts
        unsigned cnt[8], sum = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int c = lane * 8 + k;
            cnt[k] = c < C ? s_ckept[c] : 0u;
            sum += cnt[k];
        }
        unsigned xs = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned ts = __shfl_up_sync(0xffffffffu, xs, o);
            if (lane >= o) xs += ts;
        }
        unsigned es = xs - sum;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int c = lane * 8 + k;
            if (c < C) s_ckept[c] = es;
            es += cnt[k];
        }
        if (lane == 31) s_kept = xs;
    }
    __syncthreads();
    PROF(9);
    if (warp == 0) {
        const unsigned long long agg = (unsigned long long)s_kept | ((unsigned long long)(overflow ? 1 : 0) << kStOvfShift);
        unsigned long long excl = 0;
        if (img > 0) {
            if (lane == 0) st_release_u64(&F.status[img], kStFlagAgg | agg);
            long long j = img - 1;
            for (;;) {
                const long long idx = j - lane;
                unsigned long long st = kStFlagIncl;   // before image 0: inclusive prefix 0
                if (idx >= 0) {
                    st = ld_acquire_u64(&F.status[idx]);
                    while ((st & kStFlagMask) == 0) {
                        __nanosleep(40);
                        st = ld_acquire_u64(&F.status[idx]);
                    }
                }
                const unsigned incl = __ballot_sync(0xffffffffu, (st & kStFlagMask) == kStFlagIncl);
                const int stop = incl ? (__ffs(incl) - 1) : 31;   // nearest predecessor with an inclusive prefix
                unsigned long long part = (lane <= stop) ? (st & ~kStFlagMask) : 0ull;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
                excl += part;
                if (incl) break;
                j -= 32;
            }
        }
        if (lane == 0) {
            st_release_u64(&F.status[img], kStFlagIncl | (excl + agg));
            const long long base = (long long)(excl & ((1ull << kStOvfShift) - 1));
            s_base = base;
            F.out_offsets[img] = base;
            if (img == L.n_img - 1) {
                F.out_offsets[L.n_img] = base + s_kept;
                if (F.n_overflow != nullptr) *F.n_overflow = (unsigned)((excl + agg) >> kStOvfShift);
            }
        }
    }
    PROF(10);
    // source row of every output position, then a coalesced copy
    for (int r = tid; r < n_rows; r += kFusedThreads)
        if (s_rank[r] != 0xffffu) s_outsrc[s_ckept[s_cls[r]] + s_rank[r]] = (unsigned short)r;
    __syncthreads();
    if (F.out_rows != nullptr) {
        const long long base = s_base;
        const int n_out = (int)s_kept;
        for (int f = tid; f < n_out * 7; f += kFusedThreads) {
            const int q = f / 7, k = f - q * 7;
            if (base + q < F.out_cap) F.out_rows[(base + q) * 7 + k] = s_rows[(size_t)s_outsrc[q] * 7 + k];
        }
    }
    PROF(11);
    // leave the control block as it was found: this image's bucket counter now, the look-back words
    // and the counters by whichever CTA finishes last (every look-back is over by then)
    if (tid == 0) {
        F.K.n[img] = 0u;
        __threadfence();
        if (atomicAdd(F.ticket + 1, 1u) == (unsigned)L.n_img - 1u) {
            for (long long i = 0; i < L.n_img; ++i) F.status[i] = 0ull;
            F.ticket[0] = 0u;
            F.ticket[1] = 0u;
        }
    }
}

#ifdef YB_FUSED_PROF
extern "C" int yb_debug_fused_prof(unsigned long long* host, int n_words) {
    return (int)cudaMemcpyFromSymbol(host, g_fused_prof, sizeof(unsigned long long) * (size_t)n_words);
}
#endif

// ---- host side -----------------------------------------------------------------------------------
struct FusedWs {
    unsigned char* zero;          // [bucket counts | look-back status | ticket]: cleared by ONE memset
    size_t zero_bytes;
    HotBuckets K;
    unsigned long long* status;
    unsigned int* ticket;
};

static size_t fused_layout(long long n_img, int row_cap, FusedWs* W, char* base) {
    size_t off = 0;
    const size_t counts = align_up(sizeof(unsigned int) * (size_t)(n_img + 1), 256);
    const size_t status = align_up(sizeof(unsigned long long) * (size_t)(n_img + 1), 256);
    if (W) {
        W->zero = reinterpret_cast<unsigned char*>(base);
        W->K.n = reinterpret_cast<unsigned int*>(base);
        W->status = reinterpret_cast<unsigned long long*>(base + counts);
        W->ticket = reinterpret_cast<unsigned int*>(base + counts + status);
        W->zero_bytes = counts + status + 256;
        W->K.row = reinterpret_cast<FusedRow*>(base + counts + status + 256);
        W->K.cap = row_cap;
    }
    off = counts + status + 256 + align_up(sizeof(FusedRow) * (size_t)n_img * (size_t)row_cap, 256);
    return off;
}

static int fused_check(const yb_decode_params* p, int64_t n_img, int row_cap) {
    if (p == nullptr) return YB_E_NULL;
    if (p->is_f64) return YB_E_PARAM;                       // model outputs (float32) only
    if (n_img < 0 || n_img > (1 << 24)) return YB_E_SHAPE;
    if (p->class_num < 1 || p->class_num > 256) return YB_E_SHAPE;   // class in 8 bits of the row key
    if (row_cap < 32 || row_cap > YB_FUSED_MAX_ROWS) return YB_E_SHAPE;
    long long per_img = 0;
    for (int s = 0; s < p->n_scales && s < YB_MAX_SCALES; ++s) per_img += (long long)p->grid_h[s] * p->grid_w[s];
    if (per_img >= (1ll << 19)) return YB_E_SHAPE;          // (cell, box, class) key in 32 bits
    for (int s = 0; s < p->n_scales && s < YB_MAX_SCALES; ++s)
        if ((long long)p->grid_h[s] * p->grid_w[s] >= (1ll << 28) || p->bbox_num[s] > 32) return YB_E_SHAPE;
    return YB_OK;
}

// the kernel launch alone (buckets already filled by a counting pass on the same stream)
static int fused_launch(const DecodeLaunch& D, const FusedWs& W, int row_cap, double nms_threshold, int iou_mode,
                        double* out_rows, long long out_cap, long long* out_offsets, unsigned int* n_overflow,
                        cudaStream_t stream) {
    FusedLaunch F;
    memset(&F, 0, sizeof(F));
    F.D = D;
    F.K = W.K;
    F.row_cap = row_cap;
    F.nms_thr = nms_threshold;
    F.out_rows = out_rows;
    F.out_cap = out_cap;
    F.out_offsets = out_offsets;
    F.n_overflow = n_overflow;
    F.status = W.status;
    F.ticket = W.ticket;
    const FusedSmem lay(row_cap, D.C);
    if (lay.total > 220 * 1024) return YB_E_SHAPE;
    if (iou_mode == 1) {
        static SmemRaised done;
        YB_CUDA_TRY(raise_dynamic_smem_once(decode_nms_image_kernel<1>, (int)lay.total, &done));
        decode_nms_image_kernel<1><<<(unsigned)D.n_img, kFusedThreads, lay.total, stream>>>(F);
    } else {
        static SmemRaised done;
        YB_CUDA_TRY(raise_dynamic_smem_once(decode_nms_image_kernel<2>, (int)lay.total, &done));
        decode_nms_image_kernel<2><<<(unsigned)D.n_img, kFusedThreads, lay.total, stream>>>(F);
    }
    YB_CUDA_TRY(cudaGetLastError());
    return YB_OK;
}

// validation + workspace carve-up (no launches)
static int fused_setup(const void* const* preds, int64_t n_img, const yb_decode_params* p, int row_cap,
                       void* workspace, size_t workspace_bytes, DecodeLaunch& D, FusedWs& W) {
    int rc = fused_check(p, n_img, row_cap);
    if (rc != YB_OK) return rc;
    rc = decode_fill(preds, n_img, p, D);
    if (rc != YB_OK) return rc;
    if (workspace == nullptr) return YB_E_NULL;
    if (workspace_bytes < fused_layout(n_img, row_cap, nullptr, nullptr) || ((uintptr_t)workspace & 255))
        return YB_E_WORKSPACE;
    for (int s = 0; s < D.n_scales; ++s)
        if (D.n_img * D.cells[s] > 0xffffffffll || D.B[s] > 32) return YB_E_SHAPE;
    fused_layout(n_img, row_cap, &W, reinterpret_cast<char*>(workspace));
    return YB_OK;
}

// Shared with loss.cu (yb_loss_decode_nms_fused): fused_setup + memset, then the launch.
int fused_prepare(const void* const* preds, int64_t n_img, const yb_decode_params* p, int row_cap, void* workspace,
                  size_t workspace_bytes, DecodeLaunch& D, HotBuckets& K, cudaStream_t stream, bool clear) {
    FusedWs W;
    const int rc = fused_setup(preds, n_img, p, row_cap, workspace, workspace_bytes, D, W);
    if (rc != YB_OK) return rc;
    if (clear) YB_CUDA_TRY(cudaMemsetAsync(W.zero, 0, W.zero_bytes, stream));
    K = W.K;
    return YB_OK;
}

int fused_finish(const DecodeLaunch& D, int64_t n_img, int row_cap, void* workspace, double nms_threshold,
                 int iou_mode, double* out_rows, int64_t out_capacity, int64_t* out_offsets,
                 unsigned int* n_overflow, cudaStream_t stream) {
    FusedWs W;
    fused_layout(n_img, row_cap, &W, reinterpret_cast<char*>(workspace));
    return fused_launch(D, W, row_cap, nms_threshold, iou_mode, out_rows, out_capacity,
                        reinterpret_cast<long long*>(out_offsets), n_overflow, stream);
}

}  // namespace yb

using namespace yb;

extern "C" size_t yb_decode_nms_workspace_bytes(const yb_decode_params* p, int64_t n_img, int rows_per_img_cap) {
    if (fused_check(p, n_img, rows_per_img_cap) != YB_OK) return 0;
    return fused_layout(n_img, rows_per_img_cap, nullptr, nullptr);
}

extern "C" int yb_decode_nms(const void* const* preds, int64_t n_img, const yb_decode_params* p,
                             double nms_threshold, int iou_mode, int rows_per_img_cap, double* out_rows,
                             int64_t out_capacity, int64_t* out_offsets, unsigned int* n_overflow,
                             void* workspace, size_t workspace_bytes, yb_stream_t stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    if (out_offsets == nullptr) return YB_E_NULL;
    if (out_rows == nullptr && out_capacity > 0) return YB_E_NULL;
    if (out_capacity < 0) return YB_E_CAPACITY;
    if (iou_mode != 1 && iou_mode != 2) return YB_E_PARAM;
    if (n_img == 0) {
        int rc0 = fused_check(p, n_img, rows_per_img_cap);
        if (rc0 != YB_OK) return rc0;
        YB_CUDA_TRY(cudaMemsetAsync(out_offsets, 0, sizeof(int64_t), stream));
        if (n_overflow != nullptr) YB_CUDA_TRY(cudaMemsetAsync(n_overflow, 0, sizeof(unsigned int), stream));
        return YB_OK;
    }
    DecodeLaunch D;
    HotBuckets K;
    int rc = fused_prepare(preds, n_img, p, rows_per_img_cap, workspace, workspace_bytes, D, K, stream);
    if (rc != YB_OK) return rc;
    rc = decode_count(D, false, decode_sink(D, nullptr, nullptr, nullptr, K), stream);
    if (rc != YB_OK) return rc;
    return fused_finish(D, n_img, rows_per_img_cap, workspace, nms_threshold, iou_mode, out_rows, out_capacity,
                        out_offsets, n_overflow, stream);
}

// Second half of a split step: the per-image buckets are already in `workspace` (left there by
// yb_loss_decode_nms_fused called with out_offsets == NULL).
extern "C" int yb_decode_nms_finish(const void* const* preds, int64_t n_img, const yb_decode_params* p,
                                    double nms_threshold, int iou_mode, int rows_per_img_cap, double* out_rows,
                                    int64_t out_capacity, int64_t* out_offsets, unsigned int* n_overflow,
                                    void* workspace, size_t workspace_bytes, yb_stream_t stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    if (out_offsets == nullptr || workspace == nullptr) return YB_E_NULL;
    if (out_rows == nullptr && out_capacity > 0) return YB_E_NULL;
    if (out_capacity < 0) return YB_E_CAPACITY;
    if (iou_mode != 1 && iou_mode != 2) return YB_E_PARAM;
    DecodeLaunch D;
    FusedWs W;
    const int rc = fused_setup(preds, n_img, p, rows_per_img_cap, workspace, workspace_bytes, D, W);
    if (rc != YB_OK || n_img == 0) return rc;
    return fused_launch(D, W, rows_per_img_cap, nms_threshold, iou_mode, out_rows, out_capacity,
                        reinterpret_cast<long long*>(out_offsets), n_overflow, stream);
}
