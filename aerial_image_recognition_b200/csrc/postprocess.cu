// K4 / K4' / K5 / K6 -- everything between the raw head maps and georeferenced detections.
//
//   decode      v8: DFL softmax-expectation + anchor decode + sigmoid (Ultralytics Detect [EXT],
//                   SURVEY.md section 8a row a5);  v7: in-graph sigmoid/grid/anchor decode (Appendix A.4).
//   filter      `boxes[boxes[:,4] >= thr]`           simple_detector.py:479-481, :672-673;
//                                                    _script/gpu_handler.py:166-170 (top-10 at :173)
//   select      per-tile ordering + (optional) greedy IoU-NMS with Ultralytics' arithmetic
//               (class-offset boxes, suppress iff IoU > thr, max_det)  -- `model(window)` at
//               x_arch/02_analyze_images:1 (cell 6)
//   georef      pixel centre -> lon/lat or CRS metres in fp64 without FMA contraction:
//               simple_detector.py:484-502, _script/gpu_handler.py:178-190, pixel_to_geo
//
// Layout: head maps are NHWC fp32 so one anchor's logits are contiguous; the decode kernels give
// each anchor to 4 lanes (one per box side) so a warp reads 8 anchors x 256 B = 2 KB contiguous.
// Candidates are compacted with warp ballots + one atomic per warp; determinism comes from the
// per-tile sort in `select` (key = confidence, anchor index), never from arrival order.
#include "common.cuh"

#include <math.h>

namespace {

__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

// ---- v8: one anchor handled by 4 consecutive lanes; returns the decoded row on every lane ----
struct Row { float cx, cy, w, h, conf; int cls; };

__device__ __forceinline__ float dfl_side(const float* p) {
    float v[16];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float4 q = __ldg((const float4*)p + j);
        v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w;
    }
    float m = v[0];
#pragma unroll
    for (int j = 1; j < 16; ++j) m = fmaxf(m, v[j]);
    float s = 0.f, e = 0.f;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const float t = expf(v[j] - m);
        s += t;
        e += t * (float)j;
    }
    return e / s;
}

__device__ __forceinline__ bool passes(float conf, float thr, int inclusive) { return inclusive ? (conf >= thr) : (conf > thr); }

// The pyramid level of head row `a`: rows are numbered level by level
__device__ __forceinline__ const HeadLevel& head_level(const HeadDesc& h, int a, bool in_range) {
    int lvl = 0;
    if (in_range) { while (lvl + 1 < h.nlevels && a >= h.lv[lvl + 1].row0) ++lvl; }
    return h.lv[lvl];
}

// v8 anchor `a` (DFL and OBB heads): its grid cell and its logits in the NHWC map of its level
struct V8Anchor { const float* pix; int gx, gy; float stride; };

__device__ __forceinline__ V8Anchor v8_anchor(const HeadDesc& h, int tile, int a, bool in_range) {
    const HeadLevel& L = head_level(h, a, in_range);
    const int cell = in_range ? a - L.row0 : 0;
    V8Anchor v;
    v.gy = cell / L.hw; v.gx = cell - v.gy * L.hw;
    v.pix = L.buf + ((size_t)tile * L.hw * L.hw + cell) * L.c;
    v.stride = (float)L.stride;
    return v;
}

// Best class, the threshold (MODE 1) and the DFL distances l, t, r, b of a v8 anchor, whose 4 lanes decode one side each and
// then gather all four.  Returns false, on every lane, when no anchor of the warp is wanted: the caller leaves.
template <int MODE>
__device__ __forceinline__ bool v8_sides(const float* pix, int nc, bool in_range, float thr, int inclusive, float scale, float* conf,
                                         int* cls, bool* want, float* ltrb) {
    float best = 0.f;
    int bi = 0;
    *want = in_range;
    if (in_range) {
        best = -1.f;
        for (int k = 0; k < nc; ++k) {
            const float s = sigmoid_f(__ldg(pix + 64 + k));
            if (s > best) { best = s; bi = k; }
        }
        if (MODE == 1) { best = __fmul_rn(best, scale); *want = passes(best, thr, inclusive); }   // scale: gpu_handler.py:236-238
    }
    *conf = best; *cls = bi;
    // the 4 lanes of an anchor agree on `want`; decode only where some anchor of the warp needs it
    if (__ballot_sync(0xffffffffu, *want) == 0) return false;
    const int side = threadIdx.x & 3, base_lane = (threadIdx.x & 31) & ~3;
    const float d = *want ? dfl_side(pix + side * 16) : 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) ltrb[k] = __shfl_sync(0xffffffffu, d, base_lane + k);
    return true;
}

// dist2bbox: the anchor point minus (l, t) and plus (r, b), as centre and size in pixels
__device__ __forceinline__ Row v8_box(const float* ltrb, int gx, int gy, float stride) {
    const float ax = (float)gx + 0.5f, ay = (float)gy + 0.5f;
    const float x1 = __fsub_rn(ax, ltrb[0]), y1 = __fsub_rn(ay, ltrb[1]), x2 = __fadd_rn(ax, ltrb[2]), y2 = __fadd_rn(ay, ltrb[3]);
    Row o;
    o.cx = __fmul_rn(__fmul_rn(__fadd_rn(x1, x2), 0.5f), stride);
    o.cy = __fmul_rn(__fmul_rn(__fadd_rn(y1, y2), 0.5f), stride);
    o.w = __fmul_rn(__fsub_rn(x2, x1), stride);
    o.h = __fmul_rn(__fsub_rn(y2, y1), stride);
    o.conf = 0.f; o.cls = 0;
    return o;
}

// ---- v7: one thread per (anchor box, cell) ------------------------------------------------------
__device__ __forceinline__ Row v7_row(const float* cell, int nc, int gx, int gy, float stride, float aw, float ah) {
    Row o;
    const float sx = sigmoid_f(__ldg(cell + 0)), sy = sigmoid_f(__ldg(cell + 1));
    const float sw = sigmoid_f(__ldg(cell + 2)), sh = sigmoid_f(__ldg(cell + 3));
    o.cx = __fmul_rn(__fadd_rn(__fsub_rn(__fmul_rn(sx, 2.0f), 0.5f), (float)gx), stride);
    o.cy = __fmul_rn(__fadd_rn(__fsub_rn(__fmul_rn(sy, 2.0f), 0.5f), (float)gy), stride);
    const float tw = __fmul_rn(sw, 2.0f), th = __fmul_rn(sh, 2.0f);
    o.w = __fmul_rn(__fmul_rn(tw, tw), aw);
    o.h = __fmul_rn(__fmul_rn(th, th), ah);
    o.conf = sigmoid_f(__ldg(cell + 4));
    float best = -1.f; int bi = 0;
    for (int k = 0; k < nc; ++k) {
        const float s = sigmoid_f(__ldg(cell + 5 + k));
        if (s > best) { best = s; bi = k; }
    }
    o.cls = bi;
    return o;
}

// Warp-aggregated append to a tile's candidate list: one atomicAdd per warp, slots in lane order.  Every lane of the warp must
// call it, converged (full-mask ballot and shuffle).  Returns the lane's slot, or -1 when it does not emit or the list is full.
__device__ __forceinline__ int append_candidate(bool emit, int& cand_count, int cand_cap) {
    const unsigned em = __ballot_sync(0xffffffffu, emit);
    if (!em) return -1;
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(em) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(&cand_count, __popc(em));
    base = __shfl_sync(0xffffffffu, base, leader);
    const int slot = base + __popc(em & ((1u << lane) - 1));
    return emit && slot < cand_cap ? slot : -1;
}

// Shared body: MODE 0 = dense rows, MODE 1 = thresholded candidates.
template <int MODE>
__global__ void __launch_bounds__(256) head_kernel(HeadDesc h, float thr, int inclusive, float scale, float* rows, b2d_det* cand,
                                                   int* cand_count, int cand_cap) {
    const int tile = blockIdx.y;
    int a;
    bool out;       // this lane stores anchor a's row (MODE 0) or emits it as a candidate (MODE 1)
    Row r;
    if (h.kind == B2D_HEAD_V8_DFL) {
        a = (blockIdx.x * blockDim.x + threadIdx.x) >> 2;    // 4 lanes per anchor, one per box side
        const bool in_range = a < h.rows_total;
        const V8Anchor v = v8_anchor(h, tile, a, in_range);
        float conf, ltrb[4]; int cls; bool want;
        if (!v8_sides<MODE>(v.pix, h.nc, in_range, thr, inclusive, scale, &conf, &cls, &want, ltrb)) return;
        r = v8_box(ltrb, v.gx, v.gy, v.stride);
        r.conf = conf; r.cls = cls;
        out = want && (threadIdx.x & 3) == 0;
    } else {
        a = blockIdx.x * blockDim.x + threadIdx.x;   // row index inside the tile
        const bool in_range = a < h.rows_total;
        const HeadLevel& L = head_level(h, a, in_range);
        const int no = h.nc + 5;
        const int rel = in_range ? a - L.row0 : 0;
        const int cells = L.hw * L.hw;
        const int ai = rel / cells, cell = rel - ai * cells;     // rows ordered anchor, y, x inside a level
        const int gy = cell / L.hw, gx = cell - gy * L.hw;
        r.conf = -1.f;
        if (in_range) {
            const float* p = L.buf + ((size_t)tile * cells + cell) * L.c + ai * no;
            r = v7_row(p, h.nc, gx, gy, (float)L.stride, L.anchors[2 * ai], L.anchors[2 * ai + 1]);
            if (MODE == 1) r.conf = __fmul_rn(r.conf, scale);
        }
        out = in_range && (MODE == 0 || passes(r.conf, thr, inclusive));
    }
    if (MODE == 0) {
        if (out) {
            float* o = rows + ((size_t)tile * h.rows_total + a) * 6;
            o[0] = r.cx; o[1] = r.cy; o[2] = r.w; o[3] = r.h; o[4] = r.conf; o[5] = (float)r.cls;
        }
    } else {
        const int slot = append_candidate(out, cand_count[tile], cand_cap);
        if (slot >= 0) {
            b2d_det d;
            d.cx = r.cx; d.cy = r.cy; d.w = r.w; d.h = r.h; d.conf = r.conf; d.cls = r.cls; d.tile = tile; d.anchor = a;
            cand[(size_t)tile * cand_cap + slot] = d;
        }
    }
}

// candidates from already-decoded rows [n][num_rows][ncol]
__global__ void __launch_bounds__(256) rows_filter_kernel(const float* __restrict__ rows, int num_rows, int ncol, float thr,
                                                           int inclusive, float scale, b2d_det* cand, int* cand_count, int cand_cap) {
    const int tile = blockIdx.y;
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_range = a < num_rows;
    const float* p = rows + ((size_t)tile * num_rows + (in_range ? a : 0)) * ncol;
    const float conf = in_range ? __fmul_rn(__ldg(p + 4), scale) : -1.f;
    const int slot = append_candidate(in_range && passes(conf, thr, inclusive), cand_count[tile], cand_cap);
    if (slot >= 0) {
        b2d_det d;
        d.cx = __ldg(p); d.cy = __ldg(p + 1); d.w = __ldg(p + 2); d.h = __ldg(p + 3); d.conf = conf;
        d.cls = (ncol > 5) ? (int)__ldg(p + 5) : 0;
        d.tile = tile; d.anchor = a;
        cand[(size_t)tile * cand_cap + slot] = d;
    }
}

// ---- select: per-tile sort (+ NMS) ----------------------------------------------------------------
constexpr int kSelCand = 256;                     // candidates per NMS chunk
constexpr int kSelParts = 4;                      // thread groups sharing a chunk's work (= 64-bit words of a suppression mask)
constexpr int kSelThreads = kSelCand * kSelParts;
static_assert(kSelParts == kSelCand / 64, "one part per mask word");
constexpr int kMaxDet = 512;

__device__ void bitonic_sort(unsigned long long* keys, int n2) {
    for (int k = 2; k <= n2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n2; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = keys[i], b = keys[ixj];
                    const bool up = ((i & k) == 0);
                    if ((a > b) == up) { keys[i] = b; keys[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
}

__device__ __forceinline__ bool iou_gt(const float4& a, float aa, const float4& b, float ab, float thr) {
    // torchvision nms arithmetic: inter / (area_a + area_b - inter) > thr, fp32, no contraction.  Disjoint boxes (the common
    // case) leave before the division: there torchvision computes 0 / union = 0 (or 0 / 0 = NaN), never > thr for thr > 0.
    const float w = __fsub_rn(fminf(a.z, b.z), fmaxf(a.x, b.x));
    if (!(w > 0.f)) return false;
    const float h = __fsub_rn(fminf(a.w, b.w), fmaxf(a.y, b.y));
    if (!(h > 0.f)) return false;
    const float inter = __fmul_rn(w, h);
    const float ovr = __fdiv_rn(inter, __fsub_rn(__fadd_rn(aa, ab), inter));
    return ovr > thr;
}

// Sort kernel: one CTA of 1024 threads per tile builds the 64-bit keys (conf desc, anchor asc | row order), sorts them and
// leaves the sorted list in the scratch.  2048 .. 16384 keys (the usual case: 8400 anchors) are sorted with the keys in
// registers -- element i = m * 1024 + tid lives in r[m]; exchange distances >= 1024 stay inside a thread, distances < 32 are
// warp shuffles, only 32 <= j < 1024 goes through shared memory (35 block-wide steps instead of 105 at 16384 keys).  Smaller
// lists are sorted in shared memory, larger ones in the global scratch.
constexpr int kSortThreads = 1024;
constexpr int kSortSmemKeys = 16384;

// Key of candidate slot i: high word = confidence, descending; low word = anchor (16 bits) | slot (16 bits).  The confidence is
// mapped to an unsigned that orders like the float (negatives: all bits flipped; the rest: sign bit set), after -0.0 became +0.0
// so the two zeros tie, and complemented so that the ascending sort gives descending confidence.  Anchors are unique in a tile,
// so equal confidences keep anchor order.  Needs anchors and slots < kMaxCand (ensure_cand refuses larger tiles).
__device__ __forceinline__ unsigned long long sort_key(const b2d_det* tc, int i, int cnt, int by_conf) {
    if (i >= cnt) return ~0ull;
    const unsigned long long lo = ((unsigned long long)((unsigned)tc[i].anchor & 0xFFFFu) << 16) | (unsigned)(i & 0xFFFF);
    if (!by_conf) return lo;                                                                // row order
    const unsigned u = __float_as_uint(__fadd_rn(tc[i].conf, 0.0f));
    const unsigned ordered = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return ((unsigned long long)(~ordered) << 32) | lo;                                    // conf desc, anchor asc
}

// The candidate slot a sorted key refers to
__device__ __forceinline__ int key_slot(unsigned long long key) { return (int)(key & 0xFFFFu); }

template <int KPT>
__device__ void bitonic_sort_regs(const b2d_det* tc, int cnt, int by_conf, unsigned long long* smem, unsigned long long* out) {
    constexpr int N2 = KPT * kSortThreads;
    const int tid = threadIdx.x;
    unsigned long long r[KPT];
#pragma unroll
    for (int m = 0; m < KPT; ++m) r[m] = sort_key(tc, m * kSortThreads + tid, cnt, by_conf);
    for (int k = 2; k <= N2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= kSortThreads) {
#pragma unroll
                for (int d = KPT / 2; d >= 1; d >>= 1) {
                    if (j == d * kSortThreads) {
#pragma unroll
                        for (int m = 0; m < KPT; ++m) {
                            if ((m & d) == 0) {
                                const bool up = (((m * kSortThreads + tid) & k) == 0);
                                const unsigned long long a = r[m], b = r[m | d];
                                if ((a > b) == up) { r[m] = b; r[m | d] = a; }
                            }
                        }
                    }
                }
            } else if (j >= 32) {
#pragma unroll
                for (int m = 0; m < KPT; ++m) smem[m * kSortThreads + tid] = r[m];
                __syncthreads();
#pragma unroll
                for (int m = 0; m < KPT; ++m) {
                    const int i = m * kSortThreads + tid;
                    const unsigned long long o = smem[i ^ j];
                    const bool take_min = (((i & k) == 0) == ((i & j) == 0));     // ascending run: the lower index keeps the minimum
                    r[m] = take_min ? (r[m] < o ? r[m] : o) : (r[m] > o ? r[m] : o);
                }
                __syncthreads();
            } else {
#pragma unroll
                for (int m = 0; m < KPT; ++m) {
                    const int i = m * kSortThreads + tid;
                    const unsigned long long o = __shfl_xor_sync(0xffffffffu, r[m], j);
                    const bool take_min = (((i & k) == 0) == ((i & j) == 0));
                    r[m] = take_min ? (r[m] < o ? r[m] : o) : (r[m] > o ? r[m] : o);
                }
            }
        }
    }
#pragma unroll
    for (int m = 0; m < KPT; ++m) {
        const int i = m * kSortThreads + tid;
        if (i < cnt) out[i] = r[m];
    }
}

__global__ void __launch_bounds__(kSortThreads) sort_keys_kernel(const b2d_det* __restrict__ cand, const int* __restrict__ cand_count,
                                                                  int cand_cap, unsigned long long* keys_scratch, int keys_stride,
                                                                  int by_conf) {
    extern __shared__ unsigned long long dkeys[];
    const int tile = blockIdx.x;
    int cnt = cand_count[tile];
    if (cnt > cand_cap) cnt = cand_cap;
    if (cnt == 0) return;
    const b2d_det* tc = cand + (size_t)tile * cand_cap;
    int n2 = 1;
    while (n2 < cnt) n2 <<= 1;
    unsigned long long* out = keys_scratch + (size_t)tile * keys_stride;
    switch (n2) {
        case 2048: bitonic_sort_regs<2>(tc, cnt, by_conf, dkeys, out); return;
        case 4096: bitonic_sort_regs<4>(tc, cnt, by_conf, dkeys, out); return;
        case 8192: bitonic_sort_regs<8>(tc, cnt, by_conf, dkeys, out); return;
        case 16384: bitonic_sort_regs<16>(tc, cnt, by_conf, dkeys, out); return;
        default: break;
    }
    unsigned long long* keys = (n2 <= kSortSmemKeys) ? dkeys : out;
    for (int i = threadIdx.x; i < n2; i += blockDim.x) keys[i] = sort_key(tc, i, cnt, by_conf);
    __syncthreads();
    bitonic_sort(keys, n2);
    if (keys != out)
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) out[i] = keys[i];
}

// No NMS: the first min(cnt, top_k, cap) candidates in key order, each slot s converted by rec(s)
template <class Out, class Rec>
__device__ __forceinline__ void copy_top_k(const unsigned long long* keys, int cnt, int top_k, int cap, Out* to, int* out_count, Rec rec) {
    int m = cnt;
    if (top_k > 0 && m > top_k) m = top_k;
    if (m > cap) m = cap;
    for (int i = threadIdx.x; i < m; i += blockDim.x) to[i] = rec(key_slot(keys[i]));
    if (threadIdx.x == 0) *out_count = m;
}

__global__ void __launch_bounds__(kSelThreads) select_kernel(const b2d_det* __restrict__ cand, const int* __restrict__ cand_count,
                                                              int cand_cap, const unsigned long long* __restrict__ keys_scratch, int keys_stride,
                                                              float iou_thr, int top_k, int max_det, b2d_det* out, int* out_count,
                                                              int cap) {
    __shared__ float4 kbox[kMaxDet];
    __shared__ float karea[kMaxDet];
    __shared__ float4 cbox[kSelCand];
    __shared__ float carea[kSelCand];
    __shared__ unsigned long long cmask[kSelCand][kSelCand / 64];
    __shared__ unsigned int alive_w[kSelCand / 32];
    __shared__ int keep_slot[kSelCand];
    __shared__ int dead[kSelCand];
    __shared__ int s_nk;

    const int tile = blockIdx.x;
    const int tid = threadIdx.x;
    int cnt = cand_count[tile];
    if (cnt > cand_cap) cnt = cand_cap;
    const b2d_det* tc = cand + (size_t)tile * cand_cap;
    b2d_det* to = out + (size_t)tile * cap;
    if (cnt == 0) {
        if (tid == 0) out_count[tile] = 0;
        return;
    }
    const unsigned long long* keys = keys_scratch + (size_t)tile * keys_stride;     // sorted by sort_keys_kernel

    if (!(iou_thr > 0.f)) {
        copy_top_k(keys, cnt, top_k, cap, to, &out_count[tile], [&](int s) { return tc[s]; });
        return;
    }

    // ---- greedy NMS over the sorted list, 256 candidates at a time ----
    // One tile has one CTA, so the work of a chunk is spread over four thread groups ("parts") of 256: part p tests candidate c
    // against the kept boxes k = p, p + 4, ... and builds word p of c's suppression mask.
    if (max_det > cap) max_det = cap;                       // max_det <= kMaxDet is checked by select_launch
    if (cnt > kMaxNms) cnt = kMaxNms;                       // Ultralytics' max_nms cut of the sorted list
    const int c = tid & (kSelCand - 1), part = tid / kSelCand;
    if (tid == 0) s_nk = 0;
    __syncthreads();
    for (int base = 0; base < cnt; base += kSelCand) {
        const int nk = s_nk;
        if (nk >= max_det) break;
        const int i = base + c;
        const bool valid = i < cnt;
        b2d_det d;
        float4 bx = make_float4(0.f, 0.f, 0.f, 0.f);
        float ar = 0.f;
        if (valid) {
            d = tc[key_slot(keys[i])];
            // xywh2xyxy then + cls * max_wh, as Ultralytics
            const float hw = __fmul_rn(d.w, 0.5f), hh = __fmul_rn(d.h, 0.5f);
            const float off = __fmul_rn((float)d.cls, 7680.0f);
            bx.x = __fadd_rn(__fsub_rn(d.cx, hw), off);
            bx.y = __fadd_rn(__fsub_rn(d.cy, hh), off);
            bx.z = __fadd_rn(__fadd_rn(d.cx, hw), off);
            bx.w = __fadd_rn(__fadd_rn(d.cy, hh), off);
            ar = __fmul_rn(__fsub_rn(bx.z, bx.x), __fsub_rn(bx.w, bx.y));
        }
        if (part == 0) {
            cbox[c] = bx;
            carea[c] = ar;
            dead[c] = valid ? 0 : 1;
            keep_slot[c] = -1;
        }
        __syncthreads();
        if (valid) {
            for (int k = part; k < nk; k += kSelParts)
                if (iou_gt(kbox[k], karea[k], bx, ar, iou_thr)) { dead[c] = 1; break; }
        }
        __syncthreads();
        const bool alive = dead[c] == 0;
        if (part == 0) {
            const unsigned al = __ballot_sync(0xffffffffu, alive);
            if ((c & 31) == 0) alive_w[c >> 5] = al;
        }
        __syncthreads();
        // which later, still alive candidates of this chunk does `c` suppress?  (dead rows and dead columns are skipped:
        // after the test against the kept boxes most of a chunk is already gone)
        {
            const int w = part;
            unsigned long long m = 0;
            if (alive) {
                unsigned long long am = ((unsigned long long)alive_w[2 * w + 1] << 32) | (unsigned long long)alive_w[2 * w];
                if (w * 64 <= c) am &= (c - w * 64 >= 63) ? 0ull : (~0ull << (c - w * 64 + 1));      // only j > c
                while (am) {
                    const int jj = __ffsll((long long)am) - 1;
                    am &= am - 1;
                    const int j = w * 64 + jj;
                    if (iou_gt(bx, ar, cbox[j], carea[j], iou_thr)) m |= (1ull << jj);
                }
            }
            cmask[c][w] = m;
        }
        __syncthreads();
        if (tid == 0) {
            unsigned long long removed[kSelCand / 64] = {0, 0, 0, 0};
            int k = nk;
#pragma unroll
            for (int w = 0; w < kSelCand / 64; ++w) {
                unsigned long long am = ((unsigned long long)alive_w[2 * w + 1] << 32) | (unsigned long long)alive_w[2 * w];
                while (k < max_det) {
                    am &= ~removed[w];
                    if (!am) break;
                    const int jj = __ffsll((long long)am) - 1;
                    am &= ~(1ull << jj);
                    const int j = w * 64 + jj;
                    keep_slot[j] = k++;
#pragma unroll
                    for (int v = 0; v < kSelCand / 64; ++v) removed[v] |= cmask[j][v];
                }
            }
            s_nk = k;
        }
        __syncthreads();
        if (part == 0) {
            const int slot = keep_slot[c];
            if (slot >= 0) {
                kbox[slot] = bx;
                karea[slot] = ar;
                to[slot] = d;
            }
        }
        __syncthreads();
    }
    if (tid == 0) out_count[tile] = s_nk;
}

// ---- georef -------------------------------------------------------------------------------------
// Bounds form, simple_detector.py:487-494 -- P = west, east, south, north, crop_size, model_size: model pixel (x, y) -> lon / lat
__device__ __forceinline__ double geo_model_size(const double* P) { return P[5] > 0.0 ? P[5] : 640.0; }

__device__ __forceinline__ void geo_bounds(const double* P, double x, double y, double* gx, double* gy) {
    const double ms = geo_model_size(P);
    const double xf = __ddiv_rn(x, ms), yf = __ddiv_rn(y, ms);
    *gx = __dadd_rn(P[0], __dmul_rn(xf, __dsub_rn(P[1], P[0])));
    *gy = __dsub_rn(P[3], __dmul_rn(yf, __dsub_rn(P[3], P[2])));
}

// 6-term geotransform P[0..5] of the window-relative pixel (X, Y)
__device__ __forceinline__ void geo_affine(const double* P, double X, double Y, double* gx, double* gy) {
    *gx = __dadd_rn(__dadd_rn(P[0], __dmul_rn(X, P[1])), __dmul_rn(Y, P[2]));
    *gy = __dadd_rn(__dadd_rn(P[3], __dmul_rn(X, P[4])), __dmul_rn(Y, P[5]));
}

__global__ void __launch_bounds__(256) georef_kernel(const b2d_det* __restrict__ dets, const int* __restrict__ counts, int cap, int mode,
                                                      const double* __restrict__ params, b2d_geodet* __restrict__ out) {
    const int tile = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= counts[tile] || i >= cap) return;
    const b2d_det d = dets[(size_t)tile * cap + i];
    const double* P = params + (size_t)tile * B2D_GEO_PARAMS;
    b2d_geodet g;
    g.conf = d.conf; g.tile = tile; g.x_yolo = d.cx; g.y_yolo = d.cy; g.x_img = 0.f; g.y_img = 0.f;
    const double x = (double)d.cx, y = (double)d.cy;
    if (mode == B2D_GEO_BOUNDS) {
        const double ms = geo_model_size(P);
        g.x_img = (float)__dmul_rn(__ddiv_rn(x, ms), P[4]);
        g.y_img = (float)__dmul_rn(__ddiv_rn(y, ms), P[4]);
        geo_bounds(P, x, y, &g.x, &g.y);
    } else if (mode == B2D_GEO_GPUHANDLER) {
        // gpu_handler.py:182-190 -- P = lon_min, lat_min, lon_max, lat_max; keeps the *864/864 round trip
        const double x864 = __dmul_rn(__ddiv_rn(x, 640.0), 864.0), y864 = __dmul_rn(__ddiv_rn(y, 640.0), 864.0);
        g.x_img = (float)x864; g.y_img = (float)y864;
        g.x = __dadd_rn(P[0], __dmul_rn(__ddiv_rn(x864, 864.0), __dsub_rn(P[2], P[0])));
        g.y = __dsub_rn(P[3], __dmul_rn(__ddiv_rn(y864, 864.0), __dsub_rn(P[3], P[1])));
    } else if (mode == B2D_GEO_TENSOR_F32) {
        // gpu_handler.py:243-253 (_process_tensors): float32 CUDA-tensor arithmetic.  `boxes[:, :2] / 640` on a CUDA tensor is a
        // multiplication by the float reciprocal of the scalar; the Python scalars are cast to float32.  P = lon_min, lat_min,
        // lon_max, lat_max.
        const float inv = __fdiv_rn(1.0f, 640.0f);
        const float cxn = __fmul_rn(d.cx, inv), cyn = __fmul_rn(d.cy, inv);
        const float lon_off = (float)__dsub_rn(P[2], P[0]), lat_off = (float)__dsub_rn(P[3], P[1]);
        g.x = (double)__fadd_rn((float)P[0], __fmul_rn(cxn, lon_off));
        g.y = (double)__fsub_rn((float)P[3], __fmul_rn(cyn, lat_off));
    } else {
        // Ultralytics scale_boxes (fp32) then the notebook's centroid + pixel_to_geo (fp64)
        // P = gt[0..5], win_x, win_y, pad_x, pad_y, gain, w0, h0
        const float hw = __fmul_rn(d.w, 0.5f), hh = __fmul_rn(d.h, 0.5f);
        float x1 = __fsub_rn(d.cx, hw), y1 = __fsub_rn(d.cy, hh), x2 = __fadd_rn(d.cx, hw), y2 = __fadd_rn(d.cy, hh);
        const float px = (float)P[8], py = (float)P[9], gain = (float)P[10], w0 = (float)P[11], h0 = (float)P[12];
        x1 = __fdiv_rn(__fsub_rn(x1, px), gain); x2 = __fdiv_rn(__fsub_rn(x2, px), gain);
        y1 = __fdiv_rn(__fsub_rn(y1, py), gain); y2 = __fdiv_rn(__fsub_rn(y2, py), gain);
        x1 = fminf(fmaxf(x1, 0.f), w0); x2 = fminf(fmaxf(x2, 0.f), w0);
        y1 = fminf(fmaxf(y1, 0.f), h0); y2 = fminf(fmaxf(y2, 0.f), h0);
        // (x1 + x2) is an fp32 add; "/ 2" and "+= x" promote to float64 under the reference's NumPy 1.26
        const double cxp = __dadd_rn(__ddiv_rn((double)__fadd_rn(x1, x2), 2.0), P[6]);
        const double cyp = __dadd_rn(__ddiv_rn((double)__fadd_rn(y1, y2), 2.0), P[7]);
        g.x_img = (float)cxp; g.y_img = (float)cyp;
        geo_affine(P, cxp, cyp, &g.x, &g.y);
    }
    out[(size_t)tile * cap + i] = g;
}

// ---- oriented boxes (yolov8m-obb): Ultralytics >= 8.1 OBB head, rotated NMS, corner georeferencing [EXT] ----------------
// Decode = OBB.forward + dist2rbox: theta = (sigmoid(z) - 0.25) pi, the DFL half-differences rotated by theta around the anchor.
// Every step is the restated fp32 arithmetic, one rounding per torch op (__f*_rn: no contraction), precise expf / sincosf.
constexpr float kPiF = 3.14159265358979f;           // float(math.pi), the scalar of the torch expressions
constexpr float kHalfPiF = 1.57079632679490f;       // float(math.pi / 2)
constexpr float kProbEps = 1e-7f;

// MODE 0 = dense rows [n][A][7] (cx, cy, w, h, conf, cls, theta); MODE 1 = thresholded candidates + their angles
template <int MODE>
__global__ void __launch_bounds__(256) obb_head_kernel(HeadDesc h, float thr, int inclusive, float scale, float* rows, b2d_det* cand,
                                                       float* cand_angle, int* cand_count, int cand_cap) {
    const int tile = blockIdx.y;
    const int a = (blockIdx.x * blockDim.x + threadIdx.x) >> 2;        // 4 lanes per anchor, one per box side
    const int side = threadIdx.x & 3;
    const bool in_range = a < h.rows_total;
    const V8Anchor v = v8_anchor(h, tile, a, in_range);
    float conf, ltrb[4]; int cls; bool want;
    if (!v8_sides<MODE>(v.pix, h.nc, in_range, thr, inclusive, scale, &conf, &cls, &want, ltrb)) return;
    const float l = ltrb[0], t = ltrb[1], r = ltrb[2], b = ltrb[3];
    if (!want || side != 0) {
        if (MODE == 0) return;
    }
    float cx = 0.f, cy = 0.f, w = 0.f, hh = 0.f, th = 0.f;
    if (want && side == 0) {
        th = __fmul_rn(__fsub_rn(sigmoid_f(__ldg(v.pix + obb_angle_channel(h.nc))), 0.25f), kPiF);
        float sn, cs;
        sincosf(th, &sn, &cs);
        const float xf = __fdiv_rn(__fsub_rn(r, l), 2.0f), yf = __fdiv_rn(__fsub_rn(b, t), 2.0f);
        const float x = __fsub_rn(__fmul_rn(xf, cs), __fmul_rn(yf, sn));
        const float y = __fadd_rn(__fmul_rn(xf, sn), __fmul_rn(yf, cs));
        const float s = v.stride;
        cx = __fmul_rn(__fadd_rn(x, (float)v.gx + 0.5f), s);
        cy = __fmul_rn(__fadd_rn(y, (float)v.gy + 0.5f), s);
        w = __fmul_rn(__fadd_rn(l, r), s);
        hh = __fmul_rn(__fadd_rn(t, b), s);
    }
    if (MODE == 0) {
        float* o = rows + ((size_t)tile * h.rows_total + a) * 7;
        o[0] = cx; o[1] = cy; o[2] = w; o[3] = hh; o[4] = conf; o[5] = (float)cls; o[6] = th;
        return;
    }
    const int slot = append_candidate(want && side == 0, cand_count[tile], cand_cap);
    if (slot >= 0) {
        b2d_det d;
        d.cx = cx; d.cy = cy; d.w = w; d.h = hh; d.conf = conf; d.cls = cls; d.tile = tile; d.anchor = a;
        cand[(size_t)tile * cand_cap + slot] = d;
        cand_angle[(size_t)tile * cand_cap + slot] = th;
    }
}

// regularize_rboxes: w >= h, theta in [0, pi) -- torch's `%` on floats is fmod with the sign of the divisor
__device__ __forceinline__ b2d_obb obb_record(const b2d_det& d, float th) {
    b2d_obb o;
    o.cx = d.cx; o.cy = d.cy;
    const bool keep = d.w > d.h;
    o.w = keep ? d.w : d.h;
    o.h = keep ? d.h : d.w;
    const float t = keep ? th : __fadd_rn(th, kHalfPiF);
    float md = fmodf(t, kPiF);
    if (md != 0.f && md < 0.f) md = __fadd_rn(md, kPiF);
    o.theta = md;
    o.conf = d.conf; o.cls = d.cls; o.tile = d.tile; o.anchor = d.anchor;
    return o;
}

// ProbIoU fast NMS, one CTA per tile.  Phase 1 turns every sorted candidate (at most kMaxNms, Ultralytics' max_nms) into its
// Gaussian once -- class-offset centre, covariance (A, B, C) and P = max(A B - C^2, 0) of the log term -- in global scratch.
// Phase 2 walks the candidates in blocks of 1024: thread j tests the earlier candidates i < j, staged chunk by chunk through
// shared memory, and leaves at its first suppressor (fast NMS: a suppressed box still suppresses, so the tests are independent and
// there is no serial keep scan).  Survivors are compacted in order; the walk stops when max_det are kept.  No pair is skipped.
constexpr int kObbThreads = 1024;

// batch_probiou's Gaussian of a box (_get_covariance_matrix): a = w^2 / 12, b = h^2 / 12, A = a cos^2 + b sin^2,
// B = a sin^2 + b cos^2, C = (a - b) cos sin, and P = max(A B - C^2, 0) of the log term
struct ObbGauss { float A, B, C, P; };
__device__ __forceinline__ ObbGauss obb_gaussian(float w, float h, float th) {
    const float a = __fdiv_rn(__fmul_rn(w, w), 12.0f), b = __fdiv_rn(__fmul_rn(h, h), 12.0f);
    float sn, cs;
    sincosf(th, &sn, &cs);
    const float c2 = __fmul_rn(cs, cs), s2 = __fmul_rn(sn, sn);
    ObbGauss g;
    g.A = __fadd_rn(__fmul_rn(a, c2), __fmul_rn(b, s2));
    g.B = __fadd_rn(__fmul_rn(a, s2), __fmul_rn(b, c2));
    g.C = __fmul_rn(__fmul_rn(__fsub_rn(a, b), cs), sn);
    g.P = fmaxf(__fsub_rn(__fmul_rn(g.A, g.B), __fmul_rn(g.C, g.C)), 0.f);
    return g;
}

// batch_probiou(obb1 = box i, obb2 = box j) >= thr, from the centre difference (dx, dy) = (x_i - x_j, y_i - y_j) and the two
// Gaussians (A, B, C, P).  batch_probiou's x2 - x1 is -dx, exactly (round-to-nearest is symmetric).
__device__ __forceinline__ bool probiou_suppresses(float dx, float dy, float Ai, float Bi, float Ci, float Pi, float Aj, float Bj,
                                                   float Cj, float Pj, float thr) {
    const float a12 = __fadd_rn(Ai, Aj), b12 = __fadd_rn(Bi, Bj), c12 = __fadd_rn(Ci, Cj);
    const float den = __fsub_rn(__fmul_rn(a12, b12), __fmul_rn(c12, c12));
    const float dene = __fadd_rn(den, kProbEps);
    const float t1 = __fmul_rn(__fdiv_rn(__fadd_rn(__fmul_rn(a12, __fmul_rn(dy, dy)), __fmul_rn(b12, __fmul_rn(dx, dx))), dene), 0.25f);
    const float t2 = __fmul_rn(__fdiv_rn(__fmul_rn(__fmul_rn(c12, -dx), dy), dene), 0.5f);
    const float t3 = __fmul_rn(logf(__fadd_rn(__fdiv_rn(den, __fadd_rn(__fmul_rn(4.0f, __fsqrt_rn(__fmul_rn(Pi, Pj))), kProbEps)), kProbEps)), 0.5f);
    const float bd = fminf(fmaxf(__fadd_rn(__fadd_rn(t1, t2), t3), kProbEps), 100.0f);
    const float hd = __fsqrt_rn(__fadd_rn(__fsub_rn(1.0f, expf(-bd)), kProbEps));
    const float iou = __fsub_rn(1.0f, hd);
    return !(iou < thr);            // kept iff every earlier ProbIoU < thr (a NaN suppresses, as torch's max propagates it)
}

__global__ void __launch_bounds__(kObbThreads) obb_select_kernel(const b2d_det* __restrict__ cand, const float* __restrict__ cand_angle,
                                                                  const int* __restrict__ cand_count, int cand_cap,
                                                                  const unsigned long long* __restrict__ keys_scratch, int keys_stride,
                                                                  float4* __restrict__ prm, float iou_thr, int top_k, int max_det,
                                                                  b2d_obb* __restrict__ out, int* __restrict__ out_count, int cap) {
    __shared__ float4 sp[kObbThreads];
    __shared__ float2 sq[kObbThreads];
    __shared__ int warp_n[kObbThreads / 32];
    __shared__ int s_nk;
    const int tile = blockIdx.x;
    const int tid = threadIdx.x;
    int cnt = cand_count[tile];
    if (cnt > cand_cap) cnt = cand_cap;
    const b2d_det* tc = cand + (size_t)tile * cand_cap;
    const float* ta = cand_angle + (size_t)tile * cand_cap;
    b2d_obb* to = out + (size_t)tile * cap;
    const unsigned long long* keys = keys_scratch + (size_t)tile * keys_stride;
    if (!(iou_thr > 0.f)) {
        copy_top_k(keys, cnt, top_k, cap, to, &out_count[tile], [&](int s) { return obb_record(tc[s], ta[s]); });
        return;
    }
    if (max_det > cap) max_det = cap;
    const int m = cnt < kMaxNms ? cnt : kMaxNms;
    float4* tp = prm + (size_t)tile * keys_stride * 2;
    for (int i = tid; i < m; i += blockDim.x) {
        const int s = key_slot(keys[i]);
        const b2d_det d = tc[s];
        const float off = __fmul_rn((float)d.cls, 7680.0f);
        const ObbGauss g = obb_gaussian(d.w, d.h, ta[s]);
        tp[2 * i] = make_float4(__fadd_rn(d.cx, off), __fadd_rn(d.cy, off), g.A, g.B);
        tp[2 * i + 1] = make_float4(g.C, g.P, 0.f, 0.f);
    }
    if (tid == 0) s_nk = 0;
    __syncthreads();
    for (int jb = 0; jb < m; jb += kObbThreads) {
        const int j = jb + tid;
        bool alive = j < m;
        float4 pj = make_float4(0.f, 0.f, 0.f, 0.f);
        float2 qj = make_float2(0.f, 0.f);
        if (alive) {
            pj = tp[2 * j];
            const float4 q = tp[2 * j + 1];
            qj = make_float2(q.x, q.y);
        }
        for (int ib = 0; ib <= jb; ib += kObbThreads) {
            if (!__syncthreads_or(alive)) break;            // every box of the block already suppressed
            const int i = ib + tid;
            if (i < m) {
                sp[tid] = tp[2 * i];
                const float4 q = tp[2 * i + 1];
                sq[tid] = make_float2(q.x, q.y);
            }
            __syncthreads();
            if (alive) {
                const int end = min(kObbThreads, j - ib);   // i < j
                for (int k = 0; k < end; ++k) {
                    const float4 pi = sp[k];
                    const float2 qi = sq[k];
                    if (probiou_suppresses(__fsub_rn(pi.x, pj.x), __fsub_rn(pi.y, pj.y), pi.z, pi.w, qi.x, qi.y, pj.z, pj.w, qj.x, qj.y,
                                           iou_thr)) { alive = false; break; }
                }
            }
        }
        // compact the survivors of this block in order
        const unsigned bal = __ballot_sync(0xffffffffu, alive);
        if ((tid & 31) == 0) warp_n[tid >> 5] = __popc(bal);
        __syncthreads();
        const int nk = s_nk;
        int before = 0, total = 0;
        for (int w = 0; w < kObbThreads / 32; ++w) {
            const int c = warp_n[w];
            before += (w < (tid >> 5)) ? c : 0;
            total += c;
        }
        if (alive) {
            const int slot = nk + before + __popc(bal & ((1u << (tid & 31)) - 1));
            if (slot < max_det) {
                const int s = key_slot(keys[j]);
                to[slot] = obb_record(tc[s], ta[s]);
            }
        }
        __syncthreads();
        if (tid == 0) s_nk = min(nk + total, max_det);
        __syncthreads();
        if (s_nk >= max_det) break;
    }
    if (tid == 0) out_count[tile] = s_nk;
}

// xywhr2xyxyxyxy in fp32: v1 = (w/2 cos, w/2 sin), v2 = (-h/2 sin, h/2 cos); corners c+v1+v2, c+v1-v2, c-v1-v2, c-v1+v2
__device__ __forceinline__ void obb_corners(float cx, float cy, float w, float h, float th, float* px, float* py) {
    const float sn = sinf(th), cs = cosf(th);
    const float w2 = __fdiv_rn(w, 2.0f), h2 = __fdiv_rn(-h, 2.0f), h2p = __fdiv_rn(h, 2.0f);
    const float v1x = __fmul_rn(w2, cs), v1y = __fmul_rn(w2, sn);
    const float v2x = __fmul_rn(h2, sn), v2y = __fmul_rn(h2p, cs);
    px[0] = __fadd_rn(__fadd_rn(cx, v1x), v2x); py[0] = __fadd_rn(__fadd_rn(cy, v1y), v2y);
    px[1] = __fsub_rn(__fadd_rn(cx, v1x), v2x); py[1] = __fsub_rn(__fadd_rn(cy, v1y), v2y);
    px[2] = __fsub_rn(__fsub_rn(cx, v1x), v2x); py[2] = __fsub_rn(__fsub_rn(cy, v1y), v2y);
    px[3] = __fadd_rn(__fsub_rn(cx, v1x), v2x); py[3] = __fadd_rn(__fsub_rn(cy, v1y), v2y);
}

// B2D_GEO_AFFINE's letterbox undo of an oriented box (Ultralytics scale_boxes without clipping): centre (x - pad) / gain and
// size / gain in fp32, theta unchanged; P = gt[0..5], win_x, win_y, pad_x, pad_y, gain.  The window offset is added in fp64
// by source_px.  obb_georef_kernel and the mosaic merge (mosaic_nms_prep_kernel) both map boxes with these two, so the merged
// boxes and the georeferenced footprints are in one frame.
struct ObbUndo { float cx, cy, w, h; };
__device__ __forceinline__ ObbUndo obb_affine_undo(const b2d_obb& d, const double* P) {
    const float padx = (float)P[8], pady = (float)P[9], gain = (float)P[10];
    ObbUndo u;
    u.cx = __fdiv_rn(__fsub_rn(d.cx, padx), gain);
    u.cy = __fdiv_rn(__fsub_rn(d.cy, pady), gain);
    u.w = __fdiv_rn(d.w, gain);
    u.h = __fdiv_rn(d.h, gain);
    return u;
}
// a window pixel (fp32) in the mosaic's pixel frame: + (win_x, win_y) in fp64
__device__ __forceinline__ double2 source_px(float px, float py, const double* P) {
    return make_double2(__dadd_rn((double)px, P[6]), __dadd_rn((double)py, P[7]));
}

__global__ void __launch_bounds__(256) obb_georef_kernel(const b2d_obb* __restrict__ dets, const int* __restrict__ counts, int cap, int mode,
                                                          const double* __restrict__ params, b2d_geoobb* __restrict__ out) {
    const int tile = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= counts[tile] || i >= cap) return;
    const b2d_obb d = dets[(size_t)tile * cap + i];
    const double* P = params + (size_t)tile * B2D_GEO_PARAMS;
    b2d_geoobb g;
    g.conf = d.conf; g.theta = d.theta; g.cls = d.cls; g.tile = tile;
    float px[5], py[5];
    double gx[5], gy[5];
    if (mode == B2D_GEO_BOUNDS) {
        // the bounds form applied to the centre and to each corner; w, h scaled like x_img (model -> crop pixels)
        obb_corners(d.cx, d.cy, d.w, d.h, d.theta, px, py);
        px[4] = d.cx; py[4] = d.cy;
        const double ms = geo_model_size(P);
        g.w = (float)__dmul_rn(__ddiv_rn((double)d.w, ms), P[4]);
        g.h = (float)__dmul_rn(__ddiv_rn((double)d.h, ms), P[4]);
#pragma unroll
        for (int k = 0; k < 5; ++k) geo_bounds(P, (double)px[k], (double)py[k], &gx[k], &gy[k]);
    } else {
        // affine: undo the letterbox in fp32, corners in fp32, then the window offset and the 6-term geotransform in fp64
        const ObbUndo u = obb_affine_undo(d, P);
        g.w = u.w;
        g.h = u.h;
        obb_corners(u.cx, u.cy, u.w, u.h, d.theta, px, py);
        px[4] = u.cx; py[4] = u.cy;
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            const double2 m = source_px(px[k], py[k], P);
            geo_affine(P, m.x, m.y, &gx[k], &gy[k]);
        }
    }
    g.x = gx[4]; g.y = gy[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { g.corners[2 * k] = gx[k]; g.corners[2 * k + 1] = gy[k]; }
    out[(size_t)tile * cap + i] = g;
}

// ---- mosaic-wide oriented-box merge (b2d_mosaic_nms_obb) -------------------------------------------------------------
// Ultralytics' DOTA slice merge, fast NMS over every window's records in the mosaic's pixel frame: record j is suppressed iff
// an eligible record i of the same class and higher priority (confidence descending, then lower index k = row * cap + slot)
// has ProbIoU(i, j) >= thr.  The fate of j depends on its higher-priority neighbours only, not on theirs, so there is no sort
// and no rounds: keep starts as "eligible", and every examined pair that suppresses stores 0 into the keep byte of its
// lower-priority member.  The store is idempotent and the set of pairs examined does not depend on scheduling, so the result
// is deterministic.  Which pairs must be examined:
//
// A record is REGULAR when X, Y, w', h', theta are finite, |X|, |Y| < 2^31, its short side s = min(w', h') >= 1 px, its
// long side L <= kMnmsAspect s and L <= the grid's reach (below).  For two regular boxes (exact arithmetic first), with
// S = Sigma_i + Sigma_j and d = the centre difference:
//   t1 + t2 = 1/4 d^T S^-1 d * det S / (det S + eps)  >=  |d|^2 / (4 lmax(S)) * (1 - eps / det S),
//   lmax(S) <= lmax(Sigma_i) + lmax(Sigma_j) = (L_i^2 + L_j^2) / 12,
//   det S >= (sqrt det Sigma_i + sqrt det Sigma_j)^2 >= 4 sqrt(P_i P_j)   (Minkowski), so t3 >= 1/2 ln(1 / (1 + eps / (4 sqrt(P_i P_j)))),
// and s >= 1 gives P >= 1/144, det S >= 1/36: eps / det S <= 3.6e-6.  ProbIoU >= thr needs bd <= bd* = -ln(1 + eps - (1 - thr)^2).
// fp32: u = 2^-24, rho = L / s <= 128, so u rho^2 <= 2^-10.  sincosf and the roundings of A, B, C perturb each Sigma by at
// most 16 u a in norm (a = L^2 / 12): its eigenvalues stay in [b (1 - 2^-6), a (1 + 16 u)], b = s^2 / 12, and it stays
// positive definite, so the bounds above hold for the computed Gaussians.  Cancellation is bounded by the condition number
// lmax / lmin <= 1.04 rho^2 of S: den = a12 b12 - c12^2 is within 8 u lmax^2 = 0.9 % of det S, each P within 0.7 %, and
// t1 + t2 (positive t1 against t2 with |t2| <= lmax |d|^2 / (4 dene)) within 15 u lmax / lmin = 1.6 %.  So the computed
//   t1 + t2 >= 0.976 * 3 |d|^2 / (L_i^2 + L_j^2)  and  t3 >= 1/2 ln(0.9919 / 1.0063) - 1 ulp >= -0.0073.
// The computed iou is 1 - sqrt(1 - expf(-bd) + eps) with expf within 2 ulp and the rest correctly rounded; iou >= thr then
// needs bd <= bd_lim = -ln(1 + eps - (1 - thr + 4u)^2 (1 + 2u) - 8u), or bd_lim = 100 where that argument is not positive
// (bd is clamped to 100, where the computed iou is 0 < thr).  Hence a regular pair can only suppress when
//   |d|^2 <= K (L_i^2 + L_j^2),   K = (bd_lim + 1/16) * 17 / 48          (>= (bd_lim + 0.008) / 2.928, the bound above)
// -- at thr 0.3, |d| <= 0.72 max(L_i, L_j) (0.67 without the rounding margins).  The pair is examined by its member with the longer side (ties: the higher index),
// within R = sqrt(2 K) L + 1 px of it (L of the partner <= L, 1 px covers the fp64 rounding of the scan window), over the cells
// of a hashed uniform grid of kMnmsCell px; a box whose R would span more than kMnmsReach cells either side is not regular.
// So one large box among millions of small ones widens its own scan only.
//
// Every other eligible record is IRREGULAR (zero-area, needle, huge, far or non-finite boxes: with eps = 1e-7 two zero-area
// boxes of one class reach ProbIoU 0.9995 at any distance).  They sit in a compacted list, and each is tested against every
// eligible record, the bound being used for none of them: O(D N) for D irregular records.
constexpr double kMnmsCell = 64.0;        // px; a power of two, so X / cell is exact
constexpr int kMnmsReach = 48;            // cells either side of a regular box's own cell
constexpr float kMnmsAspect = 128.f;
constexpr double kMnmsMaxCoord = 2147483648.0;

struct MnmsGrid {
    double2* xy;            // [N] merge-frame centre (eligible records)
    float4* gs;             // [N] Gaussian A, B, C, P (eligible records)
    float* len;             // [N] long side (regular records)
    uint8_t* kind;          // [N] 0 not eligible, 1 regular (in the grid), 2 irregular (in the list)
    int* next;              // [N] next point of the same cell
    int* irr;               // [N] the irregular records, *irr_count of them, in no particular order
    int* irr_count;
    long long* cell_key;    // [cap_mask + 1]
    int* cell_head;
    unsigned cap_mask;
};

__global__ void __launch_bounds__(256) mosaic_nms_prep_kernel(const b2d_obb* __restrict__ dets, const int* __restrict__ counts,
                                                              const double* __restrict__ params, int cap, int total, float conf_thr,
                                                              float max_len, MnmsGrid g, uint8_t* __restrict__ keep) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= total) return;
    const int r = k / cap, s = k - r * cap;
    const b2d_obb d = dets[k];
    const bool eligible = s < counts[r] && d.conf > conf_thr;
    keep[k] = eligible ? 1 : 0;
    if (!eligible) { g.kind[k] = 0; return; }
    const double* P = params + (size_t)r * B2D_GEO_PARAMS;
    const ObbUndo u = obb_affine_undo(d, P);
    const double2 m = source_px(u.cx, u.cy, P);
    const ObbGauss q = obb_gaussian(u.w, u.h, d.theta);
    g.xy[k] = m;
    g.gs[k] = make_float4(q.A, q.B, q.C, q.P);
    const float sh = fminf(u.w, u.h), L = fmaxf(u.w, u.h);
    const bool regular = fabs(m.x) < kMnmsMaxCoord && fabs(m.y) < kMnmsMaxCoord && isfinite(u.w) && isfinite(u.h) &&
                         isfinite(d.theta) && sh >= 1.f && L <= __fmul_rn(kMnmsAspect, sh) && L <= max_len;
    if (regular) {
        g.len[k] = L;
        const long long cx = (long long)floor(m.x * (1.0 / kMnmsCell)), cy = (long long)floor(m.y * (1.0 / kMnmsCell));
        const unsigned slot = cell_claim(g.cell_key, g.cap_mask, pack_cell(cx, cy));
        g.next[k] = atomicExch(&g.cell_head[slot], k);
        g.kind[k] = 1;
    } else {
        g.irr[atomicAdd(g.irr_count, 1)] = k;
        g.kind[k] = 2;
    }
}

// Examine the pair (k, t) of one class: the higher-priority member as batch_probiou's obb1, dx = (float)(X_hi - X_lo)
__device__ __forceinline__ void mnms_pair(const MnmsGrid& g, int k, double2 pk, float4 qk, float ck, int t, float ct, float thr,
                                          uint8_t* keep) {
    const bool k_first = ck > ct || (ck == ct && k < t);
    const int lo = k_first ? t : k;
    if (((volatile uint8_t*)keep)[lo] == 0) return;          // already suppressed: a keep byte never returns to 1
    const double2 pt = g.xy[t];
    const float4 qt = g.gs[t];
    const double2 ph = k_first ? pk : pt, pl = k_first ? pt : pk;
    const float4 qh = k_first ? qk : qt, ql = k_first ? qt : qk;
    if (probiou_suppresses((float)__dsub_rn(ph.x, pl.x), (float)__dsub_rn(ph.y, pl.y), qh.x, qh.y, qh.z, qh.w, ql.x, ql.y, ql.z, ql.w, thr))
        keep[lo] = 0;
}

__global__ void __launch_bounds__(256) mosaic_nms_grid_kernel(const b2d_obb* __restrict__ dets, int total, double reach_coef, float thr,
                                                              MnmsGrid g, uint8_t* keep) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= total || g.kind[k] != 1) return;
    const double2 p = g.xy[k];
    const float4 q = g.gs[k];
    const float L = g.len[k];
    const int cls = dets[k].cls;
    const float conf = dets[k].conf;
    const double R = __dadd_rn(__dmul_rn(reach_coef, (double)L), 1.0);
    const double ic = 1.0 / kMnmsCell;
    const long long x0 = (long long)floor(__dsub_rn(p.x, R) * ic), x1 = (long long)floor(__dadd_rn(p.x, R) * ic);
    const long long y0 = (long long)floor(__dsub_rn(p.y, R) * ic), y1 = (long long)floor(__dadd_rn(p.y, R) * ic);
    for (long long cx = x0; cx <= x1; ++cx)
        for (long long cy = y0; cy <= y1; ++cy)
            for (int t = cell_first(g.cell_key, g.cell_head, g.cap_mask, pack_cell(cx, cy)); t >= 0; t = g.next[t]) {
                const float Lt = g.len[t];
                if (!(Lt < L || (Lt == L && t < k))) continue;      // the pair belongs to its member with the longer side
                if (dets[t].cls != cls) continue;
                mnms_pair(g, k, p, q, conf, t, dets[t].conf, thr, keep);
            }
}

// Every eligible record against the irregular list; a pair of two irregular records is examined once, by the lower index
__global__ void __launch_bounds__(256) mosaic_nms_irregular_kernel(const b2d_obb* __restrict__ dets, int total, float thr, MnmsGrid g,
                                                                   uint8_t* keep) {
    __shared__ int s_irr[256];
    const int nd = *g.irr_count;
    if (nd == 0) return;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int kind = k < total ? g.kind[k] : 0;
    double2 p = make_double2(0.0, 0.0);
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
    int cls = 0;
    float conf = 0.f;
    if (kind) { p = g.xy[k]; q = g.gs[k]; cls = dets[k].cls; conf = dets[k].conf; }
    for (int base = 0; base < nd; base += 256) {
        __syncthreads();
        if (base + (int)threadIdx.x < nd) s_irr[threadIdx.x] = g.irr[base + threadIdx.x];
        __syncthreads();
        if (!kind) continue;
        const int m = min(256, nd - base);
        for (int i = 0; i < m; ++i) {
            const int t = s_irr[i];
            if (t == k || (kind == 2 && t < k) || dets[t].cls != cls) continue;
            mnms_pair(g, k, p, q, conf, t, dets[t].conf, thr, keep);
        }
    }
}

size_t mnms_table_cap(int total) {
    size_t cap = 1024;
    while (cap < 2 * (size_t)total) cap <<= 1;
    return cap;
}

// Sorts each tile's candidates into keys (tile stride keys_stride(cand_cap)): by confidence, else in slot order
int sort_keys_launch(const b2d_det* cand, const int* cand_count, int cand_cap, int n, unsigned long long* keys, int by_conf,
                     cudaStream_t stream) {
    B2D_CHECK(cand_cap <= kMaxCand, "postprocess: candidate capacity %d exceeds the sort key's 16-bit slot field", cand_cap);
    if (b2d_func_smem_optin((const void*)sort_keys_kernel, kSortSmemKeys * 8)) return -2;
    int need = 1;
    while (need < cand_cap && need < kSortSmemKeys) need <<= 1;       // keys that can occur, capped by the smem variant
    sort_keys_kernel<<<n, kSortThreads, (size_t)need * 8, stream>>>(cand, cand_count, cand_cap, keys, keys_stride(cand_cap), by_conf);
    B2D_LAUNCH_CHECK();
    return 0;
}

}  // namespace

int obb_decode_rows_launch(const HeadDesc* h, int n, float* rows, cudaStream_t stream) {
    if (n <= 0) return 0;
    dim3 grid(ceil_div(h->rows_total * 4, 256), n);
    obb_head_kernel<0><<<grid, 256, 0, stream>>>(*h, 0.f, 1, 1.f, rows, nullptr, nullptr, nullptr, 0);
    B2D_LAUNCH_CHECK();
    return 0;
}

int obb_postprocess_launch(const HeadDesc* h, int n, float thr, int inclusive, float scale, b2d_det* cand, float* cand_angle,
                           int* cand_count, int cand_cap, unsigned long long* keys_scratch, float4* prm, float iou_thr, int top_k,
                           int max_det, b2d_obb* out, int* out_count, int cap, cudaStream_t stream) {
    if (n <= 0) return 0;
    B2D_CUDA(cudaMemsetAsync(cand_count, 0, sizeof(int) * n, stream));
    dim3 grid(ceil_div(h->rows_total * 4, 256), n);
    obb_head_kernel<1><<<grid, 256, 0, stream>>>(*h, thr, inclusive, scale, nullptr, cand, cand_angle, cand_count, cand_cap);
    B2D_LAUNCH_CHECK();
    if (int rc = sort_keys_launch(cand, cand_count, cand_cap, n, keys_scratch, (iou_thr > 0.f) || (top_k > 0), stream)) return rc;
    obb_select_kernel<<<n, kObbThreads, 0, stream>>>(cand, cand_angle, cand_count, cand_cap, keys_scratch, keys_stride(cand_cap), prm,
                                                     iou_thr, top_k, max_det, out, out_count, cap);
    B2D_LAUNCH_CHECK();
    return 0;
}

int obb_georef_launch(const b2d_obb* dets, const int* counts, int n, int cap, int mode, const double* params, b2d_geoobb* out,
                      cudaStream_t stream) {
    if (n <= 0 || cap <= 0) return 0;
    dim3 grid(ceil_div(cap, 256), n);
    obb_georef_kernel<<<grid, 256, 0, stream>>>(dets, counts, cap, mode, params, out);
    B2D_LAUNCH_CHECK();
    return 0;
}

// Scratch of the mosaic merge: per-record arrays, then the grid's cell table, each 256-byte aligned
static size_t mnms_layout(int total, uint8_t* base, MnmsGrid* g) {
    const size_t n = (size_t)total, cap = mnms_table_cap(total);
    size_t off = 0;
    auto take = [&](size_t bytes) { uint8_t* p = base ? base + off : nullptr; off += (bytes + 255) & ~(size_t)255; return p; };
    MnmsGrid t;
    t.xy = (double2*)take(n * sizeof(double2));
    t.gs = (float4*)take(n * sizeof(float4));
    t.len = (float*)take(n * sizeof(float));
    t.kind = take(n);
    t.next = (int*)take(n * sizeof(int));
    t.irr = (int*)take(n * sizeof(int));
    t.irr_count = (int*)take(sizeof(int));
    t.cell_key = (long long*)take(cap * sizeof(long long));
    t.cell_head = (int*)take(cap * sizeof(int));
    t.cap_mask = (unsigned)(cap - 1);
    if (g) *g = t;
    return off;
}

size_t mosaic_nms_obb_scratch_bytes(int total) { return mnms_layout(total, nullptr, nullptr); }

int mosaic_nms_obb_launch(const b2d_obb* dets, const int* counts, const double* params, int n, int cap, float conf_thr, float iou_thr,
                          uint8_t* keep, void* scratch, size_t scratch_bytes, cudaStream_t stream) {
    const int total = n * cap;                 // the caller has checked that n * cap fits an int
    if (total <= 0) return 0;
    B2D_CHECK(scratch_bytes >= mosaic_nms_obb_scratch_bytes(total), "mosaic_nms_obb: scratch too small");
    MnmsGrid g;
    const size_t cell_bytes = mnms_layout(total, (uint8_t*)scratch, &g) - (size_t)((uint8_t*)g.cell_key - (uint8_t*)scratch);
    // the proof above mosaic_nms_prep_kernel: bd_lim, K and the scan radius sqrt(2 K) L of a regular box's long side L
    const double u = 1.0 / 16777216.0, eps = (double)kProbEps;
    const double hm = 1.0 - (double)iou_thr + 4.0 * u;
    const double arg = 1.0 + eps - hm * hm * (1.0 + 2.0 * u) - 8.0 * u;
    const double bd_lim = arg > exp(-100.0) ? fmin(-log(arg), 100.0) : 100.0;
    const double reach_coef = sqrt(2.0 * (bd_lim + 1.0 / 16.0) * 17.0 / 48.0);
    const float max_len = (float)((kMnmsReach * kMnmsCell - 1.0) / reach_coef);
    B2D_CUDA(cudaMemsetAsync(g.cell_key, 0xFF, cell_bytes, stream));          // cell keys and heads: -1
    B2D_CUDA(cudaMemsetAsync(g.irr_count, 0, sizeof(int), stream));
    const int blocks = ceil_div(total, 256);
    mosaic_nms_prep_kernel<<<blocks, 256, 0, stream>>>(dets, counts, params, cap, total, conf_thr, max_len, g, keep);
    mosaic_nms_grid_kernel<<<blocks, 256, 0, stream>>>(dets, total, reach_coef, iou_thr, g, keep);
    mosaic_nms_irregular_kernel<<<blocks, 256, 0, stream>>>(dets, total, iou_thr, g, keep);
    B2D_LAUNCH_CHECK();
    return 0;
}

int decode_rows_launch(const HeadDesc* h, int n, float* rows, cudaStream_t stream) {
    if (n <= 0) return 0;
    const int per = (h->kind == B2D_HEAD_V8_DFL) ? 4 : 1;
    dim3 grid(ceil_div(h->rows_total * per, 256), n);
    head_kernel<0><<<grid, 256, 0, stream>>>(*h, 0.f, 1, 1.f, rows, nullptr, nullptr, 0);
    B2D_LAUNCH_CHECK();
    return 0;
}

int candidates_from_head_launch(const HeadDesc* h, int n, float thr, int inclusive, float scale, b2d_det* cand, int* cand_count,
                                int cand_cap, cudaStream_t stream) {
    if (n <= 0) return 0;
    B2D_CUDA(cudaMemsetAsync(cand_count, 0, sizeof(int) * n, stream));
    const int per = (h->kind == B2D_HEAD_V8_DFL) ? 4 : 1;
    dim3 grid(ceil_div(h->rows_total * per, 256), n);
    head_kernel<1><<<grid, 256, 0, stream>>>(*h, thr, inclusive, scale, nullptr, cand, cand_count, cand_cap);
    B2D_LAUNCH_CHECK();
    return 0;
}

int candidates_from_rows_launch(const float* rows, int n, int num_rows, int ncol, float thr, int inclusive, float scale, b2d_det* cand,
                                int* cand_count, int cand_cap, cudaStream_t stream) {
    if (n <= 0) return 0;
    B2D_CUDA(cudaMemsetAsync(cand_count, 0, sizeof(int) * n, stream));
    dim3 grid(ceil_div(num_rows, 256), n);
    rows_filter_kernel<<<grid, 256, 0, stream>>>(rows, num_rows, ncol, thr, inclusive, scale, cand, cand_count, cand_cap);
    B2D_LAUNCH_CHECK();
    return 0;
}

int select_launch(const b2d_det* cand, const int* cand_count, int cand_cap, int n, unsigned long long* keys_scratch, float iou_thr,
                  int top_k, int max_det, b2d_det* out, int* out_count, int cap, cudaStream_t stream) {
    if (n <= 0) return 0;
    B2D_CHECK(!(iou_thr > 0.f) || max_det <= kMaxDet, "select: max_det %d exceeds the NMS kernel's %d kept boxes per tile", max_det, kMaxDet);
    if (int rc = sort_keys_launch(cand, cand_count, cand_cap, n, keys_scratch, (iou_thr > 0.f) || (top_k > 0), stream)) return rc;
    select_kernel<<<n, kSelThreads, 0, stream>>>(cand, cand_count, cand_cap, keys_scratch, keys_stride(cand_cap), iou_thr, top_k, max_det,
                                                 out, out_count, cap);
    B2D_LAUNCH_CHECK();
    return 0;
}

int georef_launch(const b2d_det* dets, const int* counts, int n, int cap, int mode, const double* params, b2d_geodet* out,
                  cudaStream_t stream) {
    if (n <= 0 || cap <= 0) return 0;
    dim3 grid(ceil_div(cap, 256), n);
    georef_kernel<<<grid, 256, 0, stream>>>(dets, counts, cap, mode, params, out);
    B2D_LAUNCH_CHECK();
    return 0;
}


// ---------------------------------------------------------------------------------------------
// Segmentation head (config C5): per-pixel argmax + softmax probability over nc <= 8 fp32 logits of an NHWC buffer with c
// channels per pixel (c * 4 bytes a multiple of 16).  HBM-bound: 16 bytes read and 1 (+4) written per pixel.
// ---------------------------------------------------------------------------------------------
namespace {
__global__ void segment_kernel(const float4* __restrict__ logits, long long npix, int c4, int nc, uint8_t* __restrict__ labels,
                               float* __restrict__ conf) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < npix; i += (long long)gridDim.x * blockDim.x) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            if (j < c4) {
                const float4 q = __ldg(logits + i * c4 + j);
                v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w;
            }
        }
        int best = 0;
        float m = v[0];
#pragma unroll
        for (int k = 1; k < 8; ++k)
            if (k < nc && v[k] > m) { m = v[k]; best = k; }
        labels[i] = (uint8_t)best;
        if (conf) {
            float sum = 0.f;
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (k < nc) sum += expf(v[k] - m);
            conf[i] = 1.0f / sum;
        }
    }
}
}  // namespace

int segment_launch(const float* logits, long long npix, int c, int nc, uint8_t* labels, float* conf, cudaStream_t stream) {
    B2D_CHECK(c % 4 == 0 && c <= 8 && nc >= 1 && nc <= c, "segment: %d classes in %d channels not supported", nc, c);
    if (npix <= 0) return 0;
    const int threads = 256;
    long long blocks = (npix + threads - 1) / threads;
    if (blocks > 148 * 16) blocks = 148 * 16;
    segment_kernel<<<(unsigned)blocks, threads, 0, stream>>>((const float4*)logits, npix, c / 4, nc, labels, conf);
    B2D_LAUNCH_CHECK();
    return 0;
}
