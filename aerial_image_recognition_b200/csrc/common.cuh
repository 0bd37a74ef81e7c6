// Shared declarations for the b2det CUDA library (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <memory>

#include "../../include/b2det.h"

void b2d_set_error(const char* fmt, ...);

#define B2D_CUDA(x)                                                                          \
    do {                                                                                     \
        cudaError_t e__ = (x);                                                               \
        if (e__ != cudaSuccess) {                                                            \
            b2d_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #x, cudaGetErrorString(e__)); \
            return -2;                                                                       \
        }                                                                                    \
    } while (0)

#define B2D_CHECK(cond, ...)                 \
    do {                                     \
        if (!(cond)) {                       \
            b2d_set_error(__VA_ARGS__);      \
            return -1;                       \
        }                                    \
    } while (0)

#define B2D_LAUNCH_CHECK() B2D_CUDA(cudaGetLastError())

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// The one owner of a cudaMalloc (Pinned = false) or cudaMallocHost (Pinned = true) block: freed by its destructor, moved,
// never copied.  bytes() is always the size of the block it holds, 0 when it holds none.
template <class T, bool Pinned>
class CudaBlock {
  public:
    T* get() const { return ptr_.get(); }
    size_t bytes() const { return bytes_; }
    void reset() { ptr_.reset(); bytes_ = 0; }
    // Grow-only: keeps the block when it holds `bytes`, else frees it and allocates `bytes`.  A refused allocation leaves
    // the owner empty and returns -2 with the error set, like B2D_CUDA.
    int reserve(size_t bytes) {
        if (bytes <= bytes_) return 0;
        reset();
        void* p = nullptr;
        const cudaError_t err = Pinned ? cudaMallocHost(&p, bytes) : cudaMalloc(&p, bytes);
        if (err != cudaSuccess) {
            cudaGetLastError();      // the refusal is reported here; the next launch check must not report it again
            b2d_set_error("%s:%d %s(%zu bytes) -> %s", __FILE__, __LINE__, Pinned ? "cudaMallocHost" : "cudaMalloc", bytes,
                          cudaGetErrorString(err));
            return -2;
        }
        ptr_.reset(static_cast<T*>(p));
        bytes_ = bytes;
        return 0;
    }

  private:
    struct Free {
        void operator()(T* p) const { Pinned ? cudaFreeHost(p) : cudaFree(p); }
    };
    std::unique_ptr<T, Free> ptr_;
    size_t bytes_ = 0;
};
template <class T> using DeviceBlock = CudaBlock<T, false>;
template <class T> using PinnedBlock = CudaBlock<T, true>;

// Hashed uniform grid (dedup.cu; the mosaic-wide oriented-box merge in postprocess.cu): an open-addressing table of
// 2^k cell keys (linear probing), each slot the head of a linked list of points, built with one atomicExch per point.
// Cell indices are biased by 2^31 so that no in-range cell packs to the empty-slot sentinel 0xFFFF...F (cell (-1, -1) did
// with plain two's-complement packing: points there were inserted but never found, so their duplicates survived).
constexpr long long kCellBias = 1ll << 31, kCellMax = (1ll << 31) - 2;
__device__ __forceinline__ unsigned long long pack_cell(long long cx, long long cy) {
    return ((unsigned long long)(cx + kCellBias) << 32) | (unsigned long long)(cy + kCellBias);
}
__device__ __forceinline__ unsigned hash_cell(unsigned long long k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL; k ^= k >> 33;
    return (unsigned)k;
}
// The slot holding cell `key`, claimed if the cell has none yet (the table must have an empty slot)
__device__ __forceinline__ unsigned cell_claim(long long* cell_key, unsigned cap_mask, unsigned long long key) {
    unsigned slot = hash_cell(key) & cap_mask;
    while (true) {
        const long long prev = atomicCAS((unsigned long long*)&cell_key[slot], (unsigned long long)-1LL, key);
        if (prev == -1LL || (unsigned long long)prev == key) return slot;
        slot = (slot + 1) & cap_mask;
    }
}
// The first point of cell `key`'s list, -1 for a cell without points
__device__ __forceinline__ int cell_first(const long long* cell_key, const int* cell_head, unsigned cap_mask, unsigned long long key) {
    unsigned slot = hash_cell(key) & cap_mask;
    while (true) {
        const long long k = cell_key[slot];
        if (k == -1LL) return -1;
        if ((unsigned long long)k == key) return cell_head[slot];
        slot = (slot + 1) & cap_mask;
    }
}

// Opt a kernel in to more than 48 KB of dynamic shared memory on the CURRENT device, once per (device, kernel): the
// attribute is per device, so a process-global "done" flag would leave the second GPU of a process without it
// (engine.cu; thread-safe).
int b2d_func_smem_optin(const void* func, int bytes);

// ---------------------------------------------------------------------------------------
// tcgen05 implicit-GEMM convolution (conv_tc.cu)
// ---------------------------------------------------------------------------------------
// which kernel runs a planned convolution (conv_tc.cu)
enum ConvKind : int {
    CONV_GENERIC,     // one TMA box per (tap, chunk); CTA-pair form when ConvTcParams::pair
    CONV_HALO,        // 3x3 stride 1 on 8-pixel-wide tiles, one halo box per chunk; CTA-pair form when ConvTcParams::pair
    CONV_DEPTHWISE,   // depthwise 3x3: halo + diagonal weight blocks
    CONV_STEM,        // the 4-channel network input through TMA: space-to-depth (stride 2) or pixel pairs (stride 1)
    CONV_DWPW,        // fused depthwise 3x3 + pointwise 1x1
    CONV_S2HALO,      // 3x3 stride 2 with one K chunk, one halo box per phase map
};

struct __align__(64) ConvTcParams {
    CUtensorMap tmA[4];   // generic: [0] stride-1 map or [py*2+px] the four stride-2 phase maps; halo: [0] the halo box map
    CUtensorMap tmB;      // packed weights [cout_pad][taps*cin_pad], K contiguous
    CUtensorMap tmO[3];   // output slice, one warp quarter's sub-box, chunk width 128 / 64 / 32 bytes
    CUtensorMap tmR[3];   // residual slice, same boxes
    int has_res;
    int stg_bufs;         // 1 or 2 staging buffers (each mt tiles x 128 rows x n_tile columns)
    uint32_t stg_off, bar_off;   // smem offsets (from the 1 KiB aligned base) of the staging region / barrier block
    const float* bias;    // [cout_pad]
    int W, H;             // output spatial size
    int cin, cout;        // true channel counts
    int n_tile, n_tiles_n;
    int chunks;           // 64-channel K chunks per tap
    int ksz, taps, stride;
    int bw, bh, bn;       // M tile = bw x bh pixels x bn images = 128 rows, row m = (y * bn + n) * bw + x
    int perm;             // 1: activation maps are (C, W, N, H) (tiles spanning images), 0: (C, W, H, N)
    int tiles_x, tiles_y;
    uint32_t rcp_nn, rcp_tx, rcp_ty;   // ceil(2^32 / d) for the tile decode (0 when d == 1)
    int act, out_f32;
    int stages;
    ConvKind kind;
    int pair;             // 1: CTA-pair kernel (cta_group::2, M = 256 across two SMs)
    int mt;               // M tiles per round (share B stages, one accumulator stage, one epilogue pass)
    int halo_w;           // bw + 2
    uint32_t halo_bytes;  // bytes of one halo buffer (1 KiB multiple)
    uint32_t halo_kh_rows;   // halo rows between kh taps = bn * (bw + 2)
    uint32_t a_bytes, b_bytes;       // smem bytes of one A tile / one B stage (padded to 1 KiB)
    uint32_t a_tx_bytes, b_tx_bytes; // TMA bytes of one A box / one B box
    uint32_t tmem_cols;
    uint32_t idesc;
    const void* w_raw;    // stem: packed weights [n_tile][64] bf16
    int f16;              // 16-bit activation / weight format: 0 bf16, 1 fp16 (B2D_PREC_FP16, B2D_PREC_FP16X2)
    int epi_parts;        // epilogue warps per TMEM lane quarter: 2 (warps 4-11) or 3 (warps 4-15), each taking every epi_parts-th 16-column unit
    int x2;               // 1: split-fp16 storage (B2D_PREC_FP16X2): inputs are [hi x 8 | lo x 8] groups, 16-bit outputs are written that way
    float acc_scale;      // the accumulator is multiplied by this before the bias (1/255 in the stem: its input is the raw pixel value)
    int b_res;            // halo kernel: 1 = all 9 * chunks weight boxes stay resident in the stage slots (loaded once per CTA)
    const float* dw_w;    // fused depthwise + pointwise kernel: [chunk][tap][64] fp32 depthwise weights, then [chunks * 64] bias (x 0.5 for SiLU)
    uint32_t dw_off;      // ... their offset in shared memory
    int dw_act;           // ... SiLU after the depthwise stage
    int rev;              // 1: this op walks its M tiles in descending order (set per op by the engine)
    int rev_last;         // per launch: index of the last M tile when walking backwards, else -1
    long long* trace;     // debug only (B2D_TRACE=1): per-role clock64 stamps of CTA 0, else nullptr
};

struct ConvTcPlan {
    ConvTcParams p;
    size_t smem_bytes;
    int sm_count;
    DeviceBlock<__nv_bfloat16> w_dev;   // packed weights
    DeviceBlock<float> bias_dev;
    DeviceBlock<float> dw_dev;          // fused depthwise + pointwise plans
    DeviceBlock<long long> trace_dev;   // debug only
};

// fused depthwise 3x3 (c channels, source slice) + pointwise 1x1 (c -> cout, destination slice), both with bias and optional SiLU
struct DwFuse { const __nv_bfloat16* src; int src_cs, src_c0; const float* w; const float* b; int act; };
int conv_tc_supported(int cin, int ksz, int stride);
int conv_tc_stem_supported(int src_cs, int cin, int ksz, int stride, int cout, int dst_f32, int has_res);
int conv_tc_plan(ConvTcPlan* plan, int sm_count, int max_batch,
                 const __nv_bfloat16* src, int src_h, int src_w, int src_cs, int src_c0, int cin,
                 void* dst, int dst_h, int dst_w, int dst_cs, int dst_c0, int cout, int dst_f32,
                 int ksz, int stride, int act, const float* w_host, const float* b_host,
                 const __nv_bfloat16* res, int res_cs, int res_c0, int depthwise = 0, int f16 = 0, int x2 = 0, float acc_scale = 1.f,
                 const DwFuse* fuse = nullptr);
int conv_tc_dw_supported(int cin, int cout, int ksz, int stride, int dst_f32, int has_res);
int conv_tc_dwpw_supported(int c, int cout, int dst_f32, int x2);
int conv_tc_launch(const ConvTcPlan* plan, int n, cudaStream_t stream);
int conv_tc_describe(const ConvTcPlan* plan, char* buf, int buflen);

// ---------------------------------------------------------------------------------------
// pools and upsample (pool.cu)
// ---------------------------------------------------------------------------------------
int maxpool_launch(const __nv_bfloat16* src, int h, int w, int src_cs, int src_c0,
                   __nv_bfloat16* dst, int oh, int ow, int dst_cs, int dst_c0, int c, int k, int stride,
                   int n, cudaStream_t stream, int f16 = 0, int x2 = 0);
int poolchain_launch(const __nv_bfloat16* src, int h, int w, int src_cs, int src_c0, __nv_bfloat16* const* dst, const int* dst_c0,
                     int dst_cs, int c, int stages, int n, cudaStream_t stream, int f16 = 0);
int poolchain_fits(int h, int w);
int upsample2x_launch(const __nv_bfloat16* src, int h, int w, int src_cs, int src_c0,
                      __nv_bfloat16* dst, int dst_cs, int dst_c0, int c, int n, cudaStream_t stream);

// ---------------------------------------------------------------------------------------
// pre / post processing
// ---------------------------------------------------------------------------------------
// OpenCV INTER_LINEAR (cv::resize, 8-bit): source taps (i0, i1) and 11-bit coefficients (a0, a1) of output index d, where
// scale = in_size / out_size.  Horizontal taps outside the image zero the fraction (fx = 0, sx clamped); the vertical pass
// keeps the fraction and clamps the two row indices separately.  The two rules give the same bytes on every down-scale
// and differ in the edge rows of an up-scale.  One IEEE rounding per operation on host and device (no contraction), so
// the host tables and the device-computed coefficients are the same numbers.
__host__ __device__ inline void cv2_linear_coef(int d, double scale, int in_size, int vertical, int* i0, int* i1, int* a0, int* a1) {
#ifdef __CUDA_ARCH__
    float f = (float)__dadd_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), -0.5);
#else
    float f = (float)(((double)d + 0.5) * scale - 0.5);     // x86-64 host code has no FMA to contract into
#endif
    int s = (int)floorf(f);
    f -= (float)s;
    if (vertical) {
        *i0 = s < 0 ? 0 : (s > in_size - 1 ? in_size - 1 : s);
        *i1 = s + 1 < 0 ? 0 : (s + 1 > in_size - 1 ? in_size - 1 : s + 1);
    } else {
        if (s < 0) { f = 0.f; s = 0; }
        if (s >= in_size - 1) { f = 0.f; s = in_size - 1; }
        *i0 = s;
        *i1 = s + 1 < in_size ? s + 1 : in_size - 1;
    }
    *a0 = (int)lrintf((1.f - f) * 2048.f);
    *a1 = (int)lrintf(f * 2048.f);
}

struct ResizeTables {     // device tables for one (mode, in_h, in_w, out)
    int mode, in_h, in_w, out_h, out_w, left, top;   // left/top: letterbox placement
    int ksize_x, ksize_y;
    int32_t* xb; int32_t* xk;   // PIL: bounds [out][2], coeffs [out][ksize]; cv2: ofs [out][2], coef [out][2]
    int32_t* yb; int32_t* yk;
    uint8_t* tmp; size_t tmp_bytes;   // PIL horizontal-pass temporary
};
int preprocess_launch(const ResizeTables* t, const uint8_t* src, int n, int pitch, long long img_stride,
                      int bgr, int out_kind, void* dst, int out_size, cudaStream_t stream);
// host: the cv2 INTER_LINEAR table of one axis (cv2_linear_coef for every output index), ofs / coef [out_size][2]
void cv2_linear_axis_table(int in_size, int out_size, int vertical, int32_t* ofs, int32_t* coef);
// mosaic windows (x0, y0, w0, h0) -> cv2 INTER_LINEAR by imgsz / win, centred on an imgsz x imgsz canvas of `fill`
int resize_windows_launch(const uint8_t* mosaic, int mh, int mw, long long pitch, const int32_t* origins, int n, int win, int imgsz,
                          int fill, int bgr, int out_kind, void* dst, cudaStream_t stream);

int input_from_f32_launch(const float* src, int n, int h, int w, void* dst, cudaStream_t stream, int f16 = 0);

struct HeadLevel { const float* buf; int hw, c, stride; float anchors[6]; int row0; };
struct HeadDesc { HeadLevel lv[3]; int nlevels; int kind; int nc; int rows_total; };

// OBB head: the angle logit sits at the first 16-byte-aligned fp32 channel after the 64 DFL and nc class channels
// (graph.obb_angle_channel)
__host__ __device__ inline int obb_angle_channel(int nc) { return (64 + nc + 3) / 4 * 4; }

// Candidates per tile: one per row, and the sort keys carry the anchor and the candidate slot in 16-bit fields
// (postprocess.cu, sort_key), so a tile may have at most this many rows
constexpr int kMaxCand = 65536;
// Ultralytics' max_nms: NMS looks at the best this many candidates of a tile only (both NMS kernels)
constexpr int kMaxNms = 30000;
// Sort keys per tile: the candidate capacity rounded up to a power of two
static inline int keys_stride(int cand_cap) {
    int s = 1;
    while (s < cand_cap) s <<= 1;
    return s;
}

int decode_rows_launch(const HeadDesc* h, int n, float* rows, cudaStream_t stream);
int candidates_from_head_launch(const HeadDesc* h, int n, float thr, int inclusive, float scale, b2d_det* cand, int* cand_count,
                                int cand_cap, cudaStream_t stream);
int candidates_from_rows_launch(const float* rows, int n, int num_rows, int ncol, float thr, int inclusive, float scale,
                                b2d_det* cand, int* cand_count, int cand_cap, cudaStream_t stream);
int select_launch(const b2d_det* cand, const int* cand_count, int cand_cap, int n, unsigned long long* keys_scratch,
                  float iou_thr, int top_k, int max_det, b2d_det* out, int* out_count, int cap, cudaStream_t stream);
// oriented boxes (yolov8m-obb): candidates are b2d_det records plus cand_angle[slot]; prm = 2 float4 per sorted candidate
int obb_decode_rows_launch(const HeadDesc* h, int n, float* rows, cudaStream_t stream);
int obb_postprocess_launch(const HeadDesc* h, int n, float thr, int inclusive, float scale, b2d_det* cand, float* cand_angle,
                           int* cand_count, int cand_cap, unsigned long long* keys_scratch, float4* prm, float iou_thr, int top_k,
                           int max_det, b2d_obb* out, int* out_count, int cap, cudaStream_t stream);
int obb_georef_launch(const b2d_obb* dets, const int* counts, int n, int cap, int mode, const double* params, b2d_geoobb* out,
                      cudaStream_t stream);
// mosaic-wide ProbIoU fast NMS over n windows' records [n][cap] (n * cap fits an int), keep [n][cap]
size_t mosaic_nms_obb_scratch_bytes(int total);
int mosaic_nms_obb_launch(const b2d_obb* dets, const int* counts, const double* params, int n, int cap, float conf_thr, float iou_thr,
                          uint8_t* keep, void* scratch, size_t scratch_bytes, cudaStream_t stream);
int segment_launch(const float* logits, long long npix, int c, int nc, uint8_t* labels, float* conf, cudaStream_t stream);
int georef_launch(const b2d_det* dets, const int* counts, int n, int cap, int mode, const double* params,
                  b2d_geodet* out, cudaStream_t stream);
int dedup_launch(const double* x, const double* y, const float* conf, const long long* tiebreak, int count, double thr,
                 int inclusive, uint8_t* keep, void* scratch, size_t scratch_bytes, cudaStream_t stream);
int closure_launch(const double* x, const double* y, int count, double thr, int inclusive, uint8_t* flag, void* scratch,
                   size_t scratch_bytes, cudaStream_t stream);
size_t dedup_scratch_bytes(int count);
int utm_forward_launch(const double* lon, const double* lat, int count, int zone, int north, double* x, double* y,
                       cudaStream_t stream);
// test-time-augmentation variants (tta.cu)
int tta_colour_launch(const uint8_t* src, long long npix, int code, uint8_t* dst, cudaStream_t stream);
int tta_clahe_launch(const uint8_t* src, int n, int h, int w, double clip_limit, int tiles_x, int tiles_y, uint8_t* luts, uint8_t* dst,
                     cudaStream_t stream);
int tta_lut_launch(const uint8_t* src, int n, long long img_bytes, const uint8_t* lut, int per_image, uint8_t* dst, cudaStream_t stream);
int tta_contrast_launch(const uint8_t* src, int n, int h, int w, float factor, unsigned long long* sums, uint8_t* luts, uint8_t* dst,
                        cudaStream_t stream);
int cut_windows_launch(const uint8_t* mosaic, int mh, int mw, long long pitch, const int32_t* origins, int n, int win,
                       int fill, uint8_t* dst, cudaStream_t stream);
