// K1 -- resize + normalise + layout, uint8 HWC -> bf16 NHWC4 (engine input) or f32 NCHW
// (the tensor the reference feeds to session.run).
//
// Reference lines replaced:
//   simple_detector.py:463-467, :655-659   PIL Image.resize((640,640)) [BICUBIC, antialias]
//                                          -> np.array -> astype(float32)/255.0 -> transpose(2,0,1)
//   _script/gpu_handler.py:67-92           cv2.resize(img,(640,640)) [INTER_LINEAR] -> /255 -> CHW
//   _script/gpu_handler.py:142-149         RGB->BGR variant (the `bgr` flag)
//   x_arch/02_analyze_images:1 (cell 6)    Ultralytics LetterBox (pad 114), via model(window)
//
// Both resamplers are integer algorithms once the per-index coefficient tables are known; the
// tables are computed on the host exactly as Pillow / OpenCV compute them (resize_tables.cpp
// section below) so the device code is integer multiply-accumulate only and bit-exact on uint8.
// Normalisation is a true IEEE division by 255.0f (__fdiv_rn), as NumPy does.
//
// These are HBM-bound byte kernels: the identity path moves 16 pixels (48 B in, 128 B out) per
// thread with 128-bit loads and stores; the resampling paths gather a few taps per output from
// L1/L2-resident rows.
#include "common.cuh"

#include <limits.h>
#include <math.h>
#include <string.h>
#include <vector>

namespace {

constexpr int PIL_BITS = 22;

__device__ __forceinline__ uint8_t clip8(int v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

// Two pixel values in the engine's network-input format: the RAW 0..255 value as bf16 / fp16 (exact in both).  The
// reference's `/ 255.0` (simple_detector.py:465, gpu_handler.py:79) is applied to the fp32 accumulator of the first
// convolution (ConvTcParams::acc_scale), so the input carries no 16-bit rounding of pixel / 255 at all.
__device__ __forceinline__ uint32_t bf16x2_of(uint8_t a, uint8_t b, int f16 = 0) {
    const float x = (float)a, y = (float)b;
    if (f16) {
        __half2 h = __floats2half2_rn(x, y);
        return *(uint32_t*)&h;
    }
    __nv_bfloat162 h = __floats2bfloat162_rn(x, y);
    return *(uint32_t*)&h;
}

// write one finished pixel in the requested layout
__device__ __forceinline__ void emit_pixel(int out_kind, void* dst, int img, int y, int x, int oh, int ow, uint8_t r, uint8_t g,
                                           uint8_t b, int bgr) {
    if (bgr) { uint8_t t = r; r = b; b = t; }
    const long long pix = ((long long)img * oh + y) * ow + x;
    if (out_kind == B2D_OUT_BF16_NHWC4 || out_kind == B2D_OUT_F16_NHWC4) {
        const int f16 = out_kind == B2D_OUT_F16_NHWC4;
        ((uint2*)dst)[pix] = make_uint2(bf16x2_of(r, g, f16), bf16x2_of(b, 0, f16));
    } else if (out_kind == B2D_OUT_F32_NCHW) {
        float* o = (float*)dst + (long long)img * 3 * oh * ow + (long long)y * ow + x;
        const long long plane = (long long)oh * ow;
        o[0] = __fdiv_rn((float)r, 255.0f);
        o[plane] = __fdiv_rn((float)g, 255.0f);
        o[2 * plane] = __fdiv_rn((float)b, 255.0f);
    } else {
        uint8_t* o = (uint8_t*)dst + pix * 3;
        o[0] = r; o[1] = g; o[2] = b;
    }
}

// ---- identity: 16 pixels per thread, 3 x 128-bit loads -> 8 x 128-bit stores ---------------
__global__ void __launch_bounds__(256) prep_identity_vec_kernel(const uint8_t* __restrict__ src, int n, int h, int w, int pitch,
                                                                 long long img_stride, uint2* __restrict__ dst, int bgr, int f16) {
    const int gw = w / 16;
    const long long total = (long long)n * h * gw;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int gx = (int)(idx % gw);
    const int y = (int)((idx / gw) % h);
    const int img = (int)(idx / ((long long)gw * h));
    const uint4* sp = (const uint4*)(src + img * img_stride + (long long)y * pitch + gx * 48);
    uint4 v[3];
    v[0] = __ldg(sp); v[1] = __ldg(sp + 1); v[2] = __ldg(sp + 2);
    const uint32_t wd[12] = {v[0].x, v[0].y, v[0].z, v[0].w, v[1].x, v[1].y, v[1].z, v[1].w, v[2].x, v[2].y, v[2].z, v[2].w};
    uint2 o[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        // byte k of the 48-byte run = (wd[k/4] >> 8*(k%4)) & 255, all indices compile-time
        uint8_t r = (uint8_t)(wd[(3 * i) >> 2] >> (8 * ((3 * i) & 3)));
        uint8_t g = (uint8_t)(wd[(3 * i + 1) >> 2] >> (8 * ((3 * i + 1) & 3)));
        uint8_t bl = (uint8_t)(wd[(3 * i + 2) >> 2] >> (8 * ((3 * i + 2) & 3)));
        if (bgr) { uint8_t t = r; r = bl; bl = t; }
        o[i] = make_uint2(bf16x2_of(r, g, f16), bf16x2_of(bl, 0, f16));
    }
    uint4* dp = (uint4*)(dst + ((long long)img * h + y) * w + gx * 16);
#pragma unroll
    for (int i = 0; i < 8; ++i) dp[i] = make_uint4(o[2 * i].x, o[2 * i].y, o[2 * i + 1].x, o[2 * i + 1].y);
}

// ---- identity, contiguous batch: every load and store instruction of a warp covers one contiguous run ---------------------
// A batch whose rows and images are packed (pitch = 3 w, img_stride = 3 w h) is one run of pixels.  Per round a warp moves
// 512 pixels: 96 coalesced 16-byte loads (1536 B) into its shared-memory slab, then 256 coalesced 16-byte stores (4096 B),
// lane l of iteration i converting pixels 2j, 2j + 1 (j = 32 i + l) from bytes 6j .. 6j + 5 of the slab.  The per-thread
// version above issues stores that each touch 32 different 128-byte lines (0.43 of the HBM peak measured).  v / 255 comes
// from a 256-entry shared table filled with the same __fdiv_rn + rounding, so the result is bit-identical.
__global__ void __launch_bounds__(256) prep_identity_run_kernel(const uint4* __restrict__ src, long long in_chunks, uint4* __restrict__ dst,
                                                                 int bgr, int f16) {
    __shared__ __align__(16) uint8_t slab[8][1536];
    __shared__ uint16_t q[256];          // byte -> its value in the 16-bit input format (see bf16x2_of)
    q[threadIdx.x] = (uint16_t)(bf16x2_of((uint8_t)threadIdx.x, 0, f16) & 0xffffu);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long rounds = (in_chunks + 95) / 96;
    const long long wstride = (long long)gridDim.x * 8;
    uint4* my = reinterpret_cast<uint4*>(slab[warp]);
    for (long long r = (long long)blockIdx.x * 8 + warp; r < rounds; r += wstride) {
        const long long c0 = r * 96;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const long long c = c0 + i * 32 + lane;
            if (c < in_chunks) my[i * 32 + lane] = __ldg(src + c);
        }
        __syncwarp();
        const long long o0 = r * 256, out_chunks = in_chunks / 3 * 8;      // 16 pixels: 3 chunks in, 8 chunks out
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int j = i * 32 + lane;
            if (o0 + j < out_chunks) {
                const uint16_t* p = reinterpret_cast<const uint16_t*>(slab[warp] + 6 * j);
                const uint32_t a = p[0], b = p[1], c = p[2];                // bytes r0 g0 | b0 r1 | g1 b1
                uint8_t r0 = a & 255, g0 = a >> 8, b0 = b & 255, r1 = b >> 8, g1 = c & 255, b1 = c >> 8;
                if (bgr) { uint8_t t = r0; r0 = b0; b0 = t; t = r1; r1 = b1; b1 = t; }
                dst[o0 + j] = make_uint4((uint32_t)q[r0] | ((uint32_t)q[g0] << 16), q[b0], (uint32_t)q[r1] | ((uint32_t)q[g1] << 16), q[b1]);
            }
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(256) prep_identity_kernel(const uint8_t* __restrict__ src, int n, int h, int w, int pitch,
                                                             long long img_stride, void* dst, int out_kind, int bgr) {
    const long long total = (long long)n * h * w;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x = (int)(idx % w);
    const int y = (int)((idx / w) % h);
    const int img = (int)(idx / ((long long)w * h));
    const uint8_t* sp = src + img * img_stride + (long long)y * pitch + x * 3;
    emit_pixel(out_kind, dst, img, y, x, h, w, sp[0], sp[1], sp[2], bgr);
}

// ---- OpenCV INTER_LINEAR (11-bit coefficients), also the resampler inside the letterbox -----
// tables: xb/yb = (i0, i1) source indices, xk/yk = (a0, a1) coefficients.
__global__ void __launch_bounds__(256) prep_linear_kernel(const uint8_t* __restrict__ src, int n, int pitch, long long img_stride,
                                                           ResizeTables t, void* dst, int out_kind, int bgr, int canvas) {
    // canvas = output tensor side; the resized image of t.out_w x t.out_h sits at (t.left, t.top)
    const long long total = (long long)n * canvas * canvas;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x = (int)(idx % canvas);
    const int y = (int)((idx / canvas) % canvas);
    const int img = (int)(idx / ((long long)canvas * canvas));
    const int rx = x - t.left, ry = y - t.top;
    if (rx < 0 || ry < 0 || rx >= t.out_w || ry >= t.out_h) {
        emit_pixel(out_kind, dst, img, y, x, canvas, canvas, 114, 114, 114, 0);
        return;
    }
    const int x0 = t.xb[2 * rx], x1 = t.xb[2 * rx + 1], a0 = t.xk[2 * rx], a1 = t.xk[2 * rx + 1];
    const int y0 = t.yb[2 * ry], y1 = t.yb[2 * ry + 1], b0 = t.yk[2 * ry], b1 = t.yk[2 * ry + 1];
    const uint8_t* base = src + img * img_stride;
    const uint8_t* r0 = base + (long long)y0 * pitch;
    const uint8_t* r1 = base + (long long)y1 * pitch;
    uint8_t o[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int s0 = r0[x0 * 3 + c] * a0 + r0[x1 * 3 + c] * a1;   // horizontal pass, scale 2^11
        const int s1 = r1[x0 * 3 + c] * a0 + r1[x1 * 3 + c] * a1;
        const int v = (((b0 * (s0 >> 4)) >> 16) + ((b1 * (s1 >> 4)) >> 16) + 2) >> 2;
        o[c] = clip8(v);
    }
    emit_pixel(out_kind, dst, img, y, x, canvas, canvas, o[0], o[1], o[2], bgr);
}

// ---- Pillow BICUBIC (antialiased): horizontal pass into a uint8 temporary, then vertical -----
__global__ void __launch_bounds__(256) pil_hpass_kernel(const uint8_t* __restrict__ src, int n, int in_h, int pitch,
                                                         long long img_stride, ResizeTables t, uint8_t* __restrict__ tmp) {
    const long long total = (long long)n * in_h * t.out_w;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x = (int)(idx % t.out_w);
    const int y = (int)((idx / t.out_w) % in_h);
    const int img = (int)(idx / ((long long)t.out_w * in_h));
    const int x0 = t.xb[2 * x], cnt = t.xb[2 * x + 1];
    const int32_t* k = t.xk + (long long)x * t.ksize_x;
    const uint8_t* sp = src + img * img_stride + (long long)y * pitch + x0 * 3;
    int s0 = 1 << (PIL_BITS - 1), s1 = s0, s2 = s0;
    for (int i = 0; i < cnt; ++i) {
        const int kk = k[i];
        s0 += sp[3 * i] * kk; s1 += sp[3 * i + 1] * kk; s2 += sp[3 * i + 2] * kk;
    }
    uint8_t* o = tmp + (((long long)img * in_h + y) * t.out_w + x) * 3;
    o[0] = clip8(s0 >> PIL_BITS); o[1] = clip8(s1 >> PIL_BITS); o[2] = clip8(s2 >> PIL_BITS);
}

__global__ void __launch_bounds__(256) pil_vpass_kernel(const uint8_t* __restrict__ src, int n, int in_h, int pitch,
                                                         long long img_stride, ResizeTables t, void* dst, int out_kind, int bgr) {
    const long long total = (long long)n * t.out_h * t.out_w;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x = (int)(idx % t.out_w);
    const int y = (int)((idx / t.out_w) % t.out_h);
    const int img = (int)(idx / ((long long)t.out_w * t.out_h));
    const int y0 = t.yb[2 * y], cnt = t.yb[2 * y + 1];
    const int32_t* k = t.yk + (long long)y * t.ksize_y;
    const uint8_t* sp = src + img * img_stride + (long long)y0 * pitch + x * 3;
    int s0 = 1 << (PIL_BITS - 1), s1 = s0, s2 = s0;
    for (int i = 0; i < cnt; ++i) {
        const int kk = k[i];
        const uint8_t* q = sp + (long long)i * pitch;
        s0 += q[0] * kk; s1 += q[1] * kk; s2 += q[2] * kk;
    }
    emit_pixel(out_kind, dst, img, y, x, t.out_h, t.out_w, clip8(s0 >> PIL_BITS), clip8(s1 >> PIL_BITS), clip8(s2 >> PIL_BITS), bgr);
}

// ---- sliding-window cutter (C4): clipped window -> centred 114 letterbox, no resample -------
__global__ void __launch_bounds__(256) cut_windows_kernel(const uint8_t* __restrict__ mosaic, int mh, int mw, long long pitch,
                                                           const int32_t* __restrict__ origins, int n, int win, int fill,
                                                           uint8_t* __restrict__ dst) {
    const long long total = (long long)n * win * win;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x = (int)(idx % win);
    const int y = (int)((idx / win) % win);
    const int i = (int)(idx / ((long long)win * win));
    const int x0 = origins[4 * i], y0 = origins[4 * i + 1], w0 = origins[4 * i + 2], h0 = origins[4 * i + 3];
    // Ultralytics LetterBox(center=True): top/left = round(d/2 - 0.1); d is an even/odd integer so
    // this is floor(d/2) for d >= 0 (banker's rounding never hits a tie at x.4)
    const int left = (win - w0) / 2, top = (win - h0) / 2;
    const int sx = x - left, sy = y - top;
    uint8_t r = (uint8_t)fill, g = (uint8_t)fill, b = (uint8_t)fill;
    if (sx >= 0 && sy >= 0 && sx < w0 && sy < h0 && x0 + sx < mw && y0 + sy < mh) {
        const uint8_t* sp = mosaic + (long long)(y0 + sy) * pitch + (long long)(x0 + sx) * 3;
        r = sp[0]; g = sp[1]; b = sp[2];
    }
    uint8_t* o = dst + idx * 3;
    o[0] = r; o[1] = g; o[2] = b;
}

// ---- windows of any size: cut + cv2 INTER_LINEAR + centred letterbox, one launch per batch ----------------------
// A CTA owns one window and walks bands of kBandRows canvas rows.  Per band, warp 0 computes each row's vertical taps
// and maps the distinct source rows they touch to slots; those rows are copied into shared memory with 16-byte loads,
// kStageRows at a time, and resampled horizontally into int16 rows (the `s >> 4` of the vertical sum); then every
// thread writes canvas pixels from two slot rows.  Each source row a band needs is read once per band (a row shared
// by two bands is read twice); the horizontal taps are computed once per CTA.  All coefficients come from
// cv2_linear_coef, so nothing is uploaded per window size.
constexpr int kBandRows = 4;
constexpr int kBandSlots = 2 * kBandRows;   // distinct source rows a band can touch
constexpr int kStageRows = 4;

struct WindowGeom { int nw, nh, left, top; };

// The geometry of mosaic.window_geometry: one gain g = imgsz / win, Python round() = rint()
__device__ __forceinline__ WindowGeom window_geom(int w0, int h0, int win, int imgsz) {
    const double g = __ddiv_rn((double)imgsz, (double)win);
    WindowGeom r;
    r.nw = max(1, (int)rint(__dmul_rn((double)w0, g)));
    r.nh = max(1, (int)rint(__dmul_rn((double)h0, g)));
    r.left = (int)rint(__dadd_rn((double)(imgsz - r.nw) * 0.5, -0.1));
    r.top = (int)rint(__dadd_rn((double)(imgsz - r.nh) * 0.5, -0.1));
    return r;
}

__host__ __device__ inline int raw_pitch(int win) { return (win * 3 + 15 + 15) / 16 * 16; }   // one source row + its 16-byte misalignment

static inline size_t resize_windows_smem(int win, int imgsz) {
    return (size_t)imgsz * sizeof(int4) + (size_t)kBandSlots * imgsz * sizeof(uint2) + (size_t)kStageRows * raw_pitch(win);
}

__global__ void __launch_bounds__(256) resize_windows_kernel(const uint8_t* __restrict__ mosaic, int mh, int mw, long long pitch,
                                                             const int32_t* __restrict__ origins, int win, int imgsz, int groups,
                                                             int fill, int bgr, int out_kind, void* dst) {
    extern __shared__ __align__(16) uint8_t smem[];
    int4* xtab = reinterpret_cast<int4*>(smem);                                    // [imgsz] byte offsets of the two taps, a0, a1
    uint2* hrow = reinterpret_cast<uint2*>(smem + (size_t)imgsz * sizeof(int4));   // [kBandSlots][imgsz] three int16 per pixel
    uint8_t* raw = smem + (size_t)imgsz * (sizeof(int4) + kBandSlots * sizeof(uint2));   // [kStageRows][rp] source bytes
    __shared__ int4 vtab[kBandRows];            // slot of each tap, b0, b1
    __shared__ int slot_row[kBandSlots];
    __shared__ int nslots;
    const int rp = raw_pitch(win);
    const int i = blockIdx.x / groups, grp = blockIdx.x % groups;
    const int x0 = origins[4 * i], y0 = origins[4 * i + 1], w0 = origins[4 * i + 2], h0 = origins[4 * i + 3];
    const bool ok = w0 >= 1 && w0 <= win && h0 >= 1 && h0 <= win && x0 >= 0 && y0 >= 0 && x0 <= mw - w0 && y0 <= mh - h0;
    WindowGeom gm = window_geom(ok ? w0 : win, ok ? h0 : win, win, imgsz);
    if (!ok) gm.nw = gm.nh = 0;             // a window the caller should have refused: all fill, nothing read
    const double sx = __ddiv_rn((double)w0, (double)gm.nw), sy = __ddiv_rn((double)h0, (double)gm.nh);
    for (int rx = threadIdx.x; rx < gm.nw; rx += blockDim.x) {
        int i0, i1, a0, a1;
        cv2_linear_coef(rx, sx, w0, 0, &i0, &i1, &a0, &a1);
        xtab[rx] = make_int4(3 * i0, 3 * i1, a0, a1);
    }
    const int nbands = (imgsz + kBandRows - 1) / kBandRows;
    const uint8_t fb = (uint8_t)fill;
    for (int band = grp; band < nbands; band += groups) {
        const int yb = band * kBandRows;
        if (threadIdx.x < 32) {
            // lane t < 2 kBandRows holds tap (t & 1) of band row t >> 1; inactive taps (pad rows) hold INT_MAX
            const int lane = threadIdx.x, ry = yb + (lane >> 1) - gm.top;
            int r0 = INT_MAX, r1 = INT_MAX, b0 = 0, b1 = 0;
            if (lane < kBandSlots && yb + (lane >> 1) < imgsz && ry >= 0 && ry < gm.nh) cv2_linear_coef(ry, sy, h0, 1, &r0, &r1, &b0, &b1);
            const int v = (lane & 1) ? r1 : r0;
            int first = v != INT_MAX, rank = 0;
            for (int k = 0; k < kBandSlots; ++k) {
                const int u = __shfl_sync(0xffffffffu, v, k);
                int ufirst = u != INT_MAX;
                for (int j = 0; j < k; ++j) ufirst &= __shfl_sync(0xffffffffu, v, j) != u;
                if (k < lane && u == v) first = 0;
                if (ufirst && u < v) ++rank;
            }
            if (lane < kBandSlots && first) slot_row[rank] = v;
            const int slot_other = __shfl_xor_sync(0xffffffffu, rank, 1);
            const unsigned firsts = __ballot_sync(0xffffffffu, lane < kBandSlots && first);
            if (lane < kBandSlots && !(lane & 1)) vtab[lane >> 1] = make_int4(rank, slot_other, b0, b1);
            if (lane == 0) nslots = __popc(firsts);
        }
        __syncthreads();
        const int ns = nslots;
        for (int s0 = 0; s0 < ns; s0 += kStageRows) {
            const int cnt = min(kStageRows, ns - s0);
            // 16-byte loads of the aligned run that holds bytes [x0 * 3, (x0 + w0) * 3) of each staged row.  The bytes read
            // before and after the row share a 16-byte block with bytes of the row, so they lie inside the mosaic's allocation.
            const int nch_max = (w0 * 3 + 30) >> 4;
            for (int p = threadIdx.x; p < cnt * nch_max; p += blockDim.x) {
                const int q = p / nch_max, c = p - q * nch_max;
                const uintptr_t a = (uintptr_t)(mosaic + (long long)(y0 + slot_row[s0 + q]) * pitch + (long long)x0 * 3);
                if (c < (int)(((a & 15) + w0 * 3 + 15) >> 4))
                    reinterpret_cast<uint4*>(raw + q * rp)[c] = __ldg(reinterpret_cast<const uint4*>(a & ~(uintptr_t)15) + c);
            }
            __syncthreads();
            for (int p = threadIdx.x; p < cnt * gm.nw; p += blockDim.x) {
                const int q = p / gm.nw, rx = p - q * gm.nw;
                const uint8_t* a = mosaic + (long long)(y0 + slot_row[s0 + q]) * pitch + (long long)x0 * 3;
                const uint8_t* r = raw + q * rp + ((uintptr_t)a & 15);
                const int4 t = xtab[rx];
                const int c0 = (r[t.x] * t.z + r[t.y] * t.w) >> 4;
                const int c1 = (r[t.x + 1] * t.z + r[t.y + 1] * t.w) >> 4;
                const int c2 = (r[t.x + 2] * t.z + r[t.y + 2] * t.w) >> 4;
                hrow[(size_t)(s0 + q) * imgsz + rx] = make_uint2((uint32_t)c0 | ((uint32_t)c1 << 16), (uint32_t)c2);
            }
            __syncthreads();
        }
        for (int p = threadIdx.x; p < kBandRows * imgsz; p += blockDim.x) {
            const int t = p / imgsz, x = p - t * imgsz, y = yb + t;
            if (y >= imgsz) break;
            const int rx = x - gm.left, ry = y - gm.top;
            uint8_t o[3] = {fb, fb, fb};
            if (rx >= 0 && rx < gm.nw && ry >= 0 && ry < gm.nh) {
                const int4 v = vtab[t];
                const uint2 h0v = hrow[(size_t)v.x * imgsz + rx], h1v = hrow[(size_t)v.y * imgsz + rx];
                const int s0[3] = {(int)(h0v.x & 0xffffu), (int)(h0v.x >> 16), (int)h0v.y};
                const int s1[3] = {(int)(h1v.x & 0xffffu), (int)(h1v.x >> 16), (int)h1v.y};
#pragma unroll
                for (int c = 0; c < 3; ++c) o[c] = clip8((((v.z * s0[c]) >> 16) + ((v.w * s1[c]) >> 16) + 2) >> 2);
            }
            emit_pixel(out_kind, dst, i, y, x, imgsz, imgsz, o[0], o[1], o[2], bgr);
        }
        __syncthreads();
    }
}


// ---- f32 NCHW in [0,1] (the tensor the reference hands to session.run) -> 16-bit NHWC4 network input ---------
__global__ void __launch_bounds__(256) input_from_f32_kernel(const float* __restrict__ src, int n, int h, int w, uint2* __restrict__ dst,
                                                              int f16) {
    const long long total = (long long)n * h * w;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long long plane = (long long)h * w;
    const int img = (int)(idx / plane);
    const long long p = idx - (long long)img * plane;
    const float* s = src + (long long)img * 3 * plane + p;
    // The network input is 8-bit: the reference only ever feeds pixel / 255 (simple_detector.py:465, gpu_handler.py:79-85),
    // so the tensor is mapped back to the pixel value it came from (exact for every u8 / 255.0f) and stored raw.
    auto px = [](float v) { return fminf(fmaxf(rintf(__fmul_rn(v, 255.0f)), 0.f), 255.f); };
    const float r = px(__ldg(s)), g = px(__ldg(s + plane)), b = px(__ldg(s + 2 * plane));
    if (f16) {
        __half2 a = __floats2half2_rn(r, g);
        __half2 c = __floats2half2_rn(b, 0.f);
        dst[idx] = make_uint2(*(uint32_t*)&a, *(uint32_t*)&c);
        return;
    }
    __nv_bfloat162 a = __floats2bfloat162_rn(r, g);
    __nv_bfloat162 c = __floats2bfloat162_rn(b, 0.f);
    dst[idx] = make_uint2(*(uint32_t*)&a, *(uint32_t*)&c);
}

}  // namespace

int input_from_f32_launch(const float* src, int n, int h, int w, void* dst, cudaStream_t stream, int f16) {
    if (n <= 0) return 0;
    const long long total = (long long)n * h * w;
    input_from_f32_kernel<<<(int)((total + 255) / 256), 256, 0, stream>>>(src, n, h, w, (uint2*)dst, f16);
    B2D_LAUNCH_CHECK();
    return 0;
}

int preprocess_launch(const ResizeTables* t, const uint8_t* src, int n, int pitch, long long img_stride, int bgr, int out_kind,
                      void* dst, int out_size, cudaStream_t stream) {
    if (n <= 0) return 0;
    if (t->mode == B2D_RESIZE_IDENTITY) {
        const bool vec = (out_kind == B2D_OUT_BF16_NHWC4 || out_kind == B2D_OUT_F16_NHWC4) && (t->in_w % 16 == 0) && (pitch % 16 == 0) && (img_stride % 16 == 0) &&
                         (((uintptr_t)src) % 16 == 0) && (((uintptr_t)dst) % 16 == 0);
        const bool packed = vec && pitch == t->in_w * 3 && img_stride == (long long)t->in_h * t->in_w * 3;
        if (packed) {
            const long long in_chunks = (long long)n * t->in_h * t->in_w * 3 / 16;
            const long long rounds = (in_chunks + 95) / 96;
            long long blocks = (rounds + 7) / 8;
            if (blocks > 148 * 8) blocks = 148 * 8;
            prep_identity_run_kernel<<<(int)blocks, 256, 0, stream>>>((const uint4*)src, in_chunks, (uint4*)dst, bgr,
                                                                      out_kind == B2D_OUT_F16_NHWC4);
        } else if (vec) {
            const long long total = (long long)n * t->in_h * (t->in_w / 16);
            prep_identity_vec_kernel<<<(int)((total + 255) / 256), 256, 0, stream>>>(src, n, t->in_h, t->in_w, pitch, img_stride,
                                                                                      (uint2*)dst, bgr, out_kind == B2D_OUT_F16_NHWC4);
        } else {
            const long long total = (long long)n * t->in_h * t->in_w;
            prep_identity_kernel<<<(int)((total + 255) / 256), 256, 0, stream>>>(src, n, t->in_h, t->in_w, pitch, img_stride, dst,
                                                                                  out_kind, bgr);
        }
    } else if (t->mode == B2D_RESIZE_CV2_LINEAR || t->mode == B2D_RESIZE_LETTERBOX) {
        const long long total = (long long)n * out_size * out_size;
        prep_linear_kernel<<<(int)((total + 255) / 256), 256, 0, stream>>>(src, n, pitch, img_stride, *t, dst, out_kind, bgr,
                                                                            out_size);
    } else if (t->mode == B2D_RESIZE_PIL_BICUBIC) {
        const uint8_t* vsrc = src;
        int vpitch = pitch;
        long long vstride = img_stride;
        if (t->in_w != t->out_w) {
            const long long total = (long long)n * t->in_h * t->out_w;
            pil_hpass_kernel<<<(int)((total + 255) / 256), 256, 0, stream>>>(src, n, t->in_h, pitch, img_stride, *t, t->tmp);
            B2D_LAUNCH_CHECK();
            vsrc = t->tmp; vpitch = t->out_w * 3; vstride = (long long)t->in_h * t->out_w * 3;
        }
        const long long total = (long long)n * t->out_h * t->out_w;
        pil_vpass_kernel<<<(int)((total + 255) / 256), 256, 0, stream>>>(vsrc, n, t->in_h, vpitch, vstride, *t, dst, out_kind, bgr);
    } else {
        B2D_CHECK(false, "preprocess: unknown resize mode %d", t->mode);
    }
    B2D_LAUNCH_CHECK();
    return 0;
}

int cut_windows_launch(const uint8_t* mosaic, int mh, int mw, long long pitch, const int32_t* origins, int n, int win, int fill,
                       uint8_t* dst, cudaStream_t stream) {
    if (n <= 0) return 0;
    const long long total = (long long)n * win * win;
    cut_windows_kernel<<<(int)((total + 255) / 256), 256, 0, stream>>>(mosaic, mh, mw, pitch, origins, n, win, fill, dst);
    B2D_LAUNCH_CHECK();
    return 0;
}

int resize_windows_launch(const uint8_t* mosaic, int mh, int mw, long long pitch, const int32_t* origins, int n, int win, int imgsz,
                          int fill, int bgr, int out_kind, void* dst, cudaStream_t stream) {
    if (n <= 0) return 0;
    const size_t smem = resize_windows_smem(win, imgsz);
    int dev = 0, optin = 0;
    cudaFuncAttributes fa;
    B2D_CUDA(cudaGetDevice(&dev));
    B2D_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    B2D_CUDA(cudaFuncGetAttributes(&fa, (const void*)resize_windows_kernel));
    const int dyn_max = optin - (int)fa.sharedSizeBytes;
    B2D_CHECK(smem <= (size_t)dyn_max, "resize_windows: window %d on a %d canvas needs %zu bytes of shared memory, the device allows %d",
              win, imgsz, smem, dyn_max);
    // opted in once per device at the largest size, so a later call with a larger window needs no second opt-in
    if (smem > 48 * 1024 && b2d_func_smem_optin((const void*)resize_windows_kernel, dyn_max)) return -2;
    // a CTA walks every groups-th band of one window: the horizontal taps are computed once per CTA, and a batch of
    // 64 windows is 1024 CTAs
    const int nbands = (imgsz + kBandRows - 1) / kBandRows;
    const int groups = nbands < 16 ? nbands : 16;
    B2D_CHECK((long long)n * groups < (1LL << 31), "resize_windows: %d windows", n);
    resize_windows_kernel<<<n * groups, 256, smem, stream>>>(mosaic, mh, mw, pitch, origins, win, imgsz, groups, fill, bgr, out_kind, dst);
    B2D_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------------------------
// host-side coefficient tables (same arithmetic as Pillow's precompute_coeffs / normalize_coeffs_8bpc
// and OpenCV's resize() table set-up; mirrored in aerial_image_recognition_b200/resample.py)
// ---------------------------------------------------------------------------------------------
static double bicubic_filter(double x) {
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}

extern "C" int b2d_resize_table(int mode, int in_size, int out_size, int32_t* bounds_out, int32_t* coef_out, int* ksize_out) {
    if (in_size <= 0 || out_size <= 0) return -1;
    if (mode == B2D_RESIZE_PIL_BICUBIC) {
        const double scale = (double)in_size / (double)out_size;
        const double filterscale = scale < 1.0 ? 1.0 : scale;
        const double support = 2.0 * filterscale;
        const int ksize = (int)ceil(support) * 2 + 1;
        if (ksize_out) *ksize_out = ksize;
        if (!bounds_out || !coef_out) return 0;
        const double ss = 1.0 / filterscale;
        std::vector<double> ws(ksize);
        for (int xx = 0; xx < out_size; ++xx) {
            const double center = (xx + 0.5) * scale;
            int xmin = (int)(center - support + 0.5);
            if (xmin < 0) xmin = 0;
            int xmax = (int)(center + support + 0.5);
            if (xmax > in_size) xmax = in_size;
            xmax -= xmin;
            double ww = 0.0;
            for (int x = 0; x < xmax; ++x) {
                ws[x] = bicubic_filter((x + xmin - center + 0.5) * ss);
                ww += ws[x];
            }
            for (int x = 0; x < ksize; ++x) {
                int v = 0;
                if (x < xmax) {
                    double w = (ww != 0.0) ? ws[x] / ww : ws[x];
                    v = (w < 0) ? (int)(-0.5 + w * (double)(1 << PIL_BITS)) : (int)(0.5 + w * (double)(1 << PIL_BITS));
                }
                coef_out[(size_t)xx * ksize + x] = v;
            }
            bounds_out[2 * xx] = xmin;
            bounds_out[2 * xx + 1] = xmax;
        }
        return 0;
    }
    if (mode == B2D_RESIZE_CV2_LINEAR) {
        if (ksize_out) *ksize_out = 2;
        if (!bounds_out || !coef_out) return 0;
        cv2_linear_axis_table(in_size, out_size, 0, bounds_out, coef_out);
        return 0;
    }
    return -1;
}

void cv2_linear_axis_table(int in_size, int out_size, int vertical, int32_t* ofs, int32_t* coef) {
    const double scale = (double)in_size / (double)out_size;
    for (int d = 0; d < out_size; ++d) {
        int i0, i1, a0, a1;
        cv2_linear_coef(d, scale, in_size, vertical, &i0, &i1, &a0, &a1);
        ofs[2 * d] = i0; ofs[2 * d + 1] = i1;
        coef[2 * d] = a0; coef[2 * d + 1] = a1;
    }
}
