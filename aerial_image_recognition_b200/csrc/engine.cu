// The C ABI (include/b2det.h): engine lifetime, plan building and stage entry points.
//
// An engine owns one GPU's buffers, packed weights, tensor maps and scratch.  The plan is the
// graph the reference gives onnxruntime as an .onnx file (_script/gpu_handler.py:61-65); here it
// is built op by op through b2d_plan_* and executed by b2d_forward as a fixed launch sequence.
#include "common.cuh"

#include <limits.h>
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <map>
#include <mutex>
#include <set>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

static_assert(sizeof(b2d_det) == 32 && sizeof(b2d_geodet) == 40, "record sizes are part of the ABI");
static_assert(sizeof(b2d_obb) == 36 && sizeof(b2d_geoobb) == 104, "record sizes are part of the ABI");

static thread_local std::string g_last_error;

void b2d_set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
}

int b2d_func_smem_optin(const void* func, int bytes) {
    static std::mutex mu;
    static std::set<std::pair<int, const void*>> done;
    int dev = 0;
    B2D_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    if (done.count({dev, func})) return 0;
    B2D_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    done.insert({dev, func});
    return 0;
}

namespace {

// Every entry point that touches the device runs with the engine's device current and restores the caller's on exit,
// so several engines (one per GPU) can live in one process and be called from any thread.
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() {
        if (switched) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};
#define B2D_ENTER(e) DeviceGuard b2d_guard__((e)->device)

struct Buffer {
    int h, w, c, f32;
    DeviceBlock<void> ptr;
};

// Owners of the engine's streams, events and graph executables
struct CudaDestroy {
    void operator()(cudaStream_t s) const { cudaStreamDestroy(s); }
    void operator()(cudaEvent_t ev) const { cudaEventDestroy(ev); }
    void operator()(cudaGraphExec_t g) const { cudaGraphExecDestroy(g); }
};
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, CudaDestroy>;
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, CudaDestroy>;
using GraphExec = std::unique_ptr<std::remove_pointer_t<cudaGraphExec_t>, CudaDestroy>;

// every stream the engine creates is non-blocking, every event has timing disabled
int create(Stream& s) {
    cudaStream_t raw;
    B2D_CUDA(cudaStreamCreateWithFlags(&raw, cudaStreamNonBlocking));
    s.reset(raw);
    return 0;
}
int create(Event& ev) {
    cudaEvent_t raw;
    B2D_CUDA(cudaEventCreateWithFlags(&raw, cudaEventDisableTiming));
    ev.reset(raw);
    return 0;
}

enum OpKind { OP_CONV_TC, OP_MAXPOOL, OP_UPSAMPLE, OP_POOLCHAIN, OP_NOP };

struct OpDesc {   // what the caller asked for (resolved into a plan at finalize)
    int kind_req;     // 0 conv, 1 dwconv, 2 maxpool, 3 upsample
    int src, src_c0, cin, dst, dst_c0, cout, k, stride, act, res, res_c0, impl;
    std::vector<float> w, b;
};

struct Op {
    OpKind kind;
    ConvTcPlan tc;
    // pool / upsample
    const __nv_bfloat16* src; __nv_bfloat16* dst;
    int h, w, src_cs, src_c0, oh, ow, dst_cs, dst_c0, c, k, stride;
    // pool chain (this op + the next chain_stages - 1 max-pools, which become OP_NOP)
    __nv_bfloat16* chain_dst[3]; int chain_c0[3]; int chain_stages; int fused_into;
};

struct TableEntry {     // t is what the kernels take; its pointers are views of the blocks beside it
    ResizeTables t;
    int canvas;
    DeviceBlock<int32_t> xb, xk, yb, yk;
    DeviceBlock<uint8_t> tmp;
};

}  // namespace

struct b2d_engine {
    int device = 0;
    int max_batch = 0;
    int sm_count = 0;
    bool finalized = false;
    int f16 = 0;                            // 16-bit activation / weight format: 0 bf16 (default), 1 fp16 (b2d_set_precision)
    int x2 = 0;                             // 1: split-fp16 storage (B2D_PREC_FP16X2): every 16-bit activation is an fp16 hi + an fp16 lo part
    std::vector<Buffer> bufs;
    std::vector<OpDesc> descs;
    std::vector<Op> ops;
    // forward() runs a depthwise 3x3 and the 1x1 conv that consumes it as ONE kernel where the pair qualifies (conv_tc_dwpw_kernel):
    // fused_at[i] = index into fused_plans when ops i and i + 1 are such a pair, else -1.  b2d_run_op always runs the single ops.
    std::vector<int> fused_at;
    std::vector<ConvTcPlan> fused_plans;
    HeadDesc head{};
    int head_levels = 0;
    std::vector<TableEntry> tables;
    // post-processing scratch; cand_cap and cand_tiles are 0 until every block below is held at their size
    DeviceBlock<b2d_det> cand;
    DeviceBlock<int> cand_count;
    DeviceBlock<unsigned long long> keys;
    int cand_cap = 0;
    int cand_tiles = 0;
    DeviceBlock<float> cand_angle;          // oriented-box engines: the angle of each candidate slot, beside `cand`
    DeviceBlock<float4> obb_prm;            // ... and the rotated NMS's per-candidate Gaussians (2 float4 per key slot)
    DeviceBlock<void> dedup_scratch;
    DeviceBlock<void> mosaic_nms_scratch;   // b2d_mosaic_nms_obb: per-record frame, Gaussian and grid links, the cell table
    float conf_scale = 1.0f;                // b2d_set_conf_scale: the TTA confidence adjustment (gpu_handler.py:236)
    // test-time-augmentation scratch: CLAHE tile tables / per-image byte tables, per-image grey sums
    DeviceBlock<uint8_t> tta_luts;
    DeviceBlock<unsigned long long> tta_sums;
    // b2d_detect_host: two staging slots (tiles, params, records, counts), a copy stream and the events that order them
    struct HostSlot {
        DeviceBlock<uint8_t> tiles;
        // cap is 0 until every record block is held at its size
        DeviceBlock<double> params; DeviceBlock<b2d_det> dets; DeviceBlock<b2d_geodet> geo; DeviceBlock<int32_t> counts; int cap = 0;
        PinnedBlock<double> params_pin; PinnedBlock<b2d_geodet> geo_pin; PinnedBlock<int32_t> counts_pin;   // pinned host staging
        Event loaded, drained;
    } host_slot[2];
    Stream copy_stream;
    // forward() as a CUDA graph per batch size: the ~94 launches of a step replay without per-launch driver work
    std::map<int, GraphExec> fwd_graphs;
    std::map<int, int> fwd_calls;
    Stream cap_stream;                      // capture happens here (the caller's stream may be the legacy default stream)
    std::vector<Stream> side_streams;       // further capture streams: independent ops become parallel graph branches
    std::vector<Event> cap_events;          // one per op + fork / join events (capture only)
};

namespace {

bool is_obb(const b2d_engine* e) { return e->head_levels > 0 && e->head.kind == B2D_HEAD_V8_OBB; }

// Room for every row of a tile to be a candidate: a tile's candidates are never truncated, larger tiles are refused
int ensure_cand(b2d_engine* e, int n, int rows) {
    B2D_CHECK(rows <= kMaxCand, "postprocess: %d rows per tile exceed the limit of %d (the sort key's 16-bit anchor and slot fields)",
              rows, kMaxCand);
    const int cap = rows;
    if (e->cand_cap >= cap && e->cand_tiles >= n) return 0;
    e->cand_cap = e->cand_tiles = 0;          // every old block goes before any new one is allocated
    e->cand.reset(); e->cand_count.reset(); e->keys.reset(); e->cand_angle.reset(); e->obb_prm.reset();
    const int tiles = n > e->max_batch ? n : e->max_batch;
    const int stride = keys_stride(cap);
    if (e->cand.reserve((size_t)tiles * cap * sizeof(b2d_det)) || e->cand_count.reserve((size_t)tiles * sizeof(int)) ||
        e->keys.reserve((size_t)tiles * stride * sizeof(unsigned long long)))
        return -2;
    if (is_obb(e) && (e->cand_angle.reserve((size_t)tiles * cap * sizeof(float)) ||
                      e->obb_prm.reserve((size_t)tiles * stride * 2 * sizeof(float4))))
        return -2;
    e->cand_cap = cap;
    e->cand_tiles = tiles;
    return 0;
}

int upload_i32(DeviceBlock<int32_t>& dst, const std::vector<int32_t>& v) {
    if (dst.reserve(v.size() * sizeof(int32_t))) return -2;
    B2D_CUDA(cudaMemcpy(dst.get(), v.data(), v.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    return 0;
}

int get_tables(b2d_engine* e, int mode, int h, int w, int out, int n, const ResizeTables** result) {
    TableEntry* te = nullptr;
    for (auto& x : e->tables)
        if (x.t.mode == mode && x.t.in_h == h && x.t.in_w == w && x.canvas == out) { te = &x; break; }
    if (!te) {
        TableEntry ne{};
        ResizeTables& t = ne.t;
        t.mode = mode; t.in_h = h; t.in_w = w; t.out_h = out; t.out_w = out;
        if (mode == B2D_RESIZE_IDENTITY) {
            B2D_CHECK(h == out && w == out, "preprocess: identity mode needs %dx%d input, got %dx%d", out, out, h, w);
        } else {
            int tmode = mode;
            if (mode == B2D_RESIZE_LETTERBOX) {
                // Ultralytics LetterBox(auto=False, scaleup=True, center=True); Python round() = rint()
                const double r = fmin((double)out / h, (double)out / w);
                t.out_w = (int)rint(w * r);
                t.out_h = (int)rint(h * r);
                const double dw = (out - t.out_w) / 2.0, dh = (out - t.out_h) / 2.0;
                t.left = (int)rint(dw - 0.1);
                t.top = (int)rint(dh - 0.1);
                tmode = B2D_RESIZE_CV2_LINEAR;
            }
            int kx = 0, ky = 0;
            b2d_resize_table(tmode, w, t.out_w, nullptr, nullptr, &kx);
            b2d_resize_table(tmode, h, t.out_h, nullptr, nullptr, &ky);
            t.ksize_x = kx; t.ksize_y = ky;
            std::vector<int32_t> xb(2 * (size_t)t.out_w), xk((size_t)kx * t.out_w), yb(2 * (size_t)t.out_h), yk((size_t)ky * t.out_h);
            B2D_CHECK(b2d_resize_table(tmode, w, t.out_w, xb.data(), xk.data(), &kx) == 0, "resize table failed");
            if (tmode == B2D_RESIZE_CV2_LINEAR)       // the row taps follow OpenCV's vertical rule (cv2_linear_coef)
                cv2_linear_axis_table(h, t.out_h, 1, yb.data(), yk.data());
            else
                B2D_CHECK(b2d_resize_table(tmode, h, t.out_h, yb.data(), yk.data(), &ky) == 0, "resize table failed");
            if (upload_i32(ne.xb, xb) || upload_i32(ne.xk, xk) || upload_i32(ne.yb, yb) || upload_i32(ne.yk, yk)) return -2;
            t.xb = ne.xb.get(); t.xk = ne.xk.get(); t.yb = ne.yb.get(); t.yk = ne.yk.get();
        }
        ne.canvas = out;
        e->tables.push_back(std::move(ne));
        te = &e->tables.back();
    }
    ResizeTables& t = te->t;
    if (mode == B2D_RESIZE_PIL_BICUBIC && t.in_w != t.out_w) {
        const int rc = te->tmp.reserve((size_t)n * t.in_h * t.out_w * 3);
        t.tmp = te->tmp.get();
        t.tmp_bytes = te->tmp.bytes();
        if (rc) return rc;
    }
    *result = &t;
    return 0;
}

int launch_op(b2d_engine* e, const Op& op, int n, cudaStream_t s) {
    switch (op.kind) {
        case OP_CONV_TC: return conv_tc_launch(&op.tc, n, s);
        case OP_MAXPOOL:
            return maxpool_launch(op.src, op.h, op.w, op.src_cs, op.src_c0, op.dst, op.oh, op.ow, op.dst_cs, op.dst_c0, op.c, op.k,
                                  op.stride, n, s, e->f16, e->x2);
        case OP_UPSAMPLE: {       // a copy: in split storage a channel is simply 4 bytes instead of 2
            const int m = e->x2 ? 2 : 1;
            return upsample2x_launch(op.src, op.h, op.w, op.src_cs * m, op.src_c0 * m, op.dst, op.dst_cs * m, op.dst_c0 * m, op.c * m, n, s);
        }
        case OP_POOLCHAIN:
            return poolchain_launch(op.src, op.h, op.w, op.src_cs, op.src_c0, op.chain_dst, op.chain_c0, op.dst_cs, op.c, op.chain_stages, n, s, e->f16);
        case OP_NOP: return 0;
    }
    return -1;
}

// op i as forward() runs it: the fused pair kernel where one starts at i, nothing for the second op of a pair
int launch_fwd_op(b2d_engine* e, int i, int n, cudaStream_t s) {
    if (e->fused_at[i] >= 0) return conv_tc_launch(&e->fused_plans[e->fused_at[i]], n, s);
    if (i > 0 && e->fused_at[i - 1] >= 0) return 0;
    return launch_op(e, e->ops[i], n, s);
}

// Launches every op of the plan into the capture: op i goes to the stream of the dependency it continues, or to another
// capture stream when that one has moved on, with event edges for every read-after-write, write-after-read and
// write-after-write between channel ranges of the same buffer.  Independent chains -- the six branches of the
// detect head, head level 0 against the rest of the PAN path -- become parallel branches of the graph, so one
// kernel's CTAs start on the SMs another kernel's tail has already left (each persistent kernel holds a whole SM, so
// nothing else can hide the ~6 us of prologue and tail per launch).
struct Range { int buf, c0, c1; };
static bool overlaps(const Range& a, const Range& b) { return a.buf == b.buf && a.buf >= 0 && a.c0 < b.c1 && b.c0 < a.c1; }

int capture_ops(b2d_engine* e, int n) {
    const int nops = (int)e->ops.size();
    const int ns = 3;                                        // capture streams
    e->side_streams.resize(ns - 1);
    for (auto& s : e->side_streams)
        if (!s && create(s)) return -2;
    e->cap_events.resize(nops + 2 * ns);
    for (auto& ev : e->cap_events)
        if (!ev && create(ev)) return -2;
    auto stream_of = [&](int k) { return k == 0 ? e->cap_stream.get() : e->side_streams[k - 1].get(); };
    // reads / writes of every launched op (a fused pool chain writes its followers' outputs too)
    std::vector<std::vector<Range>> rd(nops), wr(nops);
    for (int i = 0; i < nops; ++i) {
        const OpDesc& d = e->descs[i];
        const int cin = d.kind_req == 0 ? d.cin : d.cout;
        if (e->fused_at[i] >= 0) {                        // depthwise + pointwise pair: reads the depthwise source, writes the pointwise output
            rd[i].push_back({d.src, d.src_c0, d.src_c0 + cin});
            continue;
        }
        if (i > 0 && e->fused_at[i - 1] >= 0) {
            wr[i - 1].push_back({d.dst, d.dst_c0, d.dst_c0 + d.cout});
            continue;
        }
        const int owner = e->ops[i].kind == OP_NOP ? e->ops[i].fused_into : i;
        if (owner == i) rd[i].push_back({d.src, d.src_c0, d.src_c0 + cin});
        if (d.res >= 0) rd[owner].push_back({d.res, d.res_c0, d.res_c0 + d.cout});
        wr[owner].push_back({d.dst, d.dst_c0, d.dst_c0 + d.cout});
    }
    std::vector<int> where(nops, -1), last_on(ns, -1);
    std::vector<bool> joined(ns, false);
    joined[0] = true;
    cudaEvent_t fork_ev = e->cap_events[nops].get();
    B2D_CUDA(cudaEventRecord(fork_ev, e->cap_stream.get()));
    for (int i = 0; i < nops; ++i) {
        if (e->ops[i].kind == OP_NOP || (i > 0 && e->fused_at[i - 1] >= 0)) continue;
        std::vector<int> deps;
        for (int j = 0; j < i; ++j) {
            if (where[j] < 0) continue;
            bool dep = false;
            for (const Range& w : wr[j]) {
                for (const Range& r : rd[i]) dep = dep || overlaps(w, r);
                for (const Range& w2 : wr[i]) dep = dep || overlaps(w, w2);
            }
            for (const Range& r : rd[j])
                for (const Range& w2 : wr[i]) dep = dep || overlaps(r, w2);
            if (dep) deps.push_back(j);
        }
        int k = -1;
        for (int j : deps)                                   // continue the chain of the latest dependency that is still the tail of its stream
            if (last_on[where[j]] == j) k = where[j];
        if (k < 0) {                                         // otherwise the stream that has been idle longest
            k = 0;
            for (int t = 1; t < ns; ++t)
                if (last_on[t] < last_on[k]) k = t;
        }
        cudaStream_t s = stream_of(k);
        if (!joined[k]) {
            B2D_CUDA(cudaStreamWaitEvent(s, fork_ev, 0));
            joined[k] = true;
        }
        for (int j : deps)
            if (where[j] != k) B2D_CUDA(cudaStreamWaitEvent(s, e->cap_events[j].get(), 0));
        if (int r = launch_fwd_op(e, i, n, s)) return r;
        B2D_CUDA(cudaEventRecord(e->cap_events[i].get(), s));
        where[i] = k;
        last_on[k] = i;
    }
    for (int t = 1; t < ns; ++t)
        if (joined[t]) {
            B2D_CUDA(cudaEventRecord(e->cap_events[nops + 1 + t].get(), stream_of(t)));
            B2D_CUDA(cudaStreamWaitEvent(e->cap_stream.get(), e->cap_events[nops + 1 + t].get(), 0));
        }
    return 0;
}

}  // namespace

extern "C" {

const char* b2d_last_error(void) { return g_last_error.c_str(); }
int b2d_version(void) { return B2D_VERSION; }

int b2d_create(int device, int max_batch, b2d_engine** out) {
    B2D_CHECK(out != nullptr && max_batch > 0, "b2d_create: bad arguments");
    int count = 0;
    cudaError_t err = cudaGetDeviceCount(&count);
    B2D_CHECK(err == cudaSuccess && count > 0, "b2d_create: no CUDA device (%s) -- this engine has no CPU fallback",
              cudaGetErrorString(err));
    B2D_CHECK(device >= 0 && device < count, "b2d_create: device %d out of range (%d devices)", device, count);
    cudaDeviceProp prop;
    B2D_CUDA(cudaGetDeviceProperties(&prop, device));
    B2D_CHECK(prop.major == 10, "b2d_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major,
              prop.minor);
    DeviceGuard guard(device);
    b2d_engine* e = new b2d_engine();
    e->device = device;
    e->max_batch = max_batch;
    e->sm_count = prop.multiProcessorCount;
    *out = e;
    return 0;
}

void b2d_destroy(b2d_engine* e) {
    if (!e) return;
    B2D_ENTER(e);      // declared before the delete, so every member is released with the engine's device current
    delete e;
}

int b2d_device_sm_count(b2d_engine* e) { return e ? e->sm_count : -1; }

int b2d_set_precision(b2d_engine* e, int precision) {
    B2D_CHECK(e && !e->finalized && e->descs.empty(), "set_precision: call right after b2d_create, before planning");
    B2D_CHECK(precision == B2D_PREC_BF16 || precision == B2D_PREC_FP16 || precision == B2D_PREC_FP16X2, "set_precision: unknown precision %d", precision);
    B2D_CHECK(e->bufs.empty(), "set_precision: call before b2d_plan_buffer (the storage width of every buffer depends on it)");
    e->f16 = precision != B2D_PREC_BF16;
    e->x2 = precision == B2D_PREC_FP16X2;
    return 0;
}
int b2d_get_precision(b2d_engine* e) { return e ? (e->x2 ? B2D_PREC_FP16X2 : e->f16 ? B2D_PREC_FP16 : B2D_PREC_BF16) : -1; }

int b2d_plan_buffer(b2d_engine* e, int h, int w, int c, int is_f32) {
    B2D_CHECK(e && !e->finalized, "plan_buffer: engine finalized or null");
    B2D_CHECK(h > 0 && w > 0 && c > 0, "plan_buffer: bad shape");
    B2D_ENTER(e);
    Buffer b{h, w, c, is_f32};
    // bytes per channel: 4 (fp32 head maps), 2 (bf16 / fp16), or 2 + 2 in split storage -- except buffer 0, the network
    // input, which holds raw pixel values (exact in 16 bits) in every mode
    const bool split = e->x2 && !is_f32 && !e->bufs.empty();
    if (b.ptr.reserve((size_t)e->max_batch * h * w * c * ((is_f32 || split) ? 4 : 2))) return -2;
    B2D_CUDA(cudaMemset(b.ptr.get(), 0, b.ptr.bytes()));
    e->bufs.push_back(std::move(b));
    return (int)e->bufs.size() - 1;
}

static int check_ref(b2d_engine* e, int buf, int c0, int c, const char* what) {
    B2D_CHECK(buf >= 0 && buf < (int)e->bufs.size(), "%s: buffer %d out of range", what, buf);
    B2D_CHECK(c0 >= 0 && c > 0 && c0 + c <= e->bufs[buf].c, "%s: slice [%d,%d) outside buffer with %d channels", what, c0, c0 + c,
              e->bufs[buf].c);
    return 0;
}

int b2d_plan_conv(b2d_engine* e, int src, int src_c0, int cin, int dst, int dst_c0, int cout, int k, int stride, int act,
                  const float* weight_host, const float* bias_host, int res, int res_c0, int impl) {
    B2D_CHECK(e && !e->finalized, "plan_conv: engine finalized or null");
    if (check_ref(e, src, src_c0, src == 0 ? e->bufs[0].c : cin, "plan_conv src") || check_ref(e, dst, dst_c0, cout, "plan_conv dst")) return -1;
    if (res >= 0 && check_ref(e, res, res_c0, cout, "plan_conv res")) return -1;
    B2D_CHECK(weight_host != nullptr, "plan_conv: weights missing");
    const Buffer& sb = e->bufs[src];
    const Buffer& db = e->bufs[dst];
    B2D_CHECK((sb.h + 2 * (k / 2) - k) / stride + 1 == db.h && (sb.w + 2 * (k / 2) - k) / stride + 1 == db.w,
              "plan_conv: %dx%d -k%d s%d-> %dx%d does not match", sb.h, sb.w, k, stride, db.h, db.w);
    B2D_CHECK(!sb.f32, "plan_conv: source must be bf16");
    B2D_CHECK(res < 0 || (!e->bufs[res].f32 && e->bufs[res].h == db.h && e->bufs[res].w == db.w), "plan_conv: bad residual buffer");
    OpDesc d{};
    d.kind_req = 0; d.src = src; d.src_c0 = src_c0; d.cin = cin; d.dst = dst; d.dst_c0 = dst_c0; d.cout = cout;
    d.k = k; d.stride = stride; d.act = act; d.res = res; d.res_c0 = res_c0; d.impl = impl;
    d.w.assign(weight_host, weight_host + (size_t)cout * cin * k * k);
    if (bias_host) d.b.assign(bias_host, bias_host + cout);
    else d.b.assign(cout, 0.f);
    e->descs.push_back(std::move(d));
    return (int)e->descs.size() - 1;
}

int b2d_plan_dwconv(b2d_engine* e, int src, int src_c0, int dst, int dst_c0, int c, int act, const float* weight_host,
                    const float* bias_host) {
    B2D_CHECK(e && !e->finalized, "plan_dwconv: engine finalized or null");
    if (check_ref(e, src, src_c0, c, "plan_dwconv src") || check_ref(e, dst, dst_c0, c, "plan_dwconv dst")) return -1;
    B2D_CHECK(e->bufs[src].h == e->bufs[dst].h && e->bufs[src].w == e->bufs[dst].w, "plan_dwconv: shape mismatch");
    B2D_CHECK(!e->bufs[src].f32 && !e->bufs[dst].f32, "plan_dwconv: buffers must be bf16");
    OpDesc d{};
    d.kind_req = 1; d.src = src; d.src_c0 = src_c0; d.cin = c; d.dst = dst; d.dst_c0 = dst_c0; d.cout = c; d.k = 3; d.stride = 1;
    d.act = act; d.res = -1;
    d.w.assign(weight_host, weight_host + (size_t)c * 9);
    if (bias_host) d.b.assign(bias_host, bias_host + c);
    else d.b.assign(c, 0.f);
    e->descs.push_back(std::move(d));
    return (int)e->descs.size() - 1;
}

int b2d_plan_maxpool(b2d_engine* e, int src, int src_c0, int dst, int dst_c0, int c, int k, int stride) {
    B2D_CHECK(e && !e->finalized, "plan_maxpool: engine finalized or null");
    if (check_ref(e, src, src_c0, c, "plan_maxpool src") || check_ref(e, dst, dst_c0, c, "plan_maxpool dst")) return -1;
    const Buffer& sb = e->bufs[src];
    const Buffer& db = e->bufs[dst];
    const int oh = (stride == 1) ? sb.h : sb.h / stride;
    B2D_CHECK(oh == db.h && !sb.f32 && !db.f32, "plan_maxpool: shape/type mismatch");
    OpDesc d{};
    d.kind_req = 2; d.src = src; d.src_c0 = src_c0; d.cin = c; d.dst = dst; d.dst_c0 = dst_c0; d.cout = c; d.k = k; d.stride = stride; d.res = -1;
    e->descs.push_back(std::move(d));
    return (int)e->descs.size() - 1;
}

int b2d_plan_upsample2x(b2d_engine* e, int src, int src_c0, int dst, int dst_c0, int c) {
    B2D_CHECK(e && !e->finalized, "plan_upsample: engine finalized or null");
    if (check_ref(e, src, src_c0, c, "plan_upsample src") || check_ref(e, dst, dst_c0, c, "plan_upsample dst")) return -1;
    B2D_CHECK(e->bufs[src].h * 2 == e->bufs[dst].h && !e->bufs[src].f32 && !e->bufs[dst].f32, "plan_upsample: shape/type mismatch");
    OpDesc d{};
    d.kind_req = 3; d.src = src; d.src_c0 = src_c0; d.cin = c; d.dst = dst; d.dst_c0 = dst_c0; d.cout = c; d.res = -1;
    e->descs.push_back(std::move(d));
    return (int)e->descs.size() - 1;
}

int b2d_plan_head_level(b2d_engine* e, int kind, int buf, int stride, int nc, const float* anchors_px) {
    B2D_CHECK(e && !e->finalized, "plan_head_level: engine finalized or null");
    B2D_CHECK(buf >= 0 && buf < (int)e->bufs.size() && e->bufs[buf].f32, "plan_head_level: head buffer must be an fp32 buffer");
    B2D_CHECK(e->head_levels < 3, "plan_head_level: at most 3 levels");
    B2D_CHECK(e->head_levels == 0 || (e->head.kind == kind && e->head.nc == nc), "plan_head_level: inconsistent head");
    const Buffer& b = e->bufs[buf];
    HeadLevel& L = e->head.lv[e->head_levels];
    L.buf = (const float*)b.ptr.get(); L.hw = b.h; L.c = b.c; L.stride = stride;
    for (int i = 0; i < 6; ++i) L.anchors[i] = anchors_px ? anchors_px[i] : 0.f;
    B2D_CHECK(kind == B2D_HEAD_V8_DFL || kind == B2D_HEAD_V7_ANCHOR || kind == B2D_HEAD_V8_OBB, "plan_head_level: unknown head kind %d", kind);
    const int per = (kind == B2D_HEAD_V7_ANCHOR) ? 3 : 1;
    L.row0 = e->head.rows_total;
    const int need = kind == B2D_HEAD_V7_ANCHOR ? 3 * (nc + 5) : kind == B2D_HEAD_V8_OBB ? obb_angle_channel(nc) + 1 : 64 + nc;
    B2D_CHECK(b.c >= need, "plan_head_level: head buffer too narrow (%d channels, the head needs %d)", b.c, need);
    e->head.rows_total += per * b.h * b.w;
    e->head.kind = kind; e->head.nc = nc;
    e->head_levels += 1;
    e->head.nlevels = e->head_levels;
    return 0;
}

int b2d_plan_finalize(b2d_engine* e) {
    B2D_CHECK(e && !e->finalized, "plan_finalize: engine finalized or null");
    B2D_ENTER(e);
    e->ops.resize(e->descs.size());
    for (size_t i = 0; i < e->descs.size(); ++i) {
        OpDesc& d = e->descs[i];
        Op& op = e->ops[i];
        const Buffer& sb = e->bufs[d.src];
        const Buffer& db = e->bufs[d.dst];
        if (d.kind_req == 0) {
            const __nv_bfloat16* res = d.res >= 0 ? (const __nv_bfloat16*)e->bufs[d.res].ptr.get() : nullptr;
            const int res_cs = d.res >= 0 ? e->bufs[d.res].c : 0;
            const bool tc = (conv_tc_supported(d.cin, d.k, d.stride) && sb.c % 8 == 0 && d.src_c0 % 8 == 0) ||
                            (conv_tc_stem_supported(sb.c, d.cin, d.k, d.stride, d.cout, db.f32, d.res >= 0) && d.src_c0 == 0);
            // one backend: a shape the tensor-core kernels cannot run is an error, never a slower path
            B2D_CHECK(d.impl == B2D_CONV_AUTO || d.impl == B2D_CONV_TCGEN05, "plan_finalize: op %zu asks for conv implementation %d; only tcgen05 exists", i, d.impl);
            B2D_CHECK(tc, "plan_finalize: op %zu (conv k%d s%d cin %d, source slice %d of %d channels) has no tcgen05 kernel", i, d.k, d.stride,
                      d.cin, d.src_c0, sb.c);
            op.kind = OP_CONV_TC;
            // the network input holds raw 0..255 pixel values: the reference's `/ 255.0` is the stem's accumulator scale
            const float acc_scale = d.src == 0 ? 1.0f / 255.0f : 1.0f;
            if (conv_tc_plan(&op.tc, e->sm_count, e->max_batch, (const __nv_bfloat16*)sb.ptr.get(), sb.h, sb.w, sb.c, d.src_c0, d.cin,
                             db.ptr.get(), db.h, db.w, db.c, d.dst_c0, d.cout, db.f32, d.k, d.stride, d.act, d.w.data(), d.b.data(), res,
                             res_cs, d.res_c0, 0, e->f16, e->x2, acc_scale))
                return -1;
        } else if (d.kind_req == 1) {
            B2D_CHECK(conv_tc_dw_supported(d.cin, d.cout, 3, 1, db.f32, 0) && sb.c % 8 == 0 && d.src_c0 % 8 == 0,
                      "plan_finalize: op %zu (depthwise, %d channels) has no tcgen05 kernel", i, d.cin);
            op.kind = OP_CONV_TC;
            if (conv_tc_plan(&op.tc, e->sm_count, e->max_batch, (const __nv_bfloat16*)sb.ptr.get(), sb.h, sb.w, sb.c, d.src_c0, d.cin, db.ptr.get(), db.h,
                             db.w, db.c, d.dst_c0, d.cout, 0, 3, 1, d.act, d.w.data(), d.b.data(), nullptr, 0, 0, 1, e->f16, e->x2))
                return -1;
        } else {
            op.kind = d.kind_req == 2 ? OP_MAXPOOL : OP_UPSAMPLE;
            op.src = (const __nv_bfloat16*)sb.ptr.get(); op.dst = (__nv_bfloat16*)db.ptr.get();
            op.h = sb.h; op.w = sb.w; op.src_cs = sb.c; op.src_c0 = d.src_c0;
            op.oh = db.h; op.ow = db.w; op.dst_cs = db.c; op.dst_c0 = d.dst_c0; op.c = d.cout; op.k = d.k; op.stride = d.stride;
        }
        if (op.kind == OP_CONV_TC) op.tc.p.rev = (int)(i & 1);     // odd ops walk their tiles backwards (see conv_tc_launch)
    }
    // Depthwise 3x3 followed by the 1x1 conv that is its only reader -> one kernel in forward().
    e->fused_at.assign(e->descs.size(), -1);
    e->fused_plans.reserve(e->descs.size());
    for (size_t i = 0; i + 1 < e->descs.size(); ++i) {
        const OpDesc& d0 = e->descs[i];
        const OpDesc& d1 = e->descs[i + 1];
        if (d0.kind_req != 1 || d1.kind_req != 0 || d1.k != 1 || d1.stride != 1 || d1.res >= 0) continue;
        if (d1.src != d0.dst || d1.src_c0 != d0.dst_c0 || d1.cin != d0.cout) continue;
        const Buffer& sb = e->bufs[d0.src];
        const Buffer& db = e->bufs[d1.dst];
        if (!conv_tc_dwpw_supported(d0.cout, d1.cout, db.f32, e->x2) || sb.c % 8 != 0 || d0.src_c0 % 8 != 0) continue;
        if (e->ops[i].tc.p.bw != 8) continue;            // the depthwise plan's tile is the fused kernel's tile
        bool other_reader = false;                        // the intermediate must have no other consumer
        for (size_t j = 0; j < e->descs.size(); ++j) {
            if (j == i + 1) continue;
            const OpDesc& dj = e->descs[j];
            const int cj = dj.kind_req == 0 ? dj.cin : dj.cout;
            if (dj.src == d0.dst && dj.src_c0 < d0.dst_c0 + d0.cout && d0.dst_c0 < dj.src_c0 + cj) other_reader = true;
            if (dj.res == d0.dst && dj.res_c0 < d0.dst_c0 + d0.cout && d0.dst_c0 < dj.res_c0 + dj.cout) other_reader = true;
            if (j != i && dj.dst == d0.dst && dj.dst_c0 < d0.dst_c0 + d0.cout && d0.dst_c0 < dj.dst_c0 + dj.cout) other_reader = true;   // or another writer
        }
        if (other_reader) continue;
        DwFuse fz{(const __nv_bfloat16*)sb.ptr.get(), sb.c, d0.src_c0, d0.w.data(), d0.b.data(), d0.act};
        ConvTcPlan fp;
        if (conv_tc_plan(&fp, e->sm_count, e->max_batch, nullptr, sb.h, sb.w, 0, 0, d1.cin, db.ptr.get(), db.h, db.w, db.c, d1.dst_c0, d1.cout, 0, 1, 1,
                         d1.act, d1.w.data(), d1.b.data(), nullptr, 0, 0, 0, e->f16, 0, 1.0f, &fz))
            return -1;
        fp.p.rev = e->ops[i].tc.p.rev;
        e->fused_at[i] = (int)e->fused_plans.size();
        e->fused_plans.push_back(std::move(fp));
        ++i;
    }
    for (auto& d : e->descs) { d.w.clear(); d.w.shrink_to_fit(); }
    // Fuse chains of stride-1 max-pools into one launch: SPPF (mp5 of mp5 of mp5) and SPPCSPC (mp5, mp9, mp13 of one
    // source, which are the same three tensors because max-pooling with -inf padding composes).
    for (size_t i = 0; i + 1 < e->ops.size(); ++i) {
        Op& a = e->ops[i];
        if (e->x2) break;                        // split storage: the pools run one by one (maxpool_x2_kernel)
        if (a.kind != OP_MAXPOOL || a.stride != 1 || a.k != 5) continue;
        if (!poolchain_fits(a.h, a.w)) continue;
        int stages = 1;
        a.chain_dst[0] = a.dst; a.chain_c0[0] = a.dst_c0;
        while (stages < 3 && i + stages < e->ops.size()) {
            const Op& b = e->ops[i + stages];
            const Op& prev = e->ops[i + stages - 1];
            if (b.kind != OP_MAXPOOL || b.stride != 1 || b.c != a.c || b.dst != a.dst || b.dst_cs != a.dst_cs) break;
            const bool sppf = b.k == 5 && b.src == prev.dst && b.src_c0 == prev.dst_c0 && b.src_cs == prev.dst_cs;
            const bool spp = b.k == 5 + 4 * stages && b.src == a.src && b.src_c0 == a.src_c0;
            if (!sppf && !spp) break;
            a.chain_dst[stages] = b.dst; a.chain_c0[stages] = b.dst_c0;
            ++stages;
        }
        if (stages == 1) continue;
        a.kind = OP_POOLCHAIN;
        a.chain_stages = stages;
        for (int j = 1; j < stages; ++j) { e->ops[i + j].kind = OP_NOP; e->ops[i + j].fused_into = (int)i; }
        i += stages - 1;
    }
    e->finalized = true;
    return 0;
}

void* b2d_buffer_ptr(b2d_engine* e, int buf) { return (e && buf >= 0 && buf < (int)e->bufs.size()) ? e->bufs[buf].ptr.get() : nullptr; }
size_t b2d_buffer_bytes(b2d_engine* e, int buf) { return (e && buf >= 0 && buf < (int)e->bufs.size()) ? e->bufs[buf].ptr.bytes() : 0; }
int b2d_num_anchors(b2d_engine* e) { return e ? e->head.rows_total : -1; }
int b2d_num_ops(b2d_engine* e) { return e ? (int)e->ops.size() : -1; }
int b2d_num_kernels_per_forward(b2d_engine* e) {
    if (!e) return -1;
    int k = 0;
    for (const Op& op : e->ops) k += op.kind != OP_NOP;
    for (int f : e->fused_at) k -= f >= 0;
    return k;
}

int b2d_describe_op(b2d_engine* e, int i, char* buf, int buflen) {
    B2D_CHECK(e && e->finalized && i >= 0 && i < (int)e->ops.size(), "describe_op: bad index");
    const Op& op = e->ops[i];
    switch (op.kind) {
        case OP_CONV_TC: return conv_tc_describe(&op.tc, buf, buflen);
        case OP_MAXPOOL: return snprintf(buf, buflen, "maxpool k%d s%d c %d @ %dx%d", op.k, op.stride, op.c, op.h, op.w);
        case OP_UPSAMPLE: return snprintf(buf, buflen, "upsample2x c %d @ %dx%d", op.c, op.h, op.w);
        case OP_POOLCHAIN: return snprintf(buf, buflen, "maxpool chain x%d (k5 s1 composed) c %d @ %dx%d", op.chain_stages, op.c, op.h, op.w);
        case OP_NOP: return snprintf(buf, buflen, "maxpool k%d s1 c %d @ %dx%d (fused into op %d)", op.k, op.c, op.h, op.w, op.fused_into);
    }
    return 0;
}

int b2d_run_op(b2d_engine* e, int i, int n, void* stream) {
    B2D_CHECK(e && e->finalized && i >= 0 && i < (int)e->ops.size(), "run_op: bad index");
    B2D_CHECK(n > 0 && n <= e->max_batch, "run_op: n=%d outside [1,%d]", n, e->max_batch);
    B2D_ENTER(e);
    return launch_op(e, e->ops[i], n, (cudaStream_t)stream);
}

int b2d_fused_with_next(b2d_engine* e, int i) {
    if (!e || !e->finalized || i < 0 || i >= (int)e->fused_at.size()) return -1;
    return e->fused_at[i] >= 0 ? 1 : 0;
}

int b2d_run_op_fused(b2d_engine* e, int i, int n, void* stream) {
    B2D_CHECK(e && e->finalized && i >= 0 && i < (int)e->ops.size(), "run_op_fused: bad index");
    B2D_CHECK(e->fused_at[i] >= 0, "run_op_fused: op %d does not start a fused pair", i);
    B2D_CHECK(n > 0 && n <= e->max_batch, "run_op_fused: n=%d outside [1,%d]", n, e->max_batch);
    B2D_ENTER(e);
    return conv_tc_launch(&e->fused_plans[e->fused_at[i]], n, (cudaStream_t)stream);
}

int b2d_forward(b2d_engine* e, int n, void* stream) {
    B2D_CHECK(e && e->finalized, "forward: plan not finalized");
    B2D_CHECK(n > 0 && n <= e->max_batch, "forward: n=%d outside [1,%d]", n, e->max_batch);
    B2D_ENTER(e);
    cudaStream_t st = (cudaStream_t)stream;
    static const bool use_graph = !getenv("B2D_TRACE");      // conv_tc_launch resets and reads back the role trace per launch
    auto it = e->fwd_graphs.find(n);
    if (use_graph && it != e->fwd_graphs.end()) {
        B2D_CUDA(cudaGraphLaunch(it->second.get(), st));
        return 0;
    }
    // the first call of a batch size runs eagerly (function attributes, lazy module loading); the second is captured
    const bool capture = use_graph && e->fwd_calls[n]++ >= 1;
    if (capture) {
        if (!e->cap_stream && create(e->cap_stream)) return -2;
        B2D_CUDA(cudaStreamBeginCapture(e->cap_stream.get(), cudaStreamCaptureModeThreadLocal));
    }
    int rc = 0;
    if (!capture) {
        for (int i = 0; i < (int)e->ops.size(); ++i)
            if ((rc = launch_fwd_op(e, i, n, st)) != 0) break;
    } else {
        rc = capture_ops(e, n);
    }
    if (capture) {
        cudaGraph_t g = nullptr;
        cudaError_t err = cudaStreamEndCapture(e->cap_stream.get(), &g);
        if (rc == 0 && err == cudaSuccess && g) {
            cudaGraphExec_t ex = nullptr;
            if (cudaGraphInstantiate(&ex, g, 0) == cudaSuccess) {
                e->fwd_graphs[n].reset(ex);
                cudaGraphDestroy(g);
                B2D_CUDA(cudaGraphLaunch(ex, st));
                return 0;
            }
        }
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        B2D_CHECK(rc == 0, "forward: launch failed during graph capture");
        for (int i = 0; i < (int)e->ops.size(); ++i)    // capture or instantiation failed: plain launches
            if (int r = launch_fwd_op(e, i, n, st)) return r;
        return 0;
    }
    return rc;
}

int b2d_preprocess(b2d_engine* e, const uint8_t* src_dev, int n, int h, int w, int pitch, long long img_stride, int mode, int bgr,
                   int out_kind, void* dst_dev, void* stream) {
    B2D_CHECK(e && src_dev && n > 0, "preprocess: bad arguments");
    B2D_ENTER(e);
    B2D_CHECK(pitch >= w * 3, "preprocess: pitch %d < row bytes %d", pitch, w * 3);
    int out = 640;
    if (!e->bufs.empty()) out = e->bufs[0].h;
    if (out_kind == B2D_OUT_BF16_NHWC4 && e->f16 && dst_dev == nullptr) out_kind = B2D_OUT_F16_NHWC4;   // the engine's own input format
    if (dst_dev == nullptr) {
        B2D_CHECK((out_kind == B2D_OUT_BF16_NHWC4 || out_kind == B2D_OUT_F16_NHWC4) && !e->bufs.empty() && e->bufs[0].c == 4 && !e->bufs[0].f32,
                  "preprocess: dst NULL needs the planned 16-bit NHWC4 input buffer");
        B2D_CHECK(n <= e->max_batch, "preprocess: n=%d exceeds max_batch %d", n, e->max_batch);
        dst_dev = e->bufs[0].ptr.get();
    }
    const ResizeTables* t = nullptr;
    if (get_tables(e, mode, h, w, out, n, &t)) return -1;
    return preprocess_launch(t, src_dev, n, pitch, img_stride, bgr, out_kind, dst_dev, out, (cudaStream_t)stream);
}

int b2d_set_input_f32(b2d_engine* e, const float* src_dev, int n, void* stream) {
    B2D_CHECK(e && src_dev && n > 0 && n <= e->max_batch, "set_input_f32: bad arguments");
    B2D_ENTER(e);
    B2D_CHECK(!e->bufs.empty() && e->bufs[0].c == 4 && !e->bufs[0].f32, "set_input_f32: no planned bf16 NHWC4 input buffer");
    return input_from_f32_launch(src_dev, n, e->bufs[0].h, e->bufs[0].w, e->bufs[0].ptr.get(), (cudaStream_t)stream, e->f16);
}

int b2d_decode_rows(b2d_engine* e, int n, float* rows_dev, void* stream) {
    B2D_CHECK(e && e->finalized && e->head_levels > 0, "decode_rows: no head planned");
    B2D_CHECK(!is_obb(e), "decode_rows: the engine has an oriented-box head; use b2d_decode_rows_obb");
    B2D_ENTER(e);
    B2D_CHECK(n > 0 && n <= e->max_batch && rows_dev, "decode_rows: bad arguments");
    return decode_rows_launch(&e->head, n, rows_dev, (cudaStream_t)stream);
}

int b2d_postprocess(b2d_engine* e, int n, float conf_thr, int inclusive, float iou_thr, int top_k, int max_det, b2d_det* dets_dev,
                    int32_t* counts_dev, int cap, void* stream) {
    B2D_CHECK(e && e->finalized && e->head_levels > 0, "postprocess: no head planned");
    B2D_CHECK(!is_obb(e), "postprocess: the engine has an oriented-box head; use b2d_postprocess_obb");
    B2D_ENTER(e);
    B2D_CHECK(n > 0 && n <= e->max_batch && dets_dev && counts_dev && cap > 0, "postprocess: bad arguments");
    if (int rc = ensure_cand(e, n, e->head.rows_total)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (candidates_from_head_launch(&e->head, n, conf_thr, inclusive, e->conf_scale, e->cand.get(), e->cand_count.get(), e->cand_cap, s)) return -2;
    return select_launch(e->cand.get(), e->cand_count.get(), e->cand_cap, n, e->keys.get(), iou_thr, top_k, max_det, dets_dev, counts_dev, cap, s);
}

int b2d_postprocess_rows(b2d_engine* e, const float* rows_dev, int n, int num_rows, int ncol, float conf_thr, int inclusive,
                         float iou_thr, int top_k, int max_det, b2d_det* dets_dev, int32_t* counts_dev, int cap, void* stream) {
    B2D_CHECK(e && rows_dev && n > 0 && num_rows > 0 && ncol >= 5 && dets_dev && counts_dev && cap > 0, "postprocess_rows: bad arguments");
    B2D_CHECK(!is_obb(e), "postprocess_rows: the engine has an oriented-box head; axis-aligned rows are not its output");
    B2D_ENTER(e);
    if (int rc = ensure_cand(e, n, num_rows)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (candidates_from_rows_launch(rows_dev, n, num_rows, ncol, conf_thr, inclusive, e->conf_scale, e->cand.get(), e->cand_count.get(), e->cand_cap, s)) return -2;
    return select_launch(e->cand.get(), e->cand_count.get(), e->cand_cap, n, e->keys.get(), iou_thr, top_k, max_det, dets_dev, counts_dev, cap, s);
}

int b2d_segment(b2d_engine* e, int buf, int n, int nc, uint8_t* labels_dev, float* conf_dev, void* stream) {
    B2D_CHECK(e && e->finalized && buf >= 0 && buf < (int)e->bufs.size() && labels_dev, "segment: bad arguments");
    B2D_CHECK(n > 0 && n <= e->max_batch, "segment: n=%d outside [1,%d]", n, e->max_batch);
    const Buffer& b = e->bufs[buf];
    B2D_CHECK(b.f32, "segment: buffer %d is not an fp32 logits buffer", buf);
    B2D_ENTER(e);
    return segment_launch((const float*)b.ptr.get(), (long long)n * b.h * b.w, b.c, nc, labels_dev, conf_dev, (cudaStream_t)stream);
}

int b2d_georef(b2d_engine* e, const b2d_det* dets_dev, const int32_t* counts_dev, int n, int cap, int mode, const double* params_dev,
               b2d_geodet* out_dev, void* stream) {
    B2D_CHECK(e && dets_dev && counts_dev && params_dev && out_dev, "georef: bad arguments");
    B2D_ENTER(e);
    B2D_CHECK(mode >= 0 && mode <= 3, "georef: unknown mode %d", mode);
    B2D_CHECK(!is_obb(e), "georef: the engine has an oriented-box head; use b2d_georef_obb");
    return georef_launch(dets_dev, counts_dev, n, cap, mode, params_dev, out_dev, (cudaStream_t)stream);
}

int b2d_decode_rows_obb(b2d_engine* e, int n, float* rows_dev, void* stream) {
    B2D_CHECK(e && e->finalized && e->head_levels > 0, "decode_rows_obb: no head planned");
    B2D_CHECK(is_obb(e), "decode_rows_obb: the engine has no oriented-box head; use b2d_decode_rows");
    B2D_ENTER(e);
    B2D_CHECK(n > 0 && n <= e->max_batch && rows_dev, "decode_rows_obb: bad arguments");
    return obb_decode_rows_launch(&e->head, n, rows_dev, (cudaStream_t)stream);
}

int b2d_postprocess_obb(b2d_engine* e, int n, float conf_thr, int inclusive, float iou_thr, int top_k, int max_det, b2d_obb* dets_dev,
                        int32_t* counts_dev, int cap, void* stream) {
    B2D_CHECK(e && e->finalized && e->head_levels > 0, "postprocess_obb: no head planned");
    B2D_CHECK(is_obb(e), "postprocess_obb: the engine has no oriented-box head; use b2d_postprocess");
    B2D_ENTER(e);
    B2D_CHECK(n > 0 && n <= e->max_batch && dets_dev && counts_dev && cap > 0, "postprocess_obb: bad arguments");
    if (int rc = ensure_cand(e, n, e->head.rows_total)) return rc;
    return obb_postprocess_launch(&e->head, n, conf_thr, inclusive, e->conf_scale, e->cand.get(), e->cand_angle.get(), e->cand_count.get(), e->cand_cap,
                                  e->keys.get(), e->obb_prm.get(), iou_thr, top_k, max_det, dets_dev, counts_dev, cap, (cudaStream_t)stream);
}

int b2d_georef_obb(b2d_engine* e, const b2d_obb* dets_dev, const int32_t* counts_dev, int n, int cap, int mode, const double* params_dev,
                   b2d_geoobb* out_dev, void* stream) {
    B2D_CHECK(e && dets_dev && counts_dev && params_dev && out_dev, "georef_obb: bad arguments");
    B2D_CHECK(is_obb(e), "georef_obb: the engine has no oriented-box head; use b2d_georef");
    B2D_CHECK(mode == B2D_GEO_BOUNDS || mode == B2D_GEO_AFFINE, "georef_obb: form %d has no oriented-box variant (bounds and affine do)", mode);
    B2D_ENTER(e);
    return obb_georef_launch(dets_dev, counts_dev, n, cap, mode, params_dev, out_dev, (cudaStream_t)stream);
}

int b2d_mosaic_nms_obb(b2d_engine* e, const b2d_obb* dets_dev, const int32_t* counts_dev, const double* params_dev, int n, int cap,
                       float conf_thr, float iou_thr, uint8_t* keep_dev, void* stream) {
    B2D_CHECK(e, "mosaic_nms_obb: bad arguments");
    B2D_CHECK(is_obb(e), "mosaic_nms_obb: the engine has no oriented-box head; the merge takes b2d_obb records");
    B2D_CHECK(iou_thr > 0.f && iou_thr < 1.f, "mosaic_nms_obb: iou_thr %g is outside (0, 1)", (double)iou_thr);
    B2D_CHECK(n >= 0 && cap > 0, "mosaic_nms_obb: bad arguments (n %d, cap %d)", n, cap);
    B2D_CHECK((long long)n * cap <= INT_MAX, "mosaic_nms_obb: %d windows x %d records exceed the %d records of one call", n, cap, INT_MAX);
    B2D_ENTER(e);
    if (n == 0) return 0;
    B2D_CHECK(dets_dev && counts_dev && params_dev && keep_dev, "mosaic_nms_obb: bad arguments");
    if (e->mosaic_nms_scratch.reserve(mosaic_nms_obb_scratch_bytes(n * cap))) return -2;
    return mosaic_nms_obb_launch(dets_dev, counts_dev, params_dev, n, cap, conf_thr, iou_thr, keep_dev, e->mosaic_nms_scratch.get(),
                                 e->mosaic_nms_scratch.bytes(), (cudaStream_t)stream);
}

int b2d_dedup(b2d_engine* e, const double* x_dev, const double* y_dev, const float* conf_dev, const long long* tiebreak_dev, int count,
              double thr, int inclusive, uint8_t* keep_dev, void* stream) {
    B2D_CHECK(e && (count == 0 || (x_dev && y_dev && conf_dev && keep_dev)), "dedup: bad arguments");
    B2D_ENTER(e);
    if (count == 0) return 0;
    if (e->dedup_scratch.reserve(dedup_scratch_bytes(count))) return -2;
    return dedup_launch(x_dev, y_dev, conf_dev, tiebreak_dev, count, thr, inclusive, keep_dev, e->dedup_scratch.get(), e->dedup_scratch.bytes(),
                        (cudaStream_t)stream);
}

int b2d_seam_closure(b2d_engine* e, const double* x_dev, const double* y_dev, int count, double thr, int inclusive, uint8_t* flag_dev,
                     void* stream) {
    B2D_CHECK(e && (count == 0 || (x_dev && y_dev && flag_dev)), "seam_closure: bad arguments");
    B2D_ENTER(e);
    if (count == 0) return 0;
    if (e->dedup_scratch.reserve(dedup_scratch_bytes(count))) return -2;
    return closure_launch(x_dev, y_dev, count, thr, inclusive, flag_dev, e->dedup_scratch.get(), e->dedup_scratch.bytes(), (cudaStream_t)stream);
}

int b2d_utm_forward(b2d_engine* e, const double* lon_dev, const double* lat_dev, int count, int zone, int north, double* x_dev,
                    double* y_dev, void* stream) {
    B2D_CHECK(e && (count == 0 || (lon_dev && lat_dev && x_dev && y_dev)), "utm_forward: bad arguments");
    B2D_ENTER(e);
    B2D_CHECK(zone >= 1 && zone <= 60, "utm_forward: zone %d", zone);
    return utm_forward_launch(lon_dev, lat_dev, count, zone, north, x_dev, y_dev, (cudaStream_t)stream);
}

int b2d_cut_windows(b2d_engine* e, const uint8_t* mosaic_dev, int mh, int mw, long long pitch, const int32_t* origins_dev, int n,
                    int win, int fill, uint8_t* dst_dev, void* stream) {
    B2D_CHECK(e && mosaic_dev && origins_dev && dst_dev && n > 0, "cut_windows: bad arguments");
    B2D_ENTER(e);
    return cut_windows_launch(mosaic_dev, mh, mw, pitch, origins_dev, n, win, fill, dst_dev, (cudaStream_t)stream);
}

int b2d_resize_windows(b2d_engine* e, const uint8_t* mosaic_dev, int mh, int mw, long long pitch, const int32_t* origins_dev, int n,
                       int win, int fill, int bgr, int out_kind, void* dst_dev, void* stream) {
    B2D_CHECK(e && mosaic_dev && origins_dev && n > 0, "resize_windows: bad arguments");
    B2D_CHECK(win > 0, "resize_windows: window size %d must be positive", win);
    B2D_CHECK(mh > 0 && mw > 0 && pitch >= 3LL * mw, "resize_windows: mosaic %dx%d with pitch %lld", mh, mw, pitch);
    B2D_CHECK(fill >= 0 && fill <= 255, "resize_windows: fill %d outside 0..255", fill);
    B2D_ENTER(e);
    const int imgsz = e->bufs.empty() ? 640 : e->bufs[0].h;
    if (dst_dev == nullptr) {
        if (out_kind == B2D_OUT_BF16_NHWC4 && e->f16) out_kind = B2D_OUT_F16_NHWC4;   // the engine's own input format
        B2D_CHECK((out_kind == B2D_OUT_BF16_NHWC4 || out_kind == B2D_OUT_F16_NHWC4) && !e->bufs.empty() && e->bufs[0].c == 4 && !e->bufs[0].f32,
                  "resize_windows: dst NULL needs the planned 16-bit NHWC4 input buffer");
        B2D_CHECK(n <= e->max_batch, "resize_windows: n=%d exceeds max_batch %d", n, e->max_batch);
        dst_dev = e->bufs[0].ptr.get();
    }
    B2D_CHECK(out_kind == B2D_OUT_U8_NHWC || out_kind == B2D_OUT_BF16_NHWC4 || out_kind == B2D_OUT_F16_NHWC4,
              "resize_windows: out_kind %d is neither uint8 NHWC nor a 16-bit NHWC4 network input", out_kind);
    return resize_windows_launch(mosaic_dev, mh, mw, pitch, origins_dev, n, win, imgsz, fill, bgr, out_kind, dst_dev,
                                 (cudaStream_t)stream);
}

int b2d_set_conf_scale(b2d_engine* e, float scale) {
    B2D_CHECK(e && scale > 0.f, "set_conf_scale: bad arguments");
    e->conf_scale = scale;
    return 0;
}

static bool aligned4(const void* a, const void* b) { return (((uintptr_t)a | (uintptr_t)b) & 3) == 0; }

int b2d_colour_convert(b2d_engine* e, const uint8_t* src_dev, long long npix, int code, uint8_t* dst_dev, void* stream) {
    B2D_CHECK(e && src_dev && dst_dev && npix >= 0 && (code == B2D_COLOUR_RGB2LAB || code == B2D_COLOUR_LAB2RGB), "colour_convert: bad arguments");
    B2D_ENTER(e);
    B2D_CHECK(aligned4(src_dev, dst_dev), "colour_convert: pointers must be 4-byte aligned");
    return tta_colour_launch(src_dev, npix, code, dst_dev, (cudaStream_t)stream);
}

int b2d_tta_clahe(b2d_engine* e, const uint8_t* src_dev, int n, int h, int w, double clip_limit, int tiles_x, int tiles_y,
                  uint8_t* dst_dev, void* stream) {
    B2D_CHECK(e && src_dev && dst_dev && n > 0 && h > 0 && w > 0 && tiles_x > 0 && tiles_y > 0, "tta_clahe: bad arguments");
    B2D_ENTER(e);
    B2D_CHECK(aligned4(src_dev, dst_dev), "tta_clahe: pointers must be 4-byte aligned");
    if (e->tta_luts.reserve((size_t)n * tiles_x * tiles_y * 256)) return -2;
    return tta_clahe_launch(src_dev, n, h, w, clip_limit, tiles_x, tiles_y, e->tta_luts.get(), dst_dev, (cudaStream_t)stream);
}

int b2d_tta_lut(b2d_engine* e, const uint8_t* src_dev, int n, long long img_bytes, const uint8_t* lut_dev, int per_image,
                uint8_t* dst_dev, void* stream) {
    B2D_CHECK(e && src_dev && dst_dev && lut_dev && n > 0 && img_bytes > 0, "tta_lut: bad arguments");
    B2D_ENTER(e);
    return tta_lut_launch(src_dev, n, img_bytes, lut_dev, per_image, dst_dev, (cudaStream_t)stream);
}

int b2d_tta_contrast(b2d_engine* e, const uint8_t* src_dev, int n, int h, int w, float factor, uint8_t* dst_dev, void* stream) {
    B2D_CHECK(e && src_dev && dst_dev && n > 0 && h > 0 && w > 0, "tta_contrast: bad arguments");
    B2D_ENTER(e);
    B2D_CHECK(aligned4(src_dev, dst_dev), "tta_contrast: pointers must be 4-byte aligned");
    if (e->tta_luts.reserve((size_t)n * 256) || e->tta_sums.reserve((size_t)n * sizeof(unsigned long long))) return -2;
    return tta_contrast_launch(src_dev, n, h, w, factor, e->tta_sums.get(), e->tta_luts.get(), dst_dev, (cudaStream_t)stream);
}

int b2d_infer_tiles(b2d_engine* e, const uint8_t* src_dev, int n, int h, int w, int pitch, long long img_stride, int mode, int bgr,
                    float conf_thr, int inclusive, float iou_thr, int top_k, int max_det, b2d_det* dets_dev, int32_t* counts_dev, int cap,
                    void* stream) {
    B2D_CHECK(e != nullptr, "infer_tiles: null engine");
    B2D_CHECK(!is_obb(e), "infer_tiles: the engine has an oriented-box head; run b2d_preprocess, b2d_forward, b2d_postprocess_obb");
    B2D_ENTER(e);
    int rc = b2d_preprocess(e, src_dev, n, h, w, pitch, img_stride, mode, bgr, B2D_OUT_BF16_NHWC4, nullptr, stream);
    if (rc) return rc;
    if ((rc = b2d_forward(e, n, stream)) != 0) return rc;
    return b2d_postprocess(e, n, conf_thr, inclusive, iou_thr, top_k, max_det, dets_dev, counts_dev, cap, stream);
}

static int ensure_host_slot(b2d_engine* e, int slot, size_t tiles_bytes, int cap) {
    auto& hs = e->host_slot[slot];
    if ((!hs.loaded && create(hs.loaded)) || (!hs.drained && create(hs.drained)) || hs.tiles.reserve(tiles_bytes)) return -2;
    if (cap > hs.cap) {
        hs.cap = 0;             // every old record block goes before any new one is allocated; the device ones come first
        hs.params.reset(); hs.dets.reset(); hs.geo.reset(); hs.counts.reset();
        hs.params_pin.reset(); hs.geo_pin.reset(); hs.counts_pin.reset();
        const size_t nb = (size_t)e->max_batch;
        if (hs.params.reserve(nb * B2D_GEO_PARAMS * sizeof(double)) || hs.dets.reserve(nb * cap * sizeof(b2d_det)) ||
            hs.geo.reserve(nb * cap * sizeof(b2d_geodet)) || hs.counts.reserve(nb * sizeof(int32_t)) ||
            hs.params_pin.reserve(nb * B2D_GEO_PARAMS * sizeof(double)) || hs.geo_pin.reserve(nb * cap * sizeof(b2d_geodet)) ||
            hs.counts_pin.reserve(nb * sizeof(int32_t)))
            return -2;
        hs.cap = cap;
    }
    return 0;
}

int b2d_detect_host(b2d_engine* e, const uint8_t* tiles_host, int n, int h, int w, int mode, int bgr, float conf_thr, int inclusive,
                    float iou_thr, int top_k, int max_det, int geo_mode, const double* params_host, b2d_geodet* out_host,
                    int32_t* counts_host, int cap, void* stream) {
    B2D_CHECK(e && e->finalized && tiles_host && params_host && out_host && counts_host && n > 0 && h > 0 && w > 0 && cap > 0,
              "detect_host: bad arguments");
    B2D_CHECK(!is_obb(e), "detect_host: the engine has an oriented-box head; the host path returns axis-aligned records only");
    B2D_ENTER(e);
    cudaStream_t s = (cudaStream_t)stream;
    if (!e->copy_stream && create(e->copy_stream)) return -2;
    cudaStream_t cs = e->copy_stream.get();
    const size_t img_bytes = (size_t)h * w * 3;
    const int mb = e->max_batch;
    for (int slot = 0; slot < 2; ++slot)
        if (ensure_host_slot(e, slot, (size_t)(n < mb ? n : mb) * img_bytes, cap)) return -2;
    // The user's result arrays may be pageable (a device->host copy into pageable memory blocks the calling thread until the
    // stream has drained, which would serialise the chunks), so results land in the slot's pinned buffers and are moved to the
    // user's arrays one chunk behind, while the next chunk computes.
    int rc = 0, k = 0, prev_i0 = -1, prev_nb = 0;
    auto flush = [&](int slot, int i0, int nb) -> int {
        auto& hs = e->host_slot[slot];
        B2D_CUDA(cudaEventSynchronize(hs.drained.get()));
        memcpy(out_host + (size_t)i0 * cap, hs.geo_pin.get(), (size_t)nb * cap * sizeof(b2d_geodet));
        memcpy(counts_host + i0, hs.counts_pin.get(), (size_t)nb * sizeof(int32_t));
        return 0;
    };
    for (int i0 = 0; i0 < n && rc == 0; i0 += mb, ++k) {
        const int nb = n - i0 < mb ? n - i0 : mb;
        auto& hs = e->host_slot[k & 1];
        // copy stream: wait until the chunk that used this slot two iterations ago has been consumed, then load
        if (k >= 2) B2D_CUDA(cudaStreamWaitEvent(cs, hs.drained.get(), 0));
        memcpy(hs.params_pin.get(), params_host + (size_t)i0 * B2D_GEO_PARAMS, (size_t)nb * B2D_GEO_PARAMS * sizeof(double));
        B2D_CUDA(cudaMemcpyAsync(hs.tiles.get(), tiles_host + (size_t)i0 * img_bytes, (size_t)nb * img_bytes, cudaMemcpyHostToDevice, cs));
        B2D_CUDA(cudaMemcpyAsync(hs.params.get(), hs.params_pin.get(), (size_t)nb * B2D_GEO_PARAMS * sizeof(double), cudaMemcpyHostToDevice, cs));
        B2D_CUDA(cudaEventRecord(hs.loaded.get(), cs));
        B2D_CUDA(cudaStreamWaitEvent(s, hs.loaded.get(), 0));
        rc = b2d_infer_tiles(e, hs.tiles.get(), nb, h, w, w * 3, (long long)img_bytes, mode, bgr, conf_thr, inclusive, iou_thr, top_k, max_det,
                             hs.dets.get(), hs.counts.get(), cap, s);
        if (rc == 0) rc = b2d_georef(e, hs.dets.get(), hs.counts.get(), nb, cap, geo_mode, hs.params.get(), hs.geo.get(), s);
        if (rc) break;
        B2D_CUDA(cudaMemcpyAsync(hs.geo_pin.get(), hs.geo.get(), (size_t)nb * cap * sizeof(b2d_geodet), cudaMemcpyDeviceToHost, s));
        B2D_CUDA(cudaMemcpyAsync(hs.counts_pin.get(), hs.counts.get(), (size_t)nb * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        B2D_CUDA(cudaEventRecord(hs.drained.get(), s));
        if (prev_i0 >= 0 && flush((k & 1) ^ 1, prev_i0, prev_nb)) return -2;
        prev_i0 = i0; prev_nb = nb;
    }
    if (rc == 0 && prev_i0 >= 0 && flush((k - 1) & 1, prev_i0, prev_nb)) return -2;
    cudaError_t err = cudaStreamSynchronize(s);
    cudaStreamSynchronize(cs);
    if (rc) return rc;
    B2D_CUDA(err);
    return 0;
}

}  // extern "C"
