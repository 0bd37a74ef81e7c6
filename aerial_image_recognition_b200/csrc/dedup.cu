// K5' -- greedy centre-distance dedup in a metric CRS, and the WGS84 -> UTM forward projection
// that feeds it.
//
// Reference: SimpleDetector._remove_duplicates (simple_detector.py:540-596): sort by confidence
// (stable, descending), keep a detection iff no already-kept one lies within `thr` metres
// (`dx*dx + dy*dy <= thr*thr`, float64, :585-587); variant ResultsManager.remove_duplicates
// (_script/utils.py:229-256) with a strict `<`.
//
// The sequential greedy pass is restated as a fixed point that gives the *same* keep set:
//   a point is REMOVED as soon as one higher-priority neighbour is KEPT,
//   a point is KEPT   as soon as every higher-priority neighbour is REMOVED.
// Priority is the reference's total order (confidence descending, input index ascending), so
// the result does not depend on thread scheduling.  Neighbours come from a hashed uniform grid
// with cell size `thr` (3x3 cells), built with one atomicExch per point -- no sort.
#include "common.cuh"

#include <math.h>

namespace {

struct DedupTable {
    long long* cell_key;   // [cap] cell id ((cx + 2^31) << 32) | (cy + 2^31), -1 = empty (not a key: cells are range-checked to |c| < 2^31 - 2)
    int* cell_head;        // [cap] head of the linked list of points in the cell
    int* next;             // [n]
    uint8_t* state;        // [n] 0 undecided, 1 kept, 2 removed
    int* flag;             // [0] number of points still undecided after a round, [1] != 0: a point's cell index is out of range
    unsigned cap_mask;
};

// The cell packing, hash and table probes are common.cuh's (pack_cell, cell_claim, cell_first).
__device__ __forceinline__ bool cell_in_range(long long cx, long long cy) {
    return cx > -kCellMax && cx < kCellMax && cy > -kCellMax && cy < kCellMax;
}

__global__ void dedup_init_kernel(DedupTable t, int n, unsigned cap) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cap) { t.cell_key[i] = -1; t.cell_head[i] = -1; }
    if (i < (unsigned)n) { t.state[i] = 0; t.next[i] = -1; }
    if (i == 0) { t.flag[0] = 0; t.flag[1] = 0; }
}

__global__ void dedup_build_kernel(DedupTable t, const double* __restrict__ x, const double* __restrict__ y, int n, double inv_cell) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double fx = floor(x[i] * inv_cell), fy = floor(y[i] * inv_cell);
    if (!(fabs(fx) < (double)kCellMax && fabs(fy) < (double)kCellMax)) {      // also catches NaN / inf coordinates
        t.flag[1] = 1;
        return;                                                               // the host reports the error; the point stays unlinked
    }
    const unsigned slot = cell_claim(t.cell_key, t.cap_mask, pack_cell((long long)fx, (long long)fy));
    t.next[i] = atomicExch(&t.cell_head[slot], i);
}

__global__ void dedup_round_kernel(DedupTable t, const double* __restrict__ x, const double* __restrict__ y,
                                   const float* __restrict__ conf, const long long* __restrict__ tiebreak, int n, double inv_cell,
                                   double thr2, int inclusive) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (((volatile uint8_t*)t.state)[i] != 0) return;
    const double xi = x[i], yi = y[i];
    const float ci = conf[i];
    const long long ki = tiebreak ? tiebreak[i] : (long long)i;
    const long long cx = (long long)floor(xi * inv_cell), cy = (long long)floor(yi * inv_cell);
    bool removed = false, wait = false;
    for (int dx = -1; dx <= 1 && !removed; ++dx)
        for (int dy = -1; dy <= 1 && !removed; ++dy) {
            const int head = cell_first(t.cell_key, t.cell_head, t.cap_mask, pack_cell(cx + dx, cy + dy));
            for (int j = head; j >= 0; j = t.next[j]) {
                if (j == i) continue;
                const float cj = conf[j];
                const long long kj = tiebreak ? tiebreak[j] : (long long)j;
                if (!(cj > ci || (cj == ci && kj < ki))) continue;     // only higher-priority points matter
                const double ddx = __dsub_rn(xi, x[j]), ddy = __dsub_rn(yi, y[j]);
                const double d2 = __dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy));
                if (!(inclusive ? (d2 <= thr2) : (d2 < thr2))) continue;
                const uint8_t sj = ((volatile uint8_t*)t.state)[j];
                if (sj == 1) { removed = true; break; }
                if (sj == 0) wait = true;
            }
        }
    if (removed) t.state[i] = 2;
    else if (!wait) t.state[i] = 1;
    else atomicAdd(t.flag, 1);
}

__global__ void dedup_finish_kernel(DedupTable t, int n, uint8_t* keep) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keep[i] = (t.state[i] == 1) ? 1 : 0;
}

// WGS84 -> UTM, Krueger series to n^4 (same formulation as oracle/postproc.py::utm_forward)
__global__ void utm_forward_kernel(const double* __restrict__ lon, const double* __restrict__ lat, int n, double lon0, int north,
                                   double* __restrict__ xo, double* __restrict__ yo) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double a = 6378137.0, f = 1.0 / 298.257223563;
    const double nn = f / (2.0 - f);
    const double A = a / (1.0 + nn) * (1.0 + nn * nn / 4.0 + nn * nn * nn * nn / 64.0);
    const double n2 = nn * nn, n3 = n2 * nn, n4 = n3 * nn;
    const double al[4] = {nn / 2 - 2 * n2 / 3 + 5 * n3 / 16 + 41 * n4 / 180, 13 * n2 / 48 - 3 * n3 / 5 + 557 * n4 / 1440,
                          61 * n3 / 240 - 103 * n4 / 140, 49561 * n4 / 161280};
    const double d2r = 0.017453292519943295;
    const double phi = lat[i] * d2r, lam = lon[i] * d2r - lon0;
    const double e = sqrt(f * (2.0 - f));
    const double s = sin(phi);
    const double tt = sinh(atanh(s) - e * atanh(e * s));
    const double xi = atan2(tt, cos(lam));
    const double eta = atanh(sin(lam) / sqrt(1.0 + tt * tt));
    double X = eta, Y = xi;
    for (int j = 1; j <= 4; ++j) {
        X += al[j - 1] * cos(2 * j * xi) * sinh(2 * j * eta);
        Y += al[j - 1] * sin(2 * j * xi) * cosh(2 * j * eta);
    }
    xo[i] = 500000.0 + 0.9996 * A * X;
    yo[i] = 0.9996 * A * Y + (north ? 0.0 : 10000000.0);
}

unsigned table_cap(int n) {
    unsigned cap = 1024;
    while (cap < (unsigned)(2 * n)) cap <<= 1;
    return cap;
}

}  // namespace

size_t dedup_scratch_bytes(int count) {
    const unsigned cap = table_cap(count);
    // cell keys + cell heads + next links + flags (16 B) + state bytes, then the closure's labels and component marks
    return (size_t)cap * 8 + (size_t)cap * 4 + (size_t)count * 4 + 16 + (size_t)((count + 15) & ~15) + (size_t)count * 4 + (size_t)((count + 15) & ~15) + 64;
}

// Seam closure: flag[i] != 0 marks detections that may interact with another shard; the closure extends the flag to every
// detection connected to a flagged one through the "within thr" relation, so that every connected component of the
// suppression graph is either entirely flagged or entirely local.
//
// Connected components by label propagation with pointer jumping: label[i] starts as i; a hook round gives every point
// (and its current representative) the smallest label among its neighbours, a jump round replaces every label by its
// root.  Labels only ever point to a smaller index in the same component, and the rounds stop when no edge joins two
// different roots -- a number of rounds logarithmic in the longest chain, where flooding the flag one hop per round took
// one round per metre of chain (detections line up along image edges for kilometres; 8 800 rounds on config C4).
__global__ void closure_init_kernel(int* __restrict__ label, uint8_t* __restrict__ comp, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { label[i] = i; comp[i] = 0; }
}

__global__ void closure_hook_kernel(DedupTable t, const double* __restrict__ x, const double* __restrict__ y, int n, double inv_cell,
                                    double thr2, int inclusive, int* label) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double xi = x[i], yi = y[i];
    const long long cx = (long long)floor(xi * inv_cell), cy = (long long)floor(yi * inv_cell);
    const int li = ((volatile int*)label)[i];
    int m = li;
    for (int dx = -1; dx <= 1; ++dx)
        for (int dy = -1; dy <= 1; ++dy) {
            const int head = cell_first(t.cell_key, t.cell_head, t.cap_mask, pack_cell(cx + dx, cy + dy));
            for (int j = head; j >= 0; j = t.next[j]) {
                if (j == i) continue;
                const double ddx = __dsub_rn(xi, x[j]), ddy = __dsub_rn(yi, y[j]);
                const double d2 = __dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy));
                if (inclusive ? (d2 <= thr2) : (d2 < thr2)) {
                    const int lj = ((volatile int*)label)[j];
                    if (lj < m) m = lj;
                }
            }
        }
    if (m < li) {
        atomicMin(&label[i], m);
        atomicMin(&label[li], m);          // the old representative joins too: whole trees merge, not single points
        t.flag[0] = 1;
    }
}

__global__ void closure_jump_kernel(int* label, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int l = ((volatile int*)label)[i];
    while (true) {
        const int ll = ((volatile int*)label)[l];
        if (ll >= l) break;
        l = ll;
    }
    label[i] = l;
}

__global__ void closure_mark_kernel(const int* __restrict__ label, const uint8_t* __restrict__ flag, uint8_t* comp, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && flag[i]) comp[label[i]] = 1;
}

__global__ void closure_apply_kernel(const int* __restrict__ label, const uint8_t* __restrict__ comp, uint8_t* flag, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = comp[label[i]];
}

static int build_table(DedupTable& t, const double* x, const double* y, int count, double thr, void* scratch, size_t scratch_bytes,
                       cudaStream_t stream, double* inv_cell_out) {
    B2D_CHECK(scratch_bytes >= dedup_scratch_bytes(count), "dedup: scratch too small");
    const unsigned cap = table_cap(count);
    uint8_t* p = (uint8_t*)scratch;
    t.cell_key = (long long*)p; p += (size_t)cap * 8;
    t.cell_head = (int*)p; p += (size_t)cap * 4;
    t.next = (int*)p; p += (size_t)count * 4;
    t.flag = (int*)p; p += 16;
    t.state = p;
    t.cap_mask = cap - 1;
    const double cell = thr > 0.0 ? thr : 1.0;
    *inv_cell_out = 1.0 / cell;
    const int threads = 256;
    const unsigned m = cap > (unsigned)count ? cap : (unsigned)count;
    dedup_init_kernel<<<(m + threads - 1) / threads, threads, 0, stream>>>(t, count, cap);
    dedup_build_kernel<<<(count + threads - 1) / threads, threads, 0, stream>>>(t, x, y, count, *inv_cell_out);
    B2D_LAUNCH_CHECK();
    return 0;
}

int closure_launch(const double* x, const double* y, int count, double thr, int inclusive, uint8_t* flag, void* scratch,
                   size_t scratch_bytes, cudaStream_t stream) {
    if (count <= 0) return 0;
    DedupTable t;
    double inv_cell;
    if (build_table(t, x, y, count, thr, scratch, scratch_bytes, stream, &inv_cell)) return -1;
    int* label = (int*)(t.state + (((size_t)count + 15) & ~(size_t)15));
    uint8_t* comp = (uint8_t*)(label + count);
    const int blocks = (count + 255) / 256;
    closure_init_kernel<<<blocks, 256, 0, stream>>>(label, comp, count);
    int h_flag[2] = {1, 0};
    int closure_rounds = 0;
    for (int round = 0; h_flag[0] != 0; ++round, ++closure_rounds) {
        B2D_CUDA(cudaMemsetAsync(t.flag, 0, sizeof(int), stream));
        closure_hook_kernel<<<blocks, 256, 0, stream>>>(t, x, y, count, inv_cell, thr * thr, inclusive, label);
        closure_jump_kernel<<<blocks, 256, 0, stream>>>(label, count);
        B2D_LAUNCH_CHECK();
        B2D_CUDA(cudaMemcpyAsync(h_flag, t.flag, 2 * sizeof(int), cudaMemcpyDeviceToHost, stream));
        B2D_CUDA(cudaStreamSynchronize(stream));
        B2D_CHECK(h_flag[1] == 0, "closure: a coordinate / thr is outside the grid's +-2^31 cells (or not finite)");
        B2D_CHECK(round <= count + 8, "closure: did not converge");
    }
    if (getenv("B2D_VERBOSE")) fprintf(stderr, "b2det: seam closure of %d points: %d rounds\n", count, closure_rounds);
    closure_mark_kernel<<<blocks, 256, 0, stream>>>(label, flag, comp, count);
    closure_apply_kernel<<<blocks, 256, 0, stream>>>(label, comp, flag, count);
    B2D_LAUNCH_CHECK();
    return 0;
}

int dedup_launch(const double* x, const double* y, const float* conf, const long long* tiebreak, int count, double thr,
                 int inclusive, uint8_t* keep, void* scratch, size_t scratch_bytes, cudaStream_t stream) {
    if (count <= 0) return 0;
    DedupTable t;
    double inv_cell;
    if (build_table(t, x, y, count, thr, scratch, scratch_bytes, stream, &inv_cell)) return -1;
    const double thr2 = thr * thr;
    const int threads = 256;
    // Rounds: every round decides at least the highest-priority undecided point, so the loop ends;
    // real data needs a handful of rounds.  The host reads the undecided count back every 4 rounds.
    int h_flag[2] = {1, 0};
    int rounds_run = 0;
    for (int round = 0; h_flag[0] != 0; ++round, ++rounds_run) {
        B2D_CUDA(cudaMemsetAsync(t.flag, 0, sizeof(int), stream));
        dedup_round_kernel<<<(count + threads - 1) / threads, threads, 0, stream>>>(t, x, y, conf, tiebreak, count, inv_cell, thr2, inclusive);
        B2D_LAUNCH_CHECK();
        if ((round & 3) == 3 || count < 4096) {
            B2D_CUDA(cudaMemcpyAsync(h_flag, t.flag, 2 * sizeof(int), cudaMemcpyDeviceToHost, stream));
            B2D_CUDA(cudaStreamSynchronize(stream));
            B2D_CHECK(h_flag[1] == 0, "dedup: a coordinate / thr is outside the grid's +-2^31 cells (or not finite)");
        }
        B2D_CHECK(round <= count + 8, "dedup: did not converge");
    }
    dedup_finish_kernel<<<(count + threads - 1) / threads, threads, 0, stream>>>(t, count, keep);
    B2D_LAUNCH_CHECK();
    if (getenv("B2D_VERBOSE")) fprintf(stderr, "b2det: dedup of %d points: %d rounds\n", count, rounds_run);
    return 0;
}

int utm_forward_launch(const double* lon, const double* lat, int count, int zone, int north, double* x, double* y,
                       cudaStream_t stream) {
    if (count <= 0) return 0;
    const double lon0 = ((zone - 1) * 6 - 180 + 3) * 0.017453292519943295;
    utm_forward_kernel<<<(count + 255) / 256, 256, 0, stream>>>(lon, lat, count, lon0, north, x, y);
    B2D_LAUNCH_CHECK();
    return 0;
}
