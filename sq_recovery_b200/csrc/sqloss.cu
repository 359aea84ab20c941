// libsqloss: CUDA kernels (sm_100a) and the C ABI declared in include/sqloss.h.
//
// Kernel plan (DESIGN.md section 3): every grid loss is  plan -> column kernel -> finalize, on the caller's stream.
//   plan      one block per sample: clamp, rotation, scaled rows, exponents, culling constants in fp64 -> SampleFull
//             (scratch); the sum of |target| over the sample's pixels (ImplicitLoss); an upper bound on the cost of every
//             work item (32 grid columns) -> item appended to the queue of its cost class; items proven empty are
//             dropped for good
//   column    persistent warps take items most expensive class first; one thread per grid column (x, y) walking the
//             part of z that can hold occupancy (the rest is accounted for in closed form); grid points are generated
//             from indices, nothing per-point touches HBM; warps are autonomous: private Sample copy and sum tile in
//             shared memory, one partial row per item, no block barrier
//   finalize  one block per sample: fixed-order fp64 sum of the partial rows, Jacobians to the 12 parameters,
//             per-sample loss; the last block to finish averages the batch (fixed order, so results are
//             bit-reproducible run to run)
// The point-list loss (LeastSquares) is  prep -> lsq_kernel -> finalize.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <new>

#include "../../include/sqloss.h"
#ifdef SQ_TIMELINE      // tools/timeline.py: [0] backward blocks executed (warp level), [1] lanes that carried gradient in them
__device__ unsigned long long g_bwd_stats[2];
#endif
#if defined(SQ_TIMELINE) && defined(SQ_BWD_STATS)      // the two atomics per block slow the kernel 3x: only when asked for
#define SQ_BWD_HOOK(a) do { const unsigned m_ = __ballot_sync(0xffffffffu, (a)); if ((threadIdx.x & 31) == 0) { \
    atomicAdd(&g_bwd_stats[0], 1ull); atomicAdd(&g_bwd_stats[1], (unsigned long long)__popc(m_)); } } while (0)
#endif
#ifdef SQ_ITEMLOG      // tools/item_costs.py: per work item, what the plan kernel estimated and what the column kernel spent
__device__ float g_planlog[4 * 65536];       // cost class, estimated planes, -, -
__device__ int g_itemlog[4 * 65536];         // cycles of the item, cycles of its z walk, queued points, refined points
#endif
#ifdef SQ_COUNT         // counting build (libsqloss_count.so, bench.py): what the implicit column kernel did, per launch
// [0] warp plane steps of the z walk (32 point evaluations each)   [1] on-the-spot backward blocks (queue full)
// [2] deal-out rounds of the compacted backward (all entries)       [3] deal-out rounds of the fp64 refinement
// [4] work items processed   [5] column groups with occupancy   [6] queued gradient points   [7] of them refined in fp64
__device__ unsigned long long g_count[8];
#define SQ_COUNT_HOOK(i, n) do { if ((threadIdx.x & 31) == 0) atomicAdd(&g_count[i], (unsigned long long)(n)); } while (0)
#else
#define SQ_COUNT_HOOK(i, n) do { } while (0)
#endif
#include "sq_core.cuh"

using namespace sq;

namespace {

// Tunables (tools/tune.py builds variants with -D to measure them on the GPU; the defaults are the measured best,
// profiles/tune_r01.txt).  Per column kernel: block size, min resident blocks per SM (register cap), columns per
// thread and warp work item.
#ifndef SQ_IMPB_THREADS
#define SQ_IMPB_THREADS 128              // implicit fwd+bwd
#endif
#ifndef SQ_IMPB_MINB
// 5 blocks = 20 warps per SM at 96 registers (60 bytes of spill on cold paths): the phases of an item outside the z walk
// are dependent chains (profiles/phases_r02.txt), and a fifth warp per scheduler hides more of them than the 26 registers
// were worth -- 48.0 vs 49.2-50.1 us per call (profiles/tune_r02.txt run l).  It takes the three settings below with it:
// the reduction tile aliased onto the queue arrays and a 15-deep queue (shared memory for 5 blocks), one deal-out chain
// in flight instead of two (registers).  The round's earlier shape: -DSQ_IMPB_MINB=4 -DSQ_BWD_DEPTH=16 -DSQ_TILE_ALIAS=0
// -DSQ_DENSE_ILP=2.
#define SQ_IMPB_MINB 5
#endif
#ifndef SQ_TILE_ALIAS
#define SQ_TILE_ALIAS 1
#endif
#ifndef SQ_WALK_ESTIMATE     // cost classes of the implicit kernels from the planes a walk really visits (sq_core.cuh footprint_walk)
#define SQ_WALK_ESTIMATE 1
#endif
#ifndef SQ_DENSE_ILP
#define SQ_DENSE_ILP 1
#endif
#ifndef SQ_IMPB_CPT
#define SQ_IMPB_CPT 1
#endif
#ifndef SQ_IMPF_THREADS
#define SQ_IMPF_THREADS 256              // implicit fwd only (validation, depth rendering)
#endif
#ifndef SQ_IMPF_MINB
#define SQ_IMPF_MINB 4
#endif
#ifndef SQ_IMPF_CPT
#define SQ_IMPF_CPT 1
#endif
#ifndef SQ_EXP_THREADS
#define SQ_EXP_THREADS 256               // explicit fwd and fwd+bwd
#endif
#ifndef SQ_EXP_MINB
#define SQ_EXP_MINB 2
#endif
#ifndef SQ_EXP_CPT
#define SQ_EXP_CPT 1
#endif
#ifndef SQ_IOU_THREADS
#define SQ_IOU_THREADS 128
#endif
#ifndef SQ_IOU_MINB
#define SQ_IOU_MINB 4
#endif
#ifndef SQ_IOU_CPT
#define SQ_IOU_CPT 1
#endif
constexpr int kThreads = 256;            // block size of the small kernels (point list, field)
constexpr int kWarps = kThreads / 32;

// ------------------------------------------------------------------------------------------------ layout
// Column slots of one sample.  When n is a multiple of 8 a warp owns an 8(x) x 4(y) patch, which keeps the lanes of
// a warp at similar depth along z (the culled z range and the backward are entered per warp); otherwise slots are
// the n*n columns in x-fastest order.  Slots beyond n*n (last warp only) are masked.
// Work is handed out per WARP: warp item w of a sample covers slots [w*32*cpt, (w+1)*32*cpt).  Warps never
// synchronise with each other (no __syncthreads in the column kernels), each writes its own partial row.
struct Layout {
    int n, patched, slots, cpt, rows_per_sample;
    int rows_shift;      // log2(rows_per_sample) when it is a power of two, else -1
    int pw_shift;        // patched layout: log2(patches per row) when n / 8 is a power of two, else -1
    int jq, jr;          // patched layout: rows_per_sample / (n / 8) and the remainder (per-step patch advance of ColIter)
    __host__ __device__ __forceinline__ void split(int item, int& b, int& chunk) const {
        if (rows_shift >= 0) { b = item >> rows_shift; chunk = item & (rows_per_sample - 1); }
        else { b = item / rows_per_sample; chunk = item - b * rows_per_sample; }
    }
    __host__ __device__ __forceinline__ int sample_of(int item) const {
        return rows_shift >= 0 ? item >> rows_shift : item / rows_per_sample;
    }
};

__host__ __device__ inline Layout make_layout(int n, int max_cpt) {
    Layout L;
    L.n = n;
    L.patched = (n % 8 == 0);
    L.slots = n * n;
    L.cpt = (L.slots + 31) / 32;
    if (L.cpt > max_cpt) L.cpt = max_cpt;
    const int per_item = L.cpt * 32;
    L.rows_per_sample = (L.slots + per_item - 1) / per_item;
    L.rows_shift = -1;
    for (int sh = 0; sh < 30; ++sh) if ((1 << sh) == L.rows_per_sample) L.rows_shift = sh;
    L.pw_shift = -1; L.jq = L.jr = 0;
    if (L.patched) {
        const int pw = n >> 3;
        for (int sh = 0; sh < 30; ++sh) if ((1 << sh) == pw) L.pw_shift = sh;
        L.jq = L.rows_per_sample / pw;
        L.jr = L.rows_per_sample - L.jq * pw;
    }
    return L;
}

// Column (x, y) of lane `lane` for the k-th 32-slot group of a warp item.  Item j of a sample owns groups
// j, j + J, j + 2J, ... (J = rows_per_sample): its columns are spread over the whole image, so the items of one
// sample cost about the same (objects sit near the image centre; a contiguous tile would be all-empty or all-full).
struct ColIter {
    int ia, ib, slot;
    int pa, pb, jq, jr;       // patched layout: patch coordinates and the per-step patch advance (J / pw, J % pw)
    __device__ __forceinline__ void init(const Layout& L, int first_group, int lane) {
        slot = first_group * 32 + lane;
        if (L.patched) {
            const int pw = L.n >> 3;
            pb = L.pw_shift >= 0 ? first_group >> L.pw_shift : first_group / pw;      // once per work item
            pa = first_group - pb * pw;
            jq = L.jq;
            jr = L.jr;
            ia = (pa << 3) + (lane & 7);
            ib = (pb << 2) + (lane >> 3);
        } else {
            ib = slot / L.n;
            ia = slot - ib * L.n;
            pa = pb = jq = jr = 0;
        }
    }
    __device__ __forceinline__ void next(const Layout& L) {
        slot += 32 * L.rows_per_sample;
        if (L.patched) {
            pa += jr; pb += jq;
            if (pa >= (L.n >> 3)) { pa -= (L.n >> 3); ++pb; }
            ia = (pa << 3) + (slot & 7);
            ib = (pb << 2) + ((slot & 31) >> 3);
        } else {
            ib = slot / L.n;
            ia = slot - ib * L.n;
        }
    }
    __device__ __forceinline__ bool valid(const Layout& L) const { return slot < L.slots; }
};

// ------------------------------------------------------------------------------------------------ scratch
// Work items are handed to the persistent warps in order of estimated cost (longest first, empty last): the plan
// kernel sorts them into kClasses cost classes, one queue per class.  Class k holds items whose estimated number of
// z planes is in (max / 2^((k+1)/4), max / 2^(k/4)] (four classes per octave); the last class holds items PROVEN empty (the
// plane count is an upper bound), which the column kernels never touch.  For the implicit kernels the estimate is the
// planes a walk really visits (sq_core.cuh footprint_walk): the early exit cuts interior groups short.
#ifndef SQ_CLASSES
#define SQ_CLASSES 32
#endif
constexpr int kClasses = SQ_CLASSES;     // 8: one class per octave of cost; 16 / 32: two / four per octave -- a finer
                                         // longest-first order: the last big items handed out are the cheaper ones (-1.5 us)
static_assert(kClasses >= 4 && kClasses <= 32, "the class counters live in one warp's lanes and in the 256-byte control block");
#ifndef SQ_PLAN_THREADS
#define SQ_PLAN_THREADS 512
#endif
constexpr int kPlanThreads = SQ_PLAN_THREADS;
constexpr int kPlanThreadsSmall = 128;   // batches beyond one wave of kPlanThreads blocks (4 per SM)
constexpr int kPlanMaxItems = 8192;      // items per sample the plan kernel can classify (more: index order)

// First 256 bytes of every scratch buffer.  qcount and retired must be ZERO when a call starts: sq_scratch_init()
// zeroes them once and every kernel that uses them leaves them zero again (the last warp to retire cleans up), so no
// memset sits on the per-call critical path.  ticket and cursor are reset by the plan / prep kernel of each call.
struct Control {
    unsigned int ticket;                 // samples finalized so far (the last one averages the batch)
    unsigned int cursor;                 // work-stealing cursor of the column kernel
    unsigned int retired;                // warps that have left the column kernel
    unsigned int pad0;
    unsigned int qcount[kClasses];       // items per cost class
    unsigned int pad1[64 - 4 - kClasses];
};
static_assert(sizeof(Control) == 256, "Control block is 256 bytes");

constexpr int kRow = 20;                 // floats per partial row: the kAccN sums, then the loss-centring pair (see implicit_kernel)
struct Scratch {
    Control* ctl;
    SampleFull* pred;      // [batch]
    SampleFull* tru;       // [batch]
    float* partials;       // [batch * rows_per_sample][kRow]
    double* per_sample;    // [batch]
    double* tv_sum;        // [batch] sum |target| over the sample's pixels (ImplicitLoss)
    unsigned long long* counts;   // [batch][2] (IoU)
    unsigned char* item_class;   // [batch * rows_per_sample] cost class of every item (kClasses - 1: proven empty, no row)
    int* queue;            // [kClasses][queue_cap] item ids by cost class; nullptr: items are taken in index order
    int queue_cap;
};

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

size_t scratch_layout(int batch, int n, char* base, Scratch* s) {
    const Layout L = make_layout(n > 0 ? n : 1, 1);      // cpt = 1: the most rows any kernel configuration writes
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_ctl = take(sizeof(Control));          // always at offset 0
    const size_t o_pred = take(sizeof(SampleFull) * (size_t)batch);
    const size_t o_true = take(sizeof(SampleFull) * (size_t)batch);
    // partial rows: one per warp item for the column kernels, one per 256 pixels for the point-list kernel
    size_t rows_ps = (size_t)L.rows_per_sample;
    const size_t lsq_rows = (size_t)(L.slots + kThreads - 1) / kThreads;
    if (lsq_rows > rows_ps) rows_ps = lsq_rows;
    const size_t o_part = take(sizeof(float) * kRow * rows_ps * (size_t)batch);
    const size_t o_ps = take(sizeof(double) * (size_t)batch);
    const size_t o_tv = take(sizeof(double) * (size_t)batch);
    const size_t o_cnt = take(sizeof(unsigned long long) * 2 * (size_t)batch);
    const size_t cap = (size_t)L.rows_per_sample * (size_t)batch;
    const bool queued = L.rows_per_sample <= kPlanMaxItems && cap < (1u << 30);
    const size_t o_queue = take(queued ? sizeof(int) * kClasses * cap : 0);
    const size_t o_cls = take(queued ? cap : 0);
    if (s) {
        s->ctl = reinterpret_cast<Control*>(base + o_ctl);
        s->pred = reinterpret_cast<SampleFull*>(base + o_pred);
        s->tru = reinterpret_cast<SampleFull*>(base + o_true);
        s->partials = reinterpret_cast<float*>(base + o_part);
        s->per_sample = reinterpret_cast<double*>(base + o_ps);
        s->tv_sum = reinterpret_cast<double*>(base + o_tv);
        s->counts = reinterpret_cast<unsigned long long*>(base + o_cnt);
        s->queue = queued ? reinterpret_cast<int*>(base + o_queue) : nullptr;
        s->item_class = queued ? reinterpret_cast<unsigned char*>(base + o_cls) : nullptr;
        s->queue_cap = (int)cap;
    }
    return off;
}

// ------------------------------------------------------------------------------------------------ PDL
// Programmatic dependent launch (-DSQ_PDL): the column kernel and the finalize kernel are launched with the
// programmatic-stream-serialization attribute, so their blocks can become resident while the preceding kernel of the call
// drains; pdl_wait() returns once that kernel has completed and its writes are visible.
__device__ __forceinline__ void pdl_wait() {
#ifdef SQ_PDL
    asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
}
__device__ __forceinline__ void pdl_trigger() {
#ifdef SQ_PDL
    asm volatile("griddepcontrol.launch_dependents;");
#endif
}

// ------------------------------------------------------------------------------------------------ prep / plan
#ifdef SQ_TIMELINE     // tools/timeline.py
__device__ unsigned long long g_plan_ts[16];
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#endif
constexpr int kSampleWords = (int)(sizeof(Sample) / 4);          // the part the column kernels keep per warp
constexpr int kFullWords = (int)(sizeof(SampleFull) / 4);        // the record in HBM
static_assert(sizeof(Sample) % 8 == 0 && sizeof(SampleFull) % 8 == 0, "Sample records must be word-copyable");

__device__ __forceinline__ void load_params(const void* params, int dtype, int b, double* p) {
#pragma unroll
    for (int i = 0; i < 12; ++i)
        p[i] = dtype == SQ_F64 ? static_cast<const double*>(params)[12 * (size_t)b + i]
                               : (double)static_cast<const float*>(params)[12 * (size_t)b + i];
}

// prep (point-list and field kernels): one warp per sample; lane 0 does the fp64 work into shared memory, the warp
// copies the 328-byte record out with coalesced stores.
__global__ void __launch_bounds__(128)
prep_kernel(const void* params, int dtype, int batch, int clamp, Grid g, SampleFull* out, Control* ctl) {
    __shared__ SampleFull Ssh[4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * 4 + warp;
    if (blockIdx.x == 0 && threadIdx.x == 0 && ctl) { ctl->ticket = 0u; ctl->cursor = 0u; }
    if (b >= batch) return;
    if (lane == 0) {
        double p[12];
        load_params(params, dtype, b, p);
        prep_sample(p, clamp != 0, g, Ssh[warp]);
    }
    __syncwarp();
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&Ssh[warp]);
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + b);
    for (int w = lane; w < kFullWords; w += 32) dst[w] = src[w];
}

// Upper estimate of the z planes a 32-column group of one sample walks: the culling bounds of column_range() evaluated
// once at the centre of the group's footprint, widened by how far s can move across the footprint (so a thin object
// that slips between probe columns is never taken for empty).  Only the ORDER in which work is handed out depends on
// this, never a result.
__device__ int group_planes(const Sample& S, const Grid& g, const Layout& L, float bound, int group, float die = 0.f) {
    float cx, cy, hx, hy;                                  // centre and half extent of the footprint, in grid steps
    if (L.patched) {
        const int pw = L.n >> 3, pb = group / pw, pa = group - pb * pw;
        cx = (float)(pa << 3) + 3.5f; cy = (float)(pb << 2) + 1.5f; hx = 3.5f; hy = 1.5f;
    } else {
        xfast_group_footprint(L.n, group, cx, cy, hx, hy);
    }
    return die > 0.f ? footprint_walk(S, g, bound, die, cx, cy, hx, hy) : footprint_planes(S, g, bound, cx, cy, hx, hy);
}

// plan (column kernels): one block per sample.  Builds the Sample record(s) like prep, then estimates the cost of each
// of the sample's work items and appends the item to the queue of its cost class.  NS = SQs per item (2: true + pred).
// THREADS: kPlanThreads while the batch fits one wave of such blocks (shortest latency per sample: many threads per
// pixel sum); kPlanThreadsSmall beyond (more samples resident per SM: the kernel is then a throughput problem).
template <int NS, int THREADS>
__global__ void __launch_bounds__(THREADS)
plan_kernel(const void* params_a, const void* params_b, int dtype, int clamp, int heads, Grid g, Layout L, float bound, float die,
            SampleFull* out_a, SampleFull* out_b, Control* ctl, unsigned long long* counts, int* queue, int cap,
            unsigned char* item_class, const float* __restrict__ target, long long tstride, const int* __restrict__ row_off,
            const int* __restrict__ col_off, double* tv_sum) {
    __shared__ SampleFull Ssh[NS];
    __shared__ unsigned char cls[kPlanMaxItems];
    __shared__ unsigned int ccnt[kClasses], cbase[kClasses];
    __shared__ double tv_part[THREADS / 32];
    const int b = blockIdx.x;
#ifdef SQ_TIMELINE
    unsigned long long ts[6]; int nts = 0;
#define SQ_STAMP() do { if (nts < 6) ts[nts++] = gtime(); } while (0)
#else
#define SQ_STAMP() do { } while (0)
#endif
    SQ_STAMP();
    if (threadIdx.x < kClasses) ccnt[threadIdx.x] = 0u;
    if (threadIdx.x == 64) {
        if (b == 0) { ctl->ticket = 0u; ctl->cursor = 0u; }
        if (counts) { counts[2 * b] = 0ull; counts[2 * b + 1] = 0ull; }
    }
    if ((threadIdx.x >> 5) < NS) {       // warp 0 (and warp 1 for the second SQ): the per-sample constants, fp64, spread over lanes
        __shared__ double psh[NS][12];
        const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
        double* p = psh[w];
        const void* params = w == 0 ? params_a : params_b;
        if (lane < 12)
            p[lane] = dtype == SQ_F64 ? static_cast<const double*>(params)[12 * (size_t)b + lane]
                                      : (double)static_cast<const float*>(params)[12 * (size_t)b + lane];
        __syncwarp();
        double hp_l = 0.0, hrn = 1.0;
        if (heads) {     // rows are raw network-head outputs (sq_implicit_loss_heads): heads_forward(), one output per lane
            double v = 0.0;
            if (lane < 8) { hp_l = (double)(float)(1.0 / (1.0 + exp(-p[lane]))); v = hp_l; }
            else if (lane < 12) {
                hrn = 1.0 / sqrt(p[8] * p[8] + p[9] * p[9] + p[10] * p[10] + p[11] * p[11]);
                v = (double)(float)(p[lane] * hrn);
            }
            __syncwarp();
            if (lane < 12) p[lane] = v;
            __syncwarp();
        }
        if (lane < 4) prep_part(p, clamp != 0, g, Ssh[w], lane);        // rows 0..2 of the scaled rotation; exponents
        __syncwarp();
        if (lane == 0) prep_finish(p, clamp != 0, g, Ssh[w]);
        __syncwarp();
        if (heads) {
            if (lane < 8) Ssh[w].hp[lane] = hp_l;
            if (lane == 8) { Ssh[w].heads = 1; Ssh[w].hrn = hrn; }
        }
        SQ_STAMP();
    }
    // ImplicitLoss: sum |target| over the sample's n x n pixels, by the warps that are not busy with the fp64 prep (it
    // hides behind it).  The column kernel then only adds |depth - t| - |t| for the columns it actually walks, so
    // columns without occupancy need neither their pixel nor any other work.  Fixed order: bit-reproducible.
    if (tv_sum) {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        if (warp >= NS) {
            const int t = threadIdx.x - 32 * NS, T = THREADS - 32 * NS, npix = g.n * g.n;
            double acc0 = 0.0, acc1 = 0.0;                    // fp64: an image of nearly equal depths rounds an fp32 sum one way
            const float* img = target + (size_t)b * tstride;
            // pixel index -> (row, col): shift / mask when n is a power of two (the usual render sizes), else a division
            const int sh = (g.n & (g.n - 1)) == 0 ? __ffs(g.n) - 1 : -1;
            auto pixel = [&](int iu) {
                const int r = sh >= 0 ? iu >> sh : iu / g.n, c = sh >= 0 ? iu & (g.n - 1) : iu - r * g.n;
                return __ldg(img + row_off[r] + col_off[c]);
            };
            int i = t;
            for (; i + 7 * T < npix; i += 8 * T) {         // eight independent loads in flight per thread (they miss to HBM)
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = pixel(i + u * T);
#pragma unroll
                for (int u = 0; u < 8; u += 2) { acc0 += (double)fabsf(v[u]); acc1 += (double)fabsf(v[u + 1]); }
            }
            {
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) { const int iu = i + u * T; v[u] = iu < npix ? pixel(iu) : 0.f; }
#pragma unroll
                for (int u = 0; u < 8; u += 2) { acc0 += (double)fabsf(v[u]); acc1 += (double)fabsf(v[u + 1]); }
            }
            double d = acc0 + acc1;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
            if (lane == 0) tv_part[warp] = d;
            SQ_STAMP();
        }
    }
    __syncthreads();
    SQ_STAMP();
    if (tv_sum && threadIdx.x == 0) {
        double d = 0.0;
        for (int w = NS; w < THREADS / 32; ++w) d += tv_part[w];
        tv_sum[b] = d;
    }
    for (int w = threadIdx.x; w < NS * kFullWords; w += THREADS) {
        const int which = w / kFullWords, i = w - which * kFullWords;
        reinterpret_cast<uint32_t*>((which == 0 ? out_a : out_b) + b)[i] = reinterpret_cast<const uint32_t*>(&Ssh[which])[i];
    }
    if (!queue) return;
    const int J = L.rows_per_sample;
    const int max_cost = L.cpt * L.n * NS;
    for (int j = threadIdx.x; j < J; j += THREADS) {
        int c = kClasses - 1;                              // proven empty (group_planes is an upper bound)
        int cost = 0;
        for (int k = 0; k < L.cpt; ++k) {
            const int group = j + k * J;
            if (group * 32 >= L.slots) break;
#pragma unroll
            for (int w = 0; w < NS; ++w) cost += group_planes(Ssh[w], g, L, bound, group, NS == 1 ? die : 0.f);
        }
        if (cost > 0) {
            if (kClasses == 8) { c = 0; while (c < kClasses - 2 && (cost << (c + 1)) <= max_cost) ++c; }
            else {               // kClasses / 8 classes per octave
                c = (int)((float)(kClasses / 8) * __log2f((float)max_cost / (float)cost));
                c = c < 0 ? 0 : (c > kClasses - 2 ? kClasses - 2 : c);
            }
        }
#ifdef SQ_ITEMLOG
        if (NS == 1 && b * J + j < 65536) { float* lg = g_planlog + 4 * (b * J + j); lg[0] = (float)c; lg[1] = (float)cost; lg[2] = lg[3] = 0.f; }
#endif
        cls[j] = (unsigned char)c;
        if (item_class) item_class[(size_t)b * J + j] = (unsigned char)c;      // finalize skips the rows of proven-empty items
        atomicAdd(&ccnt[c], 1u);
    }
    __syncthreads();
    SQ_STAMP();
    if (threadIdx.x < kClasses) {
        const unsigned int c = ccnt[threadIdx.x];
        cbase[threadIdx.x] = c ? atomicAdd(&ctl->qcount[threadIdx.x], c) : 0u;
        ccnt[threadIdx.x] = 0u;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < J; j += THREADS) {
        const int c = cls[j];
        const unsigned int r = atomicAdd(&ccnt[c], 1u);
#ifdef SQ_DEBUG_BOUNDS
        if (c < 0 || c >= kClasses || cbase[c] + r >= (unsigned int)cap || b * J + j >= cap) __trap();
#endif
        queue[(size_t)c * cap + cbase[c] + r] = b * J + j;
    }
#ifdef SQ_TIMELINE
    SQ_STAMP();
    if (b == 7 && (threadIdx.x == 0 || threadIdx.x == 100)) {
        const int o = threadIdx.x == 0 ? 0 : 8;
        for (int i = 0; i < nts; ++i) g_plan_ts[o + i] = ts[i];
        g_plan_ts[o + 7] = nts;
    }
#endif
}

// ------------------------------------------------------------------------------------------------ reductions
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ void acc_to_array(const Acc& a, float* v) {
#pragma unroll
    for (int i = 0; i < 3; ++i) { v[i] = a.gs[i]; v[12 + i] = a.wa[i]; }
#pragma unroll
    for (int i = 0; i < 9; ++i) v[3 + i] = a.gm[i];
    v[15] = a.ge[0]; v[16] = a.ge[1]; v[17] = a.loss;
}

__device__ __forceinline__ void array_to_acc(const float* v, Acc& a) {
#pragma unroll
    for (int i = 0; i < 3; ++i) { a.gs[i] = v[i]; a.wa[i] = v[12 + i]; }
#pragma unroll
    for (int i = 0; i < 9; ++i) a.gm[i] = v[3 + i];
    a.ge[0] = v[15]; a.ge[1] = v[16]; a.loss = v[17];
}

// per-thread Acc -> one row of kAccN floats per WARP, through the warp's own shared-memory tile: every lane writes
// its 18 sums (5 vector stores), lane i < 18 adds up column i over the 32 lanes in a fixed order.  37 shared-memory
// instructions and 32 adds per warp instead of the 90 shuffles + 90 adds of a butterfly per value.
constexpr int kRedStride = 20;           // floats per lane in the tile (80 bytes keeps float4 alignment)
constexpr int kRedFloats = 32 * kRedStride;
static_assert(kRow == kRedStride, "a partial row is one reduced tile row");

// lane i < kRow adds up column i of the warp's tile over the 32 lanes (fixed order) and stores the partial row
__device__ __forceinline__ void tile_reduce_store(const float* tile, float* row) {
    const int lane = threadIdx.x & 31;
    __syncwarp();
    if (lane < kRow) {
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
        for (int r = 0; r < 32; r += 4) {
            s0 += tile[(r + 0) * kRedStride + lane];
            s1 += tile[(r + 1) * kRedStride + lane];
            s2 += tile[(r + 2) * kRedStride + lane];
            s3 += tile[(r + 3) * kRedStride + lane];
        }
        row[lane] = (s0 + s1) + (s2 + s3);
    }
    __syncwarp();
}

__device__ __forceinline__ void tile_put(float* tile, const float* v /*[kRedStride]*/) {
    float4* mine = reinterpret_cast<float4*>(tile + (threadIdx.x & 31) * kRedStride);
#pragma unroll
    for (int q = 0; q < kRedStride / 4; ++q) mine[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}
__device__ __forceinline__ void tile_get(const float* tile, float* v /*[kRedStride]*/) {
    const float4* mine = reinterpret_cast<const float4*>(tile + (threadIdx.x & 31) * kRedStride);
#pragma unroll
    for (int q = 0; q < kRedStride / 4; ++q) { const float4 t = mine[q]; v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w; }
}

__device__ __forceinline__ void warp_reduce_store(const Acc& a, float* tile, float* row, bool nonzero) {
    const int lane = threadIdx.x & 31;
    if (!__any_sync(0xffffffffu, nonzero)) {          // e.g. image-border patches: no object, no loss, no gradient
        if (lane < kRow) row[lane] = 0.f;
        return;
    }
    float v[kRedStride];
    acc_to_array(a, v);
    v[18] = v[19] = 0.f;
    tile_put(tile, v);
    tile_reduce_store(tile, row);
}

// The same with the 32 lanes added in fp64 and the row rounded to fp32 once (the VJP kernel: its sums cancel only across rows,
// so each row's rounding has to be as small as it can be).  Every row is written (there is no loss to tell empty ones by).
__device__ __forceinline__ void warp_reduce_store_f64(const Acc& a, float* tile, float* row) {
    const int lane = threadIdx.x & 31;
    float v[kRedStride];
    acc_to_array(a, v);
    v[18] = v[19] = 0.f;
    tile_put(tile, v);
    __syncwarp();
    if (lane < kRow) {
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int r = 0; r < 32; r += 2) {
            s0 += (double)tile[r * kRedStride + lane];
            s1 += (double)tile[(r + 1) * kRedStride + lane];
        }
        row[lane] = (float)(s0 + s1);
    }
    __syncwarp();
}

// per-thread Acc -> one row of kAccN floats per BLOCK (point-list kernel)
__device__ __forceinline__ void block_reduce_store(const Acc& a, float (*red)[kAccN], float* row) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float v[kAccN];
    acc_to_array(a, v);
#pragma unroll
    for (int i = 0; i < kAccN; ++i) {
        const float s = warp_sum(v[i]);
        if (lane == 0) red[warp][i] = s;
    }
    __syncthreads();
    if (threadIdx.x < kRow) {
        float s = 0.f;
        if (threadIdx.x < kAccN) {
#pragma unroll
            for (int w = 0; w < kWarps; ++w) s += red[w][threadIdx.x];
        }
        row[threadIdx.x] = s;                          // slots 18, 19 (loss centring, ImplicitLoss only): 0
    }
}

__device__ __forceinline__ void load_sample(Sample* dst, const SampleFull* src) {   // whole block
    const uint32_t* s = reinterpret_cast<const uint32_t*>(src);
    uint32_t* d = reinterpret_cast<uint32_t*>(dst);
    for (int i = threadIdx.x; i < kSampleWords; i += blockDim.x) d[i] = s[i];
}

// Register-staged copy of one Sample by one warp: fetch() issues the global loads (their latency overlaps whatever
// the warp does next), commit() writes them to the warp's private shared-memory copy.
constexpr int kSampleRegs = (kSampleWords + 31) / 32;
struct SampleFetch {
    uint32_t w[kSampleRegs];
    __device__ __forceinline__ void fetch(const SampleFull* src, int lane) {
        const uint32_t* s = reinterpret_cast<const uint32_t*>(src);
#pragma unroll
        for (int j = 0; j < kSampleRegs; ++j) {
            const int i = lane + 32 * j;
            w[j] = i < kSampleWords ? __ldg(s + i) : 0u;
        }
    }
    __device__ __forceinline__ void commit(Sample* dst, int lane) const {
        uint32_t* d = reinterpret_cast<uint32_t*>(dst);
        __syncwarp();                                      // everyone is done with the previous contents
#pragma unroll
        for (int j = 0; j < kSampleRegs; ++j) {
            const int i = lane + 32 * j;
            if (i < kSampleWords) d[i] = w[j];
        }
        __syncwarp();
    }
};

// ------------------------------------------------------------------------------------------------ work distribution
// Positions 0 .. total-1 of the processing order.  The first position of a warp is its global warp index (no atomic
// burst when 2400 warps start at once; every position below the warp count has exactly one owner whenever that warp
// starts), later positions come from a cursor that counts on from there.
__device__ __forceinline__ int first_position() {
    return (int)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5));
}
__device__ __forceinline__ int next_position(unsigned int* cursor, int lane) {
    int pos = 0;
    if (lane == 0) pos = (int)(atomicAdd(cursor, 1u) + gridDim.x * (blockDim.x >> 5));
    return __shfl_sync(0xffffffffu, pos, 0);
}

// position -> work item through the cost-class queues the plan kernel filled (class 0 first)
struct WorkMap {
    unsigned int excl;       // lane k < kClasses: items in classes before k; other lanes: all items
    __device__ __forceinline__ void init(const Control* ctl, int lane) {
        const unsigned int cnt = lane < kClasses ? __ldcg(&ctl->qcount[lane]) : 0u;
        unsigned int incl = cnt;
#pragma unroll
        for (int o = 1; o < kClasses; o <<= 1) {
            const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        excl = incl - cnt;
    }
    __device__ __forceinline__ int item(const int* __restrict__ queue, int cap, int pos, int lane) const {
        if (!queue) return pos;
        const unsigned int m = __ballot_sync(0xffffffffu, lane < kClasses && (unsigned int)pos >= excl);
        const int c = 31 - __clz((int)m);                  // the highest class that starts at or before pos
        const unsigned int start = __shfl_sync(0xffffffffu, excl, c);
#ifdef SQ_DEBUG_BOUNDS      // tools/sanitize_case.py --bounds (compute-sanitizer is not available on the GPU pool)
        if (c < 0 || c >= kClasses || (unsigned int)pos - start >= (unsigned int)cap) __trap();
        const int it = __ldg(queue + (size_t)c * cap + ((unsigned int)pos - start));
        if (it < 0 || it >= cap) __trap();
        return it;
#endif
        return __ldg(queue + (size_t)c * cap + ((unsigned int)pos - start));
    }
};

// Depth-1 work pipeline of a persistent warp: the current item, and the next one claimed while the current one is
// being processed (claim() is called when the last column group of the current item starts: claimed earlier, the item
// would be kept from idle warps during the end-game; claimed later, the cursor -> queue -> Sample chain of L2 round
// trips would not be hidden).  Deeper pipelines (claims 2-3 items ahead) were measured 25 % slower: they undo the
// longest-first order while the items are still expensive.
// Positions from `empty_from` on are the last cost class: items the plan kernel has PROVEN to have no occupancy on any
// of their columns (its estimate is an upper bound).  The kernels never touch them (skip_empty).
struct WorkPipe {
    WorkMap wm;
    const int* queue; unsigned int* cursor;
    int cap, total, empty_from;
    int item, next;              // current / next work item (-1: none)
    int item_pos, next_pos;      // their positions in the processing order
    bool joined;                 // this warp has read the queue counters (retire() must be told)
    __device__ __forceinline__ void start(Control* ctl, const int* q, int cap_, int total_, bool skip_empty, int lane) {
        queue = q; cursor = &ctl->cursor; cap = cap_; total = total_; empty_from = total_;
        item = next = -1; item_pos = next_pos = total_;
        const int p0 = first_position();
        joined = p0 < total_;
        if (!joined) return;
        wm.init(ctl, lane);
        if (queue) empty_from = (int)__shfl_sync(0xffffffffu, wm.excl, kClasses - 1);
        if (skip_empty) total = empty_from;
        if (p0 < total) { item = wm.item(queue, cap, p0, lane); item_pos = p0; }
    }
    __device__ __forceinline__ bool claim(int lane) {
        next_pos = next_position(cursor, lane);
        next = next_pos < total ? wm.item(queue, cap, next_pos, lane) : -1;
        return next >= 0 && next_pos < empty_from;         // true: an item that needs its Sample
    }
    // The same claim in three stages, so that its two dependent L2 round trips (cursor, queue) are spent under other work
    // of the warp instead of stalling it: issue the cursor atomic; later turn its result into a queue lookup; later use
    // the item (the caller then fetches its Sample).
    // (ptxas turns an atomic add of a warp-uniform value -- atomicAdd(), atom.add or atom.inc in inline PTX alike -- into its
    // warp-aggregated form, whose broadcast shuffle sits right behind the ATOMG and waits out the whole round trip on the
    // spot.  An increment it cannot prove uniform -- 1 + a shuffled 0 -- keeps the atomic a plain fire-and-forget one.)
    unsigned int pend_pos;
    __device__ __forceinline__ void claim_issue(int lane) {
        const unsigned int one = 1u + __shfl_sync(0xffffffffu, 0u, lane);
        pend_pos = 0u;
        if (lane == 0) asm volatile("atom.global.add.u32 %0, [%1], %2;" : "=r"(pend_pos) : "l"(cursor), "r"(one) : "memory");
    }
    __device__ __forceinline__ void claim_lookup(int lane) {
        next_pos = (int)(__shfl_sync(0xffffffffu, pend_pos, 0) + gridDim.x * (blockDim.x >> 5));
        next = next_pos < total ? wm.item(queue, cap, next_pos, lane) : -1;
    }
    // decided on the position alone: the looked-up item id is not touched before the caller forms the Sample address
    __device__ __forceinline__ bool claim_finish() const { return next_pos < total && next_pos < empty_from; }
    __device__ __forceinline__ void rotate() { item = next; item_pos = next_pos; next = -1; }
};

// Every warp that read the queue counters reports when it leaves; the last of them puts the control block back to
// its between-calls state.  (`joiners` = warps whose first position is below the item count.)
__device__ __forceinline__ void retire(Control* ctl, bool joined, int total_items, int lane) {
    if (lane == 0 && joined) {
        const unsigned int warps = gridDim.x * (blockDim.x >> 5);
        const unsigned int joiners = (unsigned int)total_items < warps ? (unsigned int)total_items : warps;
        const unsigned int before = atomicAdd(&ctl->retired, 1u);
        if (before + 1u == joiners) {
            ctl->retired = 0u;
#pragma unroll
            for (int k = 0; k < kClasses; ++k) ctl->qcount[k] = 0u;
        }
    }
}

// ------------------------------------------------------------------------------------------------ ImplicitLoss
#ifdef SQ_TIMELINE     // tools/timeline.py: per-warp start / end timestamps and item counts of the implicit kernel
__device__ unsigned long long g_timeline[3 * 8192];
__device__ unsigned int g_classes[kClasses];
#endif
#ifdef SQ_PHASES       // tools/timeline.py SQ_PHASES: SM cycles of every warp of the fwd+bwd kernel, summed per phase
// 0 item set-up (sample, pixel loads, fp32 base, ranges)  1 exact base + z walk  2 claim issue, signs, counts scan, queue look-up
// 3 fp64 refinement  4 deal-out backward  5 column values + deal-out list to shared memory, folding into the tile
// 6 item epilogue (reduction, partial row)  7 waiting for the next item (claim, sample) and loop ends
__device__ unsigned long long g_phase[8];
#define SQ_PH(i) do { const long long n_ = clock64(); ph[i] += n_ - ph_t; ph_t = n_; } while (0)
#else
#define SQ_PH(i) do { } while (0)
#endif

#ifndef SQ_EARLY_MARGIN      // measured (profiles/tune_r02.txt run k): margins 1..3 are 1-2 us SLOWER per call than none -> off
#define SQ_EARLY_MARGIN 0
#endif
// dynamic shared memory of the fwd+bwd kernel, per warp: the pool's 4 float arrays + 11 x 32 column values
constexpr size_t kImplicitBwdSmemPerWarp = (size_t)kBwdPool * 4 * sizeof(float) + 11 * 32 * sizeof(float);
static_assert(kImplicitBwdSmemPerWarp % 32 == 0, "per-warp regions stay 32-byte aligned (BwdQueue::where carries the lane in its low bits)");

// VJP (with BWD; sq_depth_projection_vjp): `target` is the upstream gradient dL/d depth [batch, n, n] in image orientation and
// takes the place of sign(depth - target) as the column's weight; no loss, no depth, partial-row slots 17-19 stay 0.
template <bool BWD, int THREADS, int MINB, int CPTMAX, bool VJP = false>      // CPTMAX: upper limit of L.cpt
__global__ void __launch_bounds__(THREADS, MINB)
implicit_kernel(const SampleFull* __restrict__ samples, Grid g, Layout L, ImplicitParams P, int total_items,
                Control* __restrict__ ctl, const int* __restrict__ queue, int cap,
                const float* __restrict__ target, long long tstride, const int* __restrict__ row_off,
                const int* __restrict__ col_off, float* __restrict__ partials, float* __restrict__ depth_out) {
    __shared__ Sample Ssh[THREADS / 32];
#if SQ_TILE_ALIAS && defined(SQ_BWD_COMPACT)
    // the fwd+bwd kernel's reduction tile lives in the warp's pool arrays, which are dead by the time the item's sums
    // are put there (one column group per item only): shared memory for 5 blocks per SM
    static_assert(!BWD || CPTMAX == 1, "SQ_TILE_ALIAS needs one column group per work item");
    static_assert(4 * kBwdPool >= kRedFloats, "pool arrays too small to hold the tile");
    __shared__ __align__(16) float tiles_static[BWD ? 1 : THREADS / 32][kRedFloats];
#else
    __shared__ __align__(16) float tiles_static[THREADS / 32][kRedFloats];
#endif
#ifdef SQ_BWD_COMPACT       // per warp, in dynamic shared memory (BWD only; implicit_bwd_smem_bytes): the pool of gradient-carrying
                            // points (BwdQueue arrays), per-column data for them
    constexpr int kQN = kBwdPool;
    extern __shared__ __align__(32) unsigned char dyn_smem[];
    float* const qbuf = reinterpret_cast<float*>(dyn_smem + (size_t)(threadIdx.x >> 5) * kImplicitBwdSmemPerWarp);      // [4][kQN]
    float* const colinfo_w = qbuf + 4 * kQN;                                                                         // [11][32]
#endif
#if SQ_TILE_ALIAS && defined(SQ_BWD_COMPACT)
    float* const tile_w = BWD ? qbuf : tiles_static[threadIdx.x >> 5];
#else
    float* const tile_w = tiles_static[threadIdx.x >> 5];
#endif
    static_assert(!VJP || BWD, "the VJP mode is a mode of the fwd+bwd kernel");
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Sample& S = Ssh[warp];
#if defined(SQ_BWD_COMPACT) && !defined(SQ_TABLES_GLOBAL)
    // the tables of the fp64 refinement, copied to shared memory once per block (3 KB; they are read with per-lane indices)
    __shared__ __align__(16) double tabs[BWD ? 384 : 130];      // (forward-only: never read)
    constexpr int kTabRegs = (384 + THREADS - 1) / THREADS;
    double tab_reg[kTabRegs];
    if (BWD) {                                              // loads issued now, stored after the first work item is claimed
#pragma unroll
        for (int r = 0; r < kTabRegs; ++r) {
            const int i = threadIdx.x + r * THREADS;
            tab_reg[r] = i < 128 ? kExp2TabDev[i] : (i < 384 ? kLog2TabDev[i - 128] : 0.0);
        }
    }
    const RefTabs tb{tabs, tabs + 128};
#else
    const RefTabs tb = default_tabs();
#endif
    // Persistent warps pull work items from a global cursor, most expensive first (plan kernel).  The next item and its
    // Sample are fetched while the current item is processed.  No block-level barrier anywhere.
    // Items the plan kernel has proven empty are never touched: depth is exactly 0 on all their columns (depth_out was
    // cleared by the host), their loss sum |target| is part of the per-sample offset the plan kernel computed, their
    // partial rows were zeroed there.  What this kernel accumulates as "loss" is |depth - t| - |t| per walked column.
    pdl_wait();                                           // the plan kernel's Samples, queues and counters
    pdl_trigger();                                        // the finalize kernel may become resident (it waits for this grid)
#ifdef SQ_TIMELINE
    const unsigned long long t_begin = gtime();
    unsigned long long t_last_fetch = t_begin, n_items = 0;
    if (BWD && blockIdx.x == 0 && threadIdx.x < kClasses) g_classes[threadIdx.x] = ctl->qcount[threadIdx.x];
#endif
    WorkPipe wp;
    wp.start(ctl, queue, cap, total_items, true, lane);
#ifdef SQ_PHASES
    long long ph[8] = {0, 0, 0, 0, 0, 0, 0, 0}, ph_t = clock64();
#endif
    {
        SampleFetch pre;
        if (wp.item >= 0) pre.fetch(samples + L.sample_of(wp.item), lane);
#if defined(SQ_BWD_COMPACT) && !defined(SQ_TABLES_GLOBAL)
        if (BWD) {
#pragma unroll
            for (int r = 0; r < kTabRegs; ++r) { const int i = threadIdx.x + r * THREADS; if (i < 384) tabs[i] = tab_reg[r]; }
            __syncthreads();                               // the only block-level barrier: every warp passes here once
        }
#endif
        while (wp.item >= 0) {
#ifdef SQ_TIMELINE
            t_last_fetch = gtime(); ++n_items;
#endif
            int b, chunk;
            L.split(wp.item, b, chunk);
#ifdef SQ_ITEMLOG
            const long long il_t0 = clock64(); long long il_walk = 0; int il_q = 0, il_qr = 0;
#endif
            SQ_PH(7);
            pre.commit(&S, lane);
            SQ_COUNT_HOOK(4, 1);

            // Per-thread sums of the item live in the warp's shared-memory tile (the layout the final reduction reads),
            // not in 18 registers: they are touched once per non-empty column.
            float loss_sum = 0.f;
            bool folded = false;
            ColIter it;
            it.init(L, chunk, lane);
            // the item's target pixels (VJP: upstream pixels): loads issued up front (they miss to HBM), used after the z walks
            float tvs[CPTMAX];
            {
                ColIter pt = it;
#pragma unroll
                for (int k = 0; k < CPTMAX; ++k) {
                    tvs[k] = 0.f;
                    if (target && k < L.cpt) {
                        if (pt.valid(L))
                            tvs[k] = VJP ? __ldg(target + ((size_t)b * g.n + (g.n - 1 - pt.ib)) * g.n + pt.ia)
                                         : __ldg(target + (size_t)b * tstride + row_off[g.n - 1 - pt.ib] + col_off[pt.ia]);
                        pt.next(L);
                    }
                }
            }
#pragma unroll 1
            for (int k = 0; k < L.cpt; ++k) {
#ifdef SQ_EARLY_CLAIM
                if (k == L.cpt - 1 && wp.claim(lane)) pre.fetch(samples + L.sample_of(wp.next), lane);
#endif
                const int ia = it.ia, ib = it.ib;
                const bool valid = it.valid(L);
                const int row = g.n - 1 - ib, col = ia;        // classes.py:279: img[row, col] = depth[x = col, y = n-1-row]
                it.next(L);
                // which planes can hold occupancy: decided from the fp32 base; the exact (fp64) one is formed only for
                // groups that have some
                float b32[3];
                column_base_f32(S, g, valid ? ia : 0, valid ? ib : 0, b32);
                int c_lo, c_hi;
                column_range(S, g, P.bound, b32, c_lo, c_hi);
                if (!valid) { c_lo = 0; c_hi = -1; }           // masked lanes do not widen the warp's range
                const int own_lo = c_hi >= c_lo ? c_lo : g.n;  // this lane's own range (the early exit of the walk looks at it)
                warp_range(g.n, c_lo, c_hi);
                if (c_hi < c_lo) {                             // warp-uniform: no occupancy anywhere, depth is exactly 0
#ifndef SQ_EARLY_CLAIM
                    if (k == L.cpt - 1 && wp.claim(lane)) pre.fetch(samples + L.sample_of(wp.next), lane);
#endif
                    continue;
                }
                SQ_COUNT_HOOK(5, 1);
                SQ_PH(0);
#ifdef SQ_ITEMLOG
                const long long il_w0 = clock64();
#endif
#if defined(SQ_BWD_COMPACT) && !defined(SQ_NO_STAGED_CLAIM) && !defined(SQ_EARLY_CLAIM) && SQ_EARLY_MARGIN > 0
                // Far from the end of the queue the cursor atomic goes out BEFORE the walk (its L2 round trip then costs
                // nothing); in the end-game -- fewer than SQ_EARLY_MARGIN items per warp left -- an item claimed before a
                // long walk would be work no idle warp can take, so the claim waits until after the walk (see below).
                const bool early = BWD && k == L.cpt - 1 &&
                                   wp.item_pos + SQ_EARLY_MARGIN * (int)(gridDim.x * (THREADS / 32)) < wp.total;
                if (early) wp.claim_issue(lane);
#else
                const bool early = false;
#endif
                float bh[3], bl[3], cg[11], dxy[2];
                column_base(S, g, valid ? ia : 0, valid ? ib : 0, bh, bl, dxy);
                float depth;
#ifndef SQ_FIXHOIST      // hoisting the exact-zero fix-up out of the walk (two copies of the loop): measured 1 us
                         // SLOWER per call once everything else was in place (profiles/tune_r01.txt) -> off
#ifdef SQ_BWD_COMPACT
                // (the entries' tags sit in the plane index's low mantissa bits: small integers, and plane 0's own "index" below 1)
                const int pool = (g.n <= kPoolMaxPlanes && S.cf0 < 1.0f) ? kQN : 0;
                float U = 0.f; int nr = 0, top = pool - 1, head = kNoLink; bool spilled = false;
                unsigned where = (unsigned)__cvta_generic_to_shared(qbuf) | (unsigned)lane;
                asm volatile("" : "+r"(where));                       // kept in a register (sq_core.cuh plane_scan)
                const BwdQueue qwarp{qbuf, qbuf + kQN, qbuf + 2 * kQN, qbuf + 3 * kQN, pool, lane, where};
                depth = implicit_column<BWD, true, BWD>(S, g, P, bh, bl, c_lo, c_hi, own_lo, cg, &qwarp, &U, &nr, &top, &spilled, &head);
#else
                depth = implicit_column<BWD, true>(S, g, P, bh, bl, c_lo, c_hi, own_lo, cg);
#endif
#else
                if (__any_sync(0xffffffffu, column_zero_possible(S, bh)))
                    depth = implicit_column<BWD, true>(S, g, P, bh, bl, c_lo, c_hi, own_lo, cg);
                else
                    depth = implicit_column<BWD, false>(S, g, P, bh, bl, c_lo, c_hi, own_lo, cg);
#endif
                SQ_PH(1);
#ifdef SQ_ITEMLOG
                il_walk += clock64() - il_w0;
#endif
#ifndef SQ_EARLY_CLAIM
                // Claim the next item only now, after the walk: the cursor -> queue -> Sample chain then stalls this warp
                // for ~1300 cycles, but the kernel is bound by instruction dispatch and the other warps of the scheduler
                // fill the gap; an item claimed at the start of a long walk, on the other hand, is work no idle warp can
                // take -- during the end-game that was the tail of the kernel.
#if defined(SQ_BWD_COMPACT) && !defined(SQ_NO_STAGED_CLAIM)
                const bool staged = BWD && k == L.cpt - 1;     // fwd+bwd: the claim is spread over the backward passes
                if (staged) { if (!early) wp.claim_issue(lane); }
                else
#else
                const bool staged = false;
#endif
                if (k == L.cpt - 1 && wp.claim(lane)) pre.fetch(samples + L.sample_of(wp.next), lane);
#endif
#if defined(SQ_BWD_COMPACT)
                if (BWD) {
                    // sign of (depth - target) per column (VJP: the upstream pixel); 0 for masked lanes
                    float wsg = 0.f;
                    // the target pixel (issued before the walk, a miss to HBM) is first touched HERE: without the fence the
                    // compiler forms |tv| right behind the load and the warp waits out the miss before it starts walking
                    float tv = tvs[0];                         // select, not an indexed load: tvs stays in registers
#pragma unroll
                    for (int q = 1; q < CPTMAX; ++q) tv = k == q ? tvs[q] : tv;
                    asm volatile("" : "+f"(tv));
                    if (valid && VJP) {
                        wsg = tv;
                    } else if (valid) {
                        if (depth_out) depth_out[((size_t)b * g.n + row) * g.n + col] = depth;
                        const float diff = depth - tv;
                        loss_sum += fabsf(diff) - fabsf(tv);
                        wsg = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
                    }
                    // the pool's front (to refine in fp64) and back entries are already compact lists: counts are warp-uniform.
                    // (Entries of a column whose sign turned out 0 stay in the lists and contribute exactly 0.)
                    const int total_r = nr, total = nr + (pool - 1 - top);
                    const bool any_spill = __any_sync(0xffffffffu, spilled && wsg != 0.f);
#ifdef SQ_ITEMLOG
                    il_q += total + (any_spill ? 1000 : 0); il_qr += total_r;
#endif
#ifndef SQ_EARLY_CLAIM
                    if (staged) {
                        wp.claim_lookup(lane);
                        if (total == 0 && wp.claim_finish()) pre.fetch(samples + L.sample_of(wp.next), lane);
                    }
#endif
                    SQ_PH(2);
                    if (total > 0 || any_spill) {
                        Acc acc;
                        float v[kRedStride];
                        if (folded) { tile_get(tile_w, v); array_to_acc(v, acc); } else acc_zero(acc);
                        if (spilled && wsg != 0.f) implicit_fold(acc, cg, wsg, dxy[0], dxy[1]);      // handled on the spot
                        if (total > 0) {
                            float* ci = colinfo_w;
                            ci[0 * 32 + lane] = bh[0]; ci[1 * 32 + lane] = bh[1]; ci[2 * 32 + lane] = bh[2];
                            ci[3 * 32 + lane] = bl[0]; ci[4 * 32 + lane] = bl[1]; ci[5 * 32 + lane] = bl[2];
                            ci[6 * 32 + lane] = wsg; ci[7 * 32 + lane] = dxy[0]; ci[8 * 32 + lane] = dxy[1];
                            ci[9 * 32 + lane] = U; ci[10 * 32 + lane] = __int_as_float(head);
                            __syncwarp();
                            SQ_COUNT_HOOK(6, total); SQ_COUNT_HOOK(7, total_r);
                            SQ_COUNT_HOOK(3, (total_r + 31) / 32); SQ_COUNT_HOOK(2, (total + 31) / 32);
                            SQ_PH(5);
                            // 1. the entries near the surface, dealt out evenly: x in fp64 (sq_core.cuh "fp64 refinement")
                            // (two rounds in flight where there are that many: measured 6 us SLOWER per call,
                            // profiles/tune_r02.txt: the second chain's registers cost the walk its allocation)
                            for (int jr = lane; jr < total_r; jr += 32) {
                                const int l_ = entry_lane(qwarp.cf[jr]);
                                queue_refine_entry(S, g.step, P.kl, qwarp, jr,
                                                   f2d(ci[0 * 32 + l_]) + f2d(ci[3 * 32 + l_]), f2d(ci[1 * 32 + l_]) + f2d(ci[4 * 32 + l_]),
                                                   f2d(ci[2 * 32 + l_]) + f2d(ci[5 * 32 + l_]), tb);
                            }
                            __syncwarp();
                            SQ_PH(3);
                            const float tau = P.tl * (float)kLn2;
#ifdef SQ_DEPTH_SHIFT       // the refined occupancies' first-order effect on the rendered depth: measured below the loss's other
                            // fp32 errors on every workload (profiles/tune_r02.txt) and 2 us per call -> off
                            if (!VJP && head != kNoLink) loss_sum = fmaf(wsg * tau * g.inv_n, queue_depth_shift(qwarp, head, U), loss_sum);
#endif
#ifndef SQ_EARLY_CLAIM
                            if (staged && wp.claim_finish()) pre.fetch(samples + L.sample_of(wp.next), lane);
#endif
                            // 2. + 3. all entries, dealt out evenly: suffix weight (corrected for the refined entries of the
                            // entry's column), forward redone, backward; two rounds in flight (two independent MUFU chains)
                            auto dealt = [&](int j, Bwd& bq, float& cfq, float& dx_, float& dy_) {
                                const bool has = j < total;
                                // front entries first, then the back ones from the pool's end; idle lane of the last round: a
                                // slot that may never have been written
                                const int at = has ? (j < total_r ? j : kQN - 1 - (j - total_r)) : 0;
                                const float tagged = has ? qwarp.cf[at] : 1.0f, x_ = has ? qwarp.x[at] : 0.0f;
                                const int l_ = entry_lane(tagged);      // (1.0f: lane 0, plane 1)
                                const float cf_ = entry_cf(S, tagged);
                                const float sw_ = has ? queue_suffix_weight(qwarp, at, __float_as_int(ci[10 * 32 + l_]), ci[9 * 32 + l_], tau) : 0.0f;
                                const float cbh[3] = {ci[0 * 32 + l_], ci[1 * 32 + l_], ci[2 * 32 + l_]};
                                const float cbl[3] = {ci[3 * 32 + l_], ci[4 * 32 + l_], ci[5 * 32 + l_]};
                                queue_entry_backward<true>(S, cbh, cbl, cf_, x_, sw_, ci[6 * 32 + l_], has, bq);
                                cfq = cf_; dx_ = ci[7 * 32 + l_]; dy_ = ci[8 * 32 + l_];
                            };
                            int j = lane;
#if SQ_DENSE_ILP == 2
                            for (; j - lane + 32 < total; j += 64) {
                                Bwd b0, b1; float c0, c1, x0, x1, y0, y1;
                                dealt(j, b0, c0, x0, y0);
                                dealt(j + 32, b1, c1, x1, y1);
                                acc_add_point(acc, b0, c0, x0, y0);
                                acc_add_point(acc, b1, c1, x1, y1);
                            }
#endif
                            for (; j - lane < total; j += 32) {
                                Bwd b0; float c0, x0, y0;
                                dealt(j, b0, c0, x0, y0);
                                acc_add_point(acc, b0, c0, x0, y0);
                            }
                            __syncwarp();
                            SQ_PH(4);
                        }
                        acc_to_array(acc, v);
                        v[18] = v[19] = 0.f;
                        tile_put(tile_w, v);
                        folded = true;
                        SQ_PH(5);
                    }
                } else
#endif
                if (valid) {
                    if (depth_out && !VJP) depth_out[((size_t)b * g.n + row) * g.n + col] = depth;
                    if (target) {
                        float tv = tvs[0];
#pragma unroll
                        for (int q = 1; q < CPTMAX; ++q) tv = k == q ? tvs[q] : tv;
                        asm volatile("" : "+f"(tv));           // first touch of the pixel after the walk (see above)
                        const float diff = VJP ? tv : depth - tv;
                        if (!VJP) loss_sum += fabsf(diff) - fabsf(tv);
                        if (BWD && diff != 0.f) {
                            float v[kRedStride];
                            Acc acc;
                            if (folded) { tile_get(tile_w, v); array_to_acc(v, acc); } else acc_zero(acc);
                            implicit_fold(acc, cg, VJP ? diff : (diff > 0.f ? 1.f : -1.f), dxy[0], dxy[1]);
                            acc_to_array(acc, v);
                            v[18] = v[19] = 0.f;
                            tile_put(tile_w, v);
                            folded = true;
                        }
                    }
                }
            }
            SQ_PH(7);
            if (target) {
                float* row = partials + ((size_t)b * L.rows_per_sample + chunk) * kRow;
                const unsigned nz = __ballot_sync(0xffffffffu, loss_sum != 0.f);
                if (!nz && !__any_sync(0xffffffffu, folded)) {
                    if (lane < kRow) row[lane] = 0.f;
                } else {
                    if (!folded) {
                        float4* mine = reinterpret_cast<float4*>(tile_w + lane * kRedStride);
#pragma unroll
                        for (int q = 0; q < kRedStride / 4; ++q) mine[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                    // The lanes' loss terms |depth - t| - |t| are all close to -|t| when the object fills the patch, and
                    // an fp32 sum of 32 nearly equal numbers rounds the same way 32 times (measured: +1e-7 on the loss of
                    // every sample, 4e-5 of a loss of 3e-3).  So the row carries the terms relative to one of them
                    // (slot 17: small numbers, summed exactly enough), that one (slot 18) and the count (slot 19);
                    // finalize adds slot 17 + slot 18 x slot 19 in fp64.
                    const float c = nz ? __shfl_sync(0xffffffffu, loss_sum, __ffs((int)nz) - 1) : 0.f;
                    tile_w[lane * kRedStride + 17] = loss_sum != 0.f ? loss_sum - c : 0.f;
                    if (lane == 0) { tile_w[18] = c; tile_w[19] = (float)__popc(nz); }
                    tile_reduce_store(tile_w, row);
                }
            }
            SQ_PH(6);
#ifdef SQ_ITEMLOG
            if (BWD && lane == 0 && wp.item < 65536) {
                int* lg = g_itemlog + 4 * wp.item;
                lg[0] = (int)(clock64() - il_t0); lg[1] = (int)il_walk; lg[2] = il_q; lg[3] = il_qr;
            }
#endif
            wp.rotate();
        }
    }
    retire(ctl, wp.joined, total_items, lane);
#ifdef SQ_PHASES
    if (BWD && lane == 0)
        for (int i = 0; i < 8; ++i) atomicAdd(&g_phase[i], (unsigned long long)ph[i]);
#endif
#ifdef SQ_TIMELINE
    if (BWD && lane == 0) {
        const int w = first_position();
        if (w < 8192) { g_timeline[3 * w] = t_begin; g_timeline[3 * w + 1] = gtime(); g_timeline[3 * w + 2] = (n_items << 40) | (t_last_fetch - t_begin); }
    }
#endif
}

// ------------------------------------------------------------------------------------------------ ExplicitLoss
template <bool BWD>
__global__ void __launch_bounds__(SQ_EXP_THREADS, SQ_EXP_MINB)
explicit_kernel(const SampleFull* __restrict__ tru, const SampleFull* __restrict__ pred, Grid g, Layout L, float kl,
                float bound, int total_items, Control* __restrict__ ctl, const int* __restrict__ queue, int cap,
                float* __restrict__ partials) {
    __shared__ Sample Tsh[SQ_EXP_THREADS / 32], Psh[SQ_EXP_THREADS / 32];
    __shared__ __align__(16) float tiles[SQ_EXP_THREADS / 32][kRedFloats];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Sample& St = Tsh[warp];
    Sample& Sp = Psh[warp];
    WorkPipe wp;
    wp.start(ctl, queue, cap, total_items, true, lane);      // proven-empty items are dropped (their rows: plan kernel)
    {
        SampleFetch pre_t, pre_p;
        if (wp.item >= 0) { pre_t.fetch(tru + L.sample_of(wp.item), lane); pre_p.fetch(pred + L.sample_of(wp.item), lane); }
        while (wp.item >= 0) {
            const int item = wp.item;
            int b, chunk;
            L.split(item, b, chunk);
            pre_t.commit(&St, lane);
            pre_p.commit(&Sp, lane);
            Acc acc;
            acc_zero(acc);
            ColIter it;
            it.init(L, chunk, lane);
            for (int k = 0; k < L.cpt; ++k, it.next(L)) {
                const bool valid = it.valid(L);
                const int ia = valid ? it.ia : 0, ib = valid ? it.ib : 0;
                float bht[3], blt[3], bhp[3], blp[3];
                float dxy[2];
                Range rt, rp;
                column_base_f32(St, g, ia, ib, bht);           // fp32 bases decide the ranges (see implicit_kernel)
                column_base_f32(Sp, g, ia, ib, bhp);
                column_range(St, g, bound, bht, rt.lo, rt.hi);
                column_range(Sp, g, bound, bhp, rp.lo, rp.hi);
                if (!valid) { rt.lo = rp.lo = 0; rt.hi = rp.hi = -1; }      // masked lanes do not widen the warp's range
                warp_range(g.n, rt.lo, rt.hi);
                warp_range(g.n, rp.lo, rp.hi);
                if (rt.hi < rt.lo && rp.hi < rp.lo) continue;               // both occupancies 0 on the whole column
                column_base(St, g, ia, ib, bht, blt);
                column_base(Sp, g, ia, ib, bhp, blp, dxy);
                Acc col;
                acc_zero(col);
                const float sq = explicit_column<BWD>(St, Sp, g, kl, bht, blt, bhp, blp, rt, rp, dxy[0], dxy[1], col);
                if (valid) {
                    acc.loss += sq;
                    if (BWD) {
#pragma unroll
                        for (int i = 0; i < 3; ++i) { acc.gs[i] += col.gs[i]; acc.wa[i] += col.wa[i]; }
#pragma unroll
                        for (int i = 0; i < 9; ++i) acc.gm[i] += col.gm[i];
                        acc.ge[0] += col.ge[0]; acc.ge[1] += col.ge[1];
                    }
                }
            }
            // claimed after the walk, not before it: see implicit_kernel
            if (wp.claim(lane)) { pre_t.fetch(tru + L.sample_of(wp.next), lane); pre_p.fetch(pred + L.sample_of(wp.next), lane); }
            warp_reduce_store(acc, tiles[warp], partials + (size_t)item * kRow, acc.loss != 0.f);
            wp.rotate();
        }
    }
    retire(ctl, wp.joined, total_items, lane);
}

// Vector-Jacobian product of the occupancy field (sq_occupancy_vjp): explicit_kernel's work loop with the predicted SQ
// alone and explicit_column's VJP mode -- the upstream voxels up[b][x][y][z] (sq_field's layout) weight the points, the cut is
// `kact` bits, the walk covers the z range culled at the same level (`bound`).  A sibling kernel rather than a third
// instantiation of explicit_kernel, so that the loss kernels keep their parameter lists and code.
__global__ void __launch_bounds__(SQ_EXP_THREADS, SQ_EXP_MINB)
explicit_vjp_kernel(const SampleFull* __restrict__ pred, Grid g, Layout L, float kl, float bound, float kact,
                    const float* __restrict__ up, int total_items, Control* __restrict__ ctl, const int* __restrict__ queue,
                    int cap, float* __restrict__ partials) {
    __shared__ Sample Psh[SQ_EXP_THREADS / 32];
    __shared__ __align__(16) float tiles[SQ_EXP_THREADS / 32][kRedFloats];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Sample& Sp = Psh[warp];
    WorkPipe wp;
    wp.start(ctl, queue, cap, total_items, true, lane);      // proven-empty items are dropped (their rows: plan kernel)
    {
        SampleFetch pre_p;
        if (wp.item >= 0) pre_p.fetch(pred + L.sample_of(wp.item), lane);
        while (wp.item >= 0) {
            const int item = wp.item;
            int b, chunk;
            L.split(item, b, chunk);
            pre_p.commit(&Sp, lane);
            Acc acc;
            acc_zero(acc);
            ColIter it;
            it.init(L, chunk, lane);
            for (int k = 0; k < L.cpt; ++k, it.next(L)) {
                const bool valid = it.valid(L);
                const int ia = valid ? it.ia : 0, ib = valid ? it.ib : 0;
                float bhp[3], blp[3];
                float dxy[2];
                Range rp;
                column_base_f32(Sp, g, ia, ib, bhp);
                column_range(Sp, g, bound, bhp, rp.lo, rp.hi);
                if (!valid) { rp.lo = 0; rp.hi = -1; }
                warp_range(g.n, rp.lo, rp.hi);
                if (rp.hi < rp.lo) continue;                                  // every point of the group below the cut
                column_base(Sp, g, ia, ib, bhp, blp, dxy);
                const float* col = valid ? up + (((size_t)b * g.n + ia) * g.n + ib) * g.n : nullptr;
                Acc c;
                acc_zero(c);
                explicit_column<true, true>(Sp, Sp, g, kl, bhp, blp, bhp, blp, Range{0, -1}, rp, dxy[0], dxy[1], c, col, kact);
                if (valid) {
#pragma unroll
                    for (int i = 0; i < 3; ++i) { acc.gs[i] += c.gs[i]; acc.wa[i] += c.wa[i]; }
#pragma unroll
                    for (int i = 0; i < 9; ++i) acc.gm[i] += c.gm[i];
                    acc.ge[0] += c.ge[0]; acc.ge[1] += c.ge[1];
                }
            }
            if (wp.claim(lane)) pre_p.fetch(pred + L.sample_of(wp.next), lane);
            warp_reduce_store_f64(acc, tiles[warp], partials + (size_t)item * kRow);
            wp.rotate();
        }
    }
    retire(ctl, wp.joined, total_items, lane);
}

// MSE of the occupancy field against voxel data (sq_voxel_loss): explicit_vjp_kernel's work loop with explicit_column's VOX
// mode -- the voxels vox[b][x][y][z] (V = float or uint8_t, times vscale) take the place of the upstream and of o_t.  Every
// voxel counts, including those the walk never visits, so no item and no column is skipped: a column group whose warp range
// is empty, and every column of an item the plan kernel proved empty (its Sample is not even fetched), adds its sum of v^2
// (voxel_sq_outside).  All terms are non-negative and each voxel is read once.  BWD = false: the same walk, loss only.
template <bool BWD, typename V>
__global__ void __launch_bounds__(SQ_EXP_THREADS, SQ_EXP_MINB)
explicit_vox_kernel(const SampleFull* __restrict__ pred, Grid g, Layout L, float kl, float bound, float kact,
                    const V* __restrict__ vox, float vscale, int total_items, Control* __restrict__ ctl,
                    const int* __restrict__ queue, int cap, float* __restrict__ partials) {
    __shared__ Sample Psh[SQ_EXP_THREADS / 32];
    __shared__ __align__(16) float tiles[SQ_EXP_THREADS / 32][kRedFloats];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Sample& Sp = Psh[warp];
    WorkPipe wp;
    wp.start(ctl, queue, cap, total_items, false, lane);     // proven-empty items too: their voxels still count
    {
        SampleFetch pre_p;
        if (wp.item >= 0) pre_p.fetch(pred + L.sample_of(wp.item), lane);
        while (wp.item >= 0) {
            const int item = wp.item;
            const bool empty = wp.item_pos >= wp.empty_from;            // warp-uniform; Sp is stale then and never read
            int b, chunk;
            L.split(item, b, chunk);
            pre_p.commit(&Sp, lane);
            Acc acc;
            acc_zero(acc);
            ColIter it;
            it.init(L, chunk, lane);
            for (int k = 0; k < L.cpt; ++k, it.next(L)) {
                const bool valid = it.valid(L);
                const int ia = valid ? it.ia : 0, ib = valid ? it.ib : 0;
                float bhp[3], blp[3];
                float dxy[2];
                Range rp{0, -1};
                if (!empty) {
                    column_base_f32(Sp, g, ia, ib, bhp);
                    column_range(Sp, g, bound, bhp, rp.lo, rp.hi);
                    if (!valid) { rp.lo = 0; rp.hi = -1; }
                    warp_range(g.n, rp.lo, rp.hi);
                }
                const V* col = valid ? vox + (((size_t)b * g.n + ia) * g.n + ib) * g.n : nullptr;
                if (rp.hi < rp.lo) {                                     // every point of the group below the cut
                    acc.loss += voxel_sq_outside(col, g.n, rp, vscale);
                    continue;
                }
                column_base(Sp, g, ia, ib, bhp, blp, dxy);
                Acc c;
                acc_zero(c);
                const float sq = explicit_column<BWD, true, true>(Sp, Sp, g, kl, bhp, blp, bhp, blp, Range{0, -1}, rp, dxy[0],
                                                                  dxy[1], c, col, kact, vscale);
                if (valid) {
                    acc.loss += sq;
                    if (BWD) {
#pragma unroll
                        for (int i = 0; i < 3; ++i) { acc.gs[i] += c.gs[i]; acc.wa[i] += c.wa[i]; }
#pragma unroll
                        for (int i = 0; i < 9; ++i) acc.gm[i] += c.gm[i];
                        acc.ge[0] += c.ge[0]; acc.ge[1] += c.ge[1];
                    }
                }
            }
            if (wp.claim(lane)) pre_p.fetch(pred + L.sample_of(wp.next), lane);
            warp_reduce_store_f64(acc, tiles[warp], partials + (size_t)item * kRow);
            wp.rotate();
        }
    }
    retire(ctl, wp.joined, total_items, lane);
}

// ------------------------------------------------------------------------------------------------ IoU
__global__ void __launch_bounds__(SQ_IOU_THREADS, SQ_IOU_MINB)
iou_kernel(const SampleFull* __restrict__ tru, const SampleFull* __restrict__ pred, Grid g, Layout L, int total_items,
           Control* __restrict__ ctl, const int* __restrict__ queue, int cap, unsigned long long* __restrict__ counts) {
    __shared__ Sample Tsh[SQ_IOU_THREADS / 32], Psh[SQ_IOU_THREADS / 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Sample& St = Tsh[warp];
    Sample& Sp = Psh[warp];
    WorkPipe wp;
    wp.start(ctl, queue, cap, total_items, true, lane);      // proven-empty items are dropped (their rows: plan kernel)
    {
        SampleFetch pre_t, pre_p;
        if (wp.item >= 0) { pre_t.fetch(tru + L.sample_of(wp.item), lane); pre_p.fetch(pred + L.sample_of(wp.item), lane); }
        while (wp.item >= 0) {
            const int item = wp.item;
            int b, chunk;
            L.split(item, b, chunk);
            pre_t.commit(&St, lane);
            pre_p.commit(&Sp, lane);
            unsigned inter = 0, uni = 0;
            ColIter it;
            it.init(L, chunk, lane);
            for (int k = 0; k < L.cpt; ++k, it.next(L)) {
                const bool valid = it.valid(L);
                const int ia = valid ? it.ia : 0, ib = valid ? it.ib : 0;
                float bht[3], blt[3], bhp[3], blp[3];
                Range rt, rp;
                column_base_f32(St, g, ia, ib, bht);           // fp32 bases decide the ranges (see implicit_kernel)
                column_base_f32(Sp, g, ia, ib, bhp);
                column_range(St, g, kIoUBound, bht, rt.lo, rt.hi);
                column_range(Sp, g, kIoUBound, bhp, rp.lo, rp.hi);
                if (!valid) { rt.lo = rp.lo = 0; rt.hi = rp.hi = -1; }
                warp_range(g.n, rt.lo, rt.hi);
                warp_range(g.n, rp.lo, rp.hi);
                if (rt.hi < rt.lo && rp.hi < rp.lo) continue;               // outside both: nothing to count
                column_base(St, g, ia, ib, bht, blt);
                column_base(Sp, g, ia, ib, bhp, blp);
                unsigned i = 0, u = 0;
                iou_column(St, Sp, tru + b, pred + b, g, ia, ib, bht, blt, bhp, blp, rt, rp, i, u);
                if (valid) { inter += i; uni += u; }
            }
            if (wp.claim(lane)) { pre_t.fetch(tru + L.sample_of(wp.next), lane); pre_p.fetch(pred + L.sample_of(wp.next), lane); }
            inter = __reduce_add_sync(0xffffffffu, inter);
            uni = __reduce_add_sync(0xffffffffu, uni);
            if (lane == 0 && (inter | uni)) {                 // integer atomics: order-independent, exact
                atomicAdd(counts + 2 * b, (unsigned long long)inter);
                atomicAdd(counts + 2 * b + 1, (unsigned long long)uni);
            }
            wp.rotate();
        }
    }
    retire(ctl, wp.joined, total_items, lane);
}

__global__ void iou_export_kernel(const unsigned long long* counts, int batch, long long* inter, long long* uni) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < batch) { inter[b] = (long long)counts[2 * b]; uni[b] = (long long)counts[2 * b + 1]; }
}

// ------------------------------------------------------------------------------------------------ LeastSquares
constexpr int kLsqPix = 4;               // pixels per thread of the point-list kernel

template <bool BWD>
__global__ void __launch_bounds__(kThreads)
lsq_kernel(const SampleFull* __restrict__ samples, int R, int items_per_sample,
           const float* __restrict__ target, long long tstride, const int* __restrict__ row_off,
           const int* __restrict__ col_off, float* __restrict__ partials) {
    __shared__ Sample S;
    __shared__ float red[kWarps][kAccN];
    const int item = blockIdx.x;
    const int b = item / items_per_sample, chunk = item - b * items_per_sample;
    load_sample(&S, samples + b);
    __syncthreads();
    Acc acc;
    acc_zero(acc);
    // kLsqPix pixels per thread, all loads issued before the first is used (they come from HBM; the kernel is a point
    // list read once, bound by memory latency x parallelism, not by arithmetic)
    float v[kLsqPix];
    int pixs[kLsqPix];
#pragma unroll
    for (int k = 0; k < kLsqPix; ++k) {
        pixs[k] = (chunk * kLsqPix + k) * kThreads + threadIdx.x;
        v[k] = 0.f;
        if (pixs[k] < R * R) {
            const int row = pixs[k] / R, col = pixs[k] - row * R;
            v[k] = __ldg(target + (size_t)b * tstride + row_off[row] + col_off[col]);
        }
    }
#pragma unroll
    for (int k = 0; k < kLsqPix; ++k) {
        if (v[k] > 0.f) {                                  // classes.py:363-368 (fp32 arithmetic, like the reference)
            const int row = pixs[k] / R, col = pixs[k] - row * R;
            const float px = (float)col / (float)R, py = 1.0f - (float)row / (float)R;
            acc.loss += lsq_point<BWD>(S, px, py, v[k], acc);
        }
    }
    block_reduce_store(acc, red, partials + (size_t)item * kRow);
}

// LeastSquares.energy_function on an explicit, compacted point list (classes.py:318-356): structure of arrays x[], y[],
// z[] (rows of `points`, `stride` floats apart) holding the lists of all samples back to back, sample b owning
// [offsets[b], offsets[b+1]).  One block per (sample, chunk of kThreads * 4 points); a thread reads four consecutive
// points of each coordinate row with one 16-byte load.  The chunk grid is aligned to multiples of four points of the
// WHOLE buffer (rows are 16-byte aligned and padded to a multiple of four), points outside the sample's range are masked.
// 12 bytes per point from HBM, read once.
template <bool BWD>
__global__ void __launch_bounds__(kThreads)
lsq_points_kernel(const SampleFull* __restrict__ samples, int chunks_per_sample, const float* __restrict__ points,
                  long long stride, const long long* __restrict__ offsets, float* __restrict__ partials) {
    __shared__ Sample S;
    __shared__ float red[kWarps][kAccN];
    const int item = blockIdx.x;
    const int b = item / chunks_per_sample, chunk = item - b * chunks_per_sample;
    load_sample(&S, samples + b);
    __syncthreads();
    Acc acc;
    acc_zero(acc);
    const long long lo = offsets[b], hi = offsets[b + 1];
    const long long base = (lo & ~3LL) + ((long long)chunk * kThreads + threadIdx.x) * 4;
    if (base < hi) {
        const float4 x4 = __ldg(reinterpret_cast<const float4*>(points + base));
        const float4 y4 = __ldg(reinterpret_cast<const float4*>(points + stride + base));
        const float4 z4 = __ldg(reinterpret_cast<const float4*>(points + 2 * stride + base));
        const float xs[4] = {x4.x, x4.y, x4.z, x4.w}, ys[4] = {y4.x, y4.y, y4.z, y4.w}, zs[4] = {z4.x, z4.y, z4.z, z4.w};
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (base + k >= lo && base + k < hi) acc.loss += lsq_point<BWD>(S, xs[k], ys[k], zs[k], acc);
    }
    block_reduce_store(acc, red, partials + (size_t)item * kRow);
}

// ------------------------------------------------------------------------------------------------ finalize
enum { FIN_IMPLICIT = 0, FIN_EXPLICIT = 1, FIN_LSQ = 2, FIN_OCC_VJP = 3 };     // FIN_OCC_VJP: z moment about plane_of_t()
                                                                               // (sq_occupancy_vjp and sq_voxel_loss)

// One block of kFinThreads per sample: every thread sums the partial rows r = t, t + kFinThreads, ... in fp64 (all loads
// independent: one L2 round trip), a fixed-order tree (shuffles inside a warp, then the warps in index order) gives the
// 18 totals, thread 0 applies the Jacobians.  The last block to arrive averages the batch in index order.  Fixed order
// everywhere: results are bit-reproducible run to run.
#ifndef SQ_FIN_THREADS
#define SQ_FIN_THREADS 128
#endif
constexpr int kFinThreads = SQ_FIN_THREADS;

template <int KIND>
__global__ void __launch_bounds__(kFinThreads)
finalize_kernel(const SampleFull* __restrict__ samples, Grid g, int batch, int items_per_sample,
                const float* __restrict__ partials, double loss_norm, double grad_scale,
                int dtype, void* __restrict__ grad, double* __restrict__ per_sample,
                double* __restrict__ per_sample_user, double* __restrict__ loss_out, unsigned int* ticket,
                const double* __restrict__ loss_offset, const unsigned char* __restrict__ item_class) {
    const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    __shared__ SampleFull S;
    __shared__ double wpart[kFinThreads / 32][kAccN];
    __shared__ double acc[kAccN];
    // the sample's record (written by the plan / prep kernel) into shared memory, while the partial rows are on their way
    for (int w = t; w < kFullWords; w += kFinThreads)
        reinterpret_cast<uint32_t*>(&S)[w] = __ldg(reinterpret_cast<const uint32_t*>(samples + b) + w);
    pdl_wait();                                           // the column kernel's partial rows
    {
        double s[kAccN];
#pragma unroll
        for (int i = 0; i < kAccN; ++i) s[i] = 0.0;
        const float* base = partials + (size_t)b * items_per_sample * kRow;
        for (int j = t; j < items_per_sample; j += kFinThreads) {
            // items the plan kernel proved empty were never processed: they have no row (and contribute nothing)
            if (item_class && item_class[(size_t)b * items_per_sample + j] == kClasses - 1) continue;
            const float4* p = reinterpret_cast<const float4*>(base + (size_t)j * kRow);      // rows are 80 bytes: 16-aligned
            float v[kRow];
#pragma unroll
            for (int i = 0; i < kRow / 4; ++i) { const float4 q = __ldcg(p + i); v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w; }
#pragma unroll
            for (int i = 0; i < kAccN - 1; ++i) s[i] += (double)v[i];
            s[17] += (double)v[17] + (double)v[18] * (double)v[19];      // loss: centred terms + constant x count (implicit_kernel)
        }
#pragma unroll
        for (int i = 0; i < kAccN; ++i) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s[i] += __shfl_xor_sync(0xffffffffu, s[i], o);
            if (lane == 0) wpart[warp][i] = s[i];
        }
    }
    __syncthreads();
    if (t < kAccN) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < kFinThreads / 32; ++w) v += wpart[w][t];
        acc[t] = v;
    }
    __syncthreads();
    const double vol = KIND == FIN_LSQ ? S.a[0] * S.a[1] * S.a[2] : 1.0;
    if (warp == 1) {
        // Loss path, next to the gradient path of warp 0: per-sample loss, then the batch mean by the last block to
        // arrive, in index order.
        unsigned int last = 0u;
        if (lane == 0) {
            const double ls = (acc[17] + (loss_offset ? loss_offset[b] : 0.0)) * loss_norm * vol;   // ImplicitLoss: + sum |target|
            per_sample[b] = ls;
            if (per_sample_user) per_sample_user[b] = ls;
            __threadfence();
            last = atomicAdd(ticket, 1u);
        }
        last = __shfl_sync(0xffffffffu, last, 0);
        if (last == (unsigned)batch - 1u) {
            __threadfence();
            double s = 0.0;
            for (int i = lane; i < batch; i += 32) s += __ldcg(per_sample + i);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0 && loss_out) *loss_out = s / (double)batch;
        }
    } else if (t == 0 && grad) {
        double gr[12];
        finalize_sample(S, g, acc, grad_scale * vol, KIND != FIN_LSQ, gr, KIND == FIN_OCC_VJP ? (double)plane_of_t(S, g) : 0.0);
        if (KIND == FIN_LSQ)
            for (int i = 0; i < 3; ++i) gr[i] += S.mask[i] * (vol * S.ia[i]) * acc[17] * (0.5 * grad_scale);   // d (a1 a2 a3) / d a_i
        if (S.heads) heads_backward(S.hp, S.hrn, S.q, gr);
        for (int i = 0; i < 12; ++i) {
            if (dtype == SQ_F64) static_cast<double*>(grad)[12 * (size_t)b + i] = gr[i];
            else static_cast<float*>(grad)[12 * (size_t)b + i] = (float)gr[i];
        }
    }
}

// ------------------------------------------------------------------------------------------------ field
__global__ void __launch_bounds__(256)
field_kernel(const SampleFull* __restrict__ samples, Grid g, int batch, int mode, float kl, float* __restrict__ out) {
    const size_t n = g.n, per = n * n * n;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= per * batch) return;
    const int b = (int)(idx / per);
    size_t r = idx - (size_t)b * per;
    const int ia = (int)(r / (n * n)); r -= (size_t)ia * n * n;
    const int ib = (int)(r / n), ic = (int)(r - (size_t)ib * n);
    const Sample& S = samples[b];
    const double dx = grid_coord(g, ia) - S.t[0], dy = grid_coord(g, ib) - S.t[1], dz = grid_coord(g, ic) - S.t[2];
    float s[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) s[i] = (float)(S.Ms[3 * i] * dx + S.Ms[3 * i + 1] * dy + S.Ms[3 * i + 2] * dz);
    Fwd f;
    float v;
    if (mode == 0) { point_forward<false>(S, s[0], s[1], s[2], f); v = f.F; }
    else { point_forward<true>(S, s[0], s[1], s[2], f); float x, eo; v = occupancy(f.F, kl, x, eo); }
    out[idx] = v;
}

// ------------------------------------------------------------------------------------------------ host-image gather
// Nearest-neighbour sampling of depth images that live in PINNED HOST memory, read directly over PCIe (zero copy):
// only the sectors that hold sampled pixels cross the bus, instead of the whole images.  PIX = float, or unsigned char for
// 8-bit depth images (the reference's data are 8-bit BMPs divided by 255, torch/test.py:29-30, classes.py:82-88): a quarter
// of the bytes again; the division happens here (scale = 1/255).
template <typename PIX>
__global__ void __launch_bounds__(256)
gather_targets_kernel(const PIX* __restrict__ host_images, long long stride_b, const int* __restrict__ row_off,
                      const int* __restrict__ col_off, int R, int batch, float scale, float* __restrict__ out) {
    const size_t total = (size_t)batch * R * R;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int col = (int)(i % R);
        const size_t t = i / R;
        const int row = (int)(t % R);
        const size_t b = t / R;
        out[i] = (float)host_images[b * (size_t)stride_b + row_off[row] + col_off[col]] * scale;
    }
}

// The same for the regular case (source width a multiple of the render size, rows 16-byte aligned): every thread pulls 16
// contiguous bytes of a sampled row -- a warp 512 contiguous bytes -- so the reads arrive at the host as a few large PCIe
// requests instead of many sector-sized ones (what limits eight GPUs reading from one host), and picks the sampled
// pixels (every sx-th) out of them.
template <typename PIX>
__global__ void __launch_bounds__(256)
gather_rows_kernel(const PIX* __restrict__ host_images, long long stride_b, const int* __restrict__ row_off, int R, int W,
                   int sx, int batch, float scale, float* __restrict__ out) {
    constexpr int PER = 16 / (int)sizeof(PIX);              // pixels per 16-byte load
    const int segs = W / PER;
    const size_t total = (size_t)batch * R * segs;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int seg = (int)(i % segs);
        const size_t t = i / segs;
        const int row = (int)(t % R);
        const size_t b = t / R;
        const int c0 = seg * PER, first = (c0 + sx - 1) / sx * sx;      // first sampled source column at or after c0
        if (first >= c0 + PER) continue;                                 // no sampled pixel in this segment
        const uint4 v = *reinterpret_cast<const uint4*>(host_images + b * (size_t)stride_b + row_off[row] + c0);
        const PIX* px = reinterpret_cast<const PIX*>(&v);
        float* dst = out + (b * R + row) * (size_t)R;
#pragma unroll
        for (int k = 0; k < PER; ++k)
            if (c0 + k >= first && (c0 + k - first) % sx == 0) dst[(c0 + k) / sx] = (float)px[k] * scale;
    }
}

// ------------------------------------------------------------------------------------------------ host helpers
#define SQ_TRY(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return (int)e_; } while (0)

// One-shot event pair around the next column kernel launched by this thread (sq_profile_events()).
thread_local cudaEvent_t t_ev_before = nullptr, t_ev_after = nullptr;

struct ColumnKernelTimer {
    cudaStream_t st; cudaEvent_t after;
    explicit ColumnKernelTimer(cudaStream_t s) : st(s), after(t_ev_after) {
        if (t_ev_before) cudaEventRecord(t_ev_before, st);
        t_ev_before = nullptr; t_ev_after = nullptr;
    }
    ~ColumnKernelTimer() { if (after) cudaEventRecord(after, st); }
};

int check_scratch(int batch, int n, void* scratch, size_t bytes, Scratch* s) {
    if (batch <= 0 || n <= 0) return (int)cudaErrorInvalidValue;
    const size_t need = scratch_layout(batch, n, nullptr, nullptr);
    if (!scratch || bytes < need) return (int)cudaErrorInvalidValue;
    scratch_layout(batch, n, static_cast<char*>(scratch), s);
    return 0;
}

// kernel launch that may overlap the tail of the preceding kernel in the stream (the kernel must call pdl_wait())
template <typename... KArgs, typename... Args>
cudaError_t launch_dependent(void (*kernel)(KArgs...), int grid, int block, size_t dyn_smem, cudaStream_t st, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)block); cfg.dynamicSmemBytes = dyn_smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

int device_sm_count() {
    static int sms[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (sms[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        sms[dev] = n;
    }
    return sms[dev];
}

// blocks of a persistent column kernel: enough to fill every SM at the kernel's occupancy, no more than the work
int persistent_blocks(int items, int warps_per_block, int min_blocks_per_sm) {
    const int need = (items + warps_per_block - 1) / warps_per_block;
    const int fill = device_sm_count() * min_blocks_per_sm;
    return need < fill ? need : fill;
}

// Static + dynamic shared memory of the fwd+bwd kernels exceed 48 KB: opt in once per kernel and device (not a stream
// operation).  The kernel is a template argument so that every kernel has its own `opted` table (the fwd+bwd kernels
// share one function-pointer type).
template <auto KERNEL>
cudaError_t opt_in_dyn_smem(size_t dyn) {
    static bool opted[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !opted[dev]) {
        const cudaError_t e = cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
        if (e != cudaSuccess) return e;
        opted[dev] = true;
    }
    return cudaSuccess;
}

int launch_prep(const void* params, int dtype, int batch, bool clamp, const Grid& g, SampleFull* out, Control* ctl,
                cudaStream_t st) {
    if (dtype != SQ_F32 && dtype != SQ_F64) return (int)cudaErrorInvalidValue;
    prep_kernel<<<(batch + 3) / 4, 128, 0, st>>>(params, dtype, batch, clamp ? 1 : 0, g, out, ctl);
    return (int)cudaGetLastError();
}

// plan kernel of a column-kernel call: Samples, per-sample counters, cost-class queues
struct PlanTarget { const float* target; long long tstride; const int* row_off; const int* col_off; };

int launch_plan(const void* params_a, const void* params_b, int dtype, int batch, bool clamp, const Grid& g,
                const Layout& L, float bound, const Scratch& s, unsigned long long* counts, unsigned char* item_class,
                const PlanTarget* pt, cudaStream_t st, bool heads = false, float die = 0.f) {
    if (dtype != SQ_F32 && dtype != SQ_F64) return (int)cudaErrorInvalidValue;
    int* queue = L.rows_per_sample <= kPlanMaxItems ? s.queue : nullptr;
    const PlanTarget none{nullptr, 0, nullptr, nullptr};
    const PlanTarget& t = pt ? *pt : none;
    const bool small = batch > 4 * device_sm_count();      // more samples than one wave of the large blocks
    if (params_b) {
        auto k = small ? plan_kernel<2, kPlanThreadsSmall> : plan_kernel<2, kPlanThreads>;
        k<<<batch, small ? kPlanThreadsSmall : kPlanThreads, 0, st>>>(params_a, params_b, dtype, clamp ? 1 : 0, 0, g, L, bound, 0.f, s.tru, s.pred,
                                                                      s.ctl, counts, queue, s.queue_cap, queue ? item_class : nullptr,
                                                                      nullptr, 0, nullptr, nullptr, nullptr);
    } else {
        auto k = small ? plan_kernel<1, kPlanThreadsSmall> : plan_kernel<1, kPlanThreads>;
        k<<<batch, small ? kPlanThreadsSmall : kPlanThreads, 0, st>>>(params_a, nullptr, dtype, clamp ? 1 : 0, heads ? 1 : 0, g, L, bound, die, s.pred,
                                                                      nullptr, s.ctl, counts, queue, s.queue_cap, queue ? item_class : nullptr,
                                                                      t.target, t.tstride, t.row_off, t.col_off, pt ? s.tv_sum : nullptr);
    }
    return (int)cudaGetLastError();
}

}  // namespace

// ================================================================================================ C ABI
extern "C" {

const char* sq_version(void) { return "sqloss-b200 0.1 (sm_100a)"; }

const char* sq_error_string(int err) { return cudaGetErrorString((cudaError_t)err); }

int sq_device_sm_count(int device, int* sm_count) {
    return (int)cudaDeviceGetAttribute(sm_count, cudaDevAttrMultiProcessorCount, device);
}

#ifdef SQ_COUNT
int sq_debug_counters(unsigned long long* host_out, int reset) {
    cudaError_t e = cudaMemcpyFromSymbol(host_out, g_count, sizeof(unsigned long long) * 8);
    if (e == cudaSuccess && reset) {
        const unsigned long long zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        e = cudaMemcpyToSymbol(g_count, zero, sizeof zero);
    }
    return (int)e;
}
#endif

#ifdef SQ_ITEMLOG
int sq_debug_itemlog(float* plan_out, int* item_out, int n) {
    int rc = (int)cudaMemcpyFromSymbol(plan_out, g_planlog, sizeof(float) * 4 * (size_t)n);
    if (!rc) rc = (int)cudaMemcpyFromSymbol(item_out, g_itemlog, sizeof(int) * 4 * (size_t)n);
    return rc;
}
#endif
#ifdef SQ_PHASES
int sq_debug_phases(unsigned long long* host_out, int reset) {
    int rc = (int)cudaMemcpyFromSymbol(host_out, g_phase, sizeof(unsigned long long) * 8);
    if (!rc && reset) { unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0}; rc = (int)cudaMemcpyToSymbol(g_phase, z, sizeof z); }
    return rc;
}
#endif
#ifdef SQ_TIMELINE
int sq_debug_timeline(unsigned long long* host_out, int n) {
    return (int)cudaMemcpyFromSymbol(host_out, g_timeline, sizeof(unsigned long long) * 3 * (size_t)n);
}
int sq_debug_bwd(unsigned long long* host_out) {
    return (int)cudaMemcpyFromSymbol(host_out, g_bwd_stats, sizeof(unsigned long long) * 2);
}
int sq_debug_plan(unsigned long long* host_out) {
    return (int)cudaMemcpyFromSymbol(host_out, g_plan_ts, sizeof(unsigned long long) * 16);
}
int sq_debug_classes(unsigned int* host_out) {
    return (int)cudaMemcpyFromSymbol(host_out, g_classes, sizeof(unsigned int) * kClasses);
}
#endif

void sq_profile_events(void* ev_before, void* ev_after) {
    t_ev_before = static_cast<cudaEvent_t>(ev_before);
    t_ev_after = static_cast<cudaEvent_t>(ev_after);
}

size_t sq_scratch_bytes(int batch, int n) {
    if (batch <= 0 || n <= 0) return 0;
    return scratch_layout(batch, n, nullptr, nullptr);
}

int sq_scratch_init(void* scratch, size_t scratch_bytes, sq_stream_t stream) {
    if (!scratch || scratch_bytes < sizeof(Control)) return (int)cudaErrorInvalidValue;
    return (int)cudaMemsetAsync(scratch, 0, sizeof(Control), static_cast<cudaStream_t>(stream));
}

static int implicit_loss_impl(const void* pred, int pred_dtype, int batch, int n, double step, double z0,
                              const float* target, long long target_stride_b, const int* row_off, const int* col_off,
                              float tau, float sharpness, double* loss_out, double* per_sample, void* grad_pred,
                              float* depth_out, void* scratch, size_t scratch_bytes, sq_stream_t stream, bool heads) {
    Scratch s;
    int rc = check_scratch(batch, n, scratch, scratch_bytes, &s);
    if (rc) return rc;
    if (target && (!row_off || !col_off)) return (int)cudaErrorInvalidValue;
    if (grad_pred && !target) return (int)cudaErrorInvalidValue;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Grid g = make_grid(n, step, z0);
    const Layout L = make_layout(n, grad_pred ? SQ_IMPB_CPT : SQ_IMPF_CPT);
    const ImplicitParams P{sharpness * kLog2e, tau * kLog2e, implicit_cull_bound(sharpness * kLog2e), implicit_active_bits(sharpness * kLog2e, n, batch)};
    if (depth_out)      // the column kernel writes the depth only where a column group can hold occupancy
        SQ_TRY(cudaMemsetAsync(depth_out, 0, sizeof(float) * (size_t)batch * n * n, st));
#ifdef SQ_SKIP_COLUMN      // timing experiment: without the column kernel nobody restores the control block
    SQ_TRY(cudaMemsetAsync(s.ctl, 0, sizeof(Control), st));
#endif
    const PlanTarget pt{target, target_stride_b, row_off, col_off};
    rc = launch_plan(pred, nullptr, pred_dtype, batch, true, g, L, P.bound, s, nullptr, target ? s.item_class : nullptr,
                     target ? &pt : nullptr, st, heads, SQ_WALK_ESTIMATE ? 32.0f / P.tl : 0.f);
    if (rc) return rc;
    const int items = batch * L.rows_per_sample;
    const int* queue = L.rows_per_sample <= kPlanMaxItems ? s.queue : nullptr;
#ifdef SQ_PDL
    const bool pdl = (t_ev_before == nullptr && t_ev_after == nullptr);   // an event record in between breaks the chain
#else
    const bool pdl = false;
#endif
#ifndef SQ_SKIP_COLUMN      // timing experiments only (tools/tune.py): leave out the column and / or finalize kernel
    {
        ColumnKernelTimer timer(st);
        if (grad_pred) {
            const int blocks = persistent_blocks(items, SQ_IMPB_THREADS / 32, SQ_IMPB_MINB);
            constexpr size_t dyn = kImplicitBwdSmemPerWarp * (SQ_IMPB_THREADS / 32);
            SQ_TRY((opt_in_dyn_smem<implicit_kernel<true, SQ_IMPB_THREADS, SQ_IMPB_MINB, SQ_IMPB_CPT>>(dyn)));
            SQ_TRY(launch_dependent(implicit_kernel<true, SQ_IMPB_THREADS, SQ_IMPB_MINB, SQ_IMPB_CPT>, blocks, SQ_IMPB_THREADS, dyn, st, pdl,
                                    s.pred, g, L, P, items, s.ctl, queue, s.queue_cap, target, target_stride_b, row_off, col_off,
                                    s.partials, depth_out));
        } else {
            const int blocks = persistent_blocks(items, SQ_IMPF_THREADS / 32, SQ_IMPF_MINB);
            SQ_TRY(launch_dependent(implicit_kernel<false, SQ_IMPF_THREADS, SQ_IMPF_MINB, SQ_IMPF_CPT>, blocks, SQ_IMPF_THREADS, 0, st, pdl,
                                    s.pred, g, L, P, items, s.ctl, queue, s.queue_cap, target, target_stride_b, row_off, col_off,
                                    s.partials, depth_out));
        }
    }
    SQ_TRY(cudaGetLastError());
#endif
#ifndef SQ_SKIP_FINALIZE
    if (target) {
        const double nn = (double)n * n;
        SQ_TRY(launch_dependent(finalize_kernel<FIN_IMPLICIT>, batch, kFinThreads, 0, st, pdl,
                                s.pred, g, batch, L.rows_per_sample, s.partials, 1.0 / nn,
                                -(double)sharpness * (double)tau / (nn * n * (double)batch), pred_dtype, grad_pred, s.per_sample,
                                per_sample, loss_out, &s.ctl->ticket, s.tv_sum, queue ? s.item_class : nullptr));
        SQ_TRY(cudaGetLastError());
    }
#endif
    return 0;
}

int sq_implicit_loss(const void* pred, int pred_dtype, int batch, int n, double step, double z0,
                     const float* target, long long target_stride_b, const int* row_off, const int* col_off,
                     float tau, float sharpness, double* loss_out, double* per_sample, void* grad_pred,
                     float* depth_out, void* scratch, size_t scratch_bytes, sq_stream_t stream) {
    return implicit_loss_impl(pred, pred_dtype, batch, n, step, z0, target, target_stride_b, row_off, col_off, tau, sharpness,
                              loss_out, per_sample, grad_pred, depth_out, scratch, scratch_bytes, stream, false);
}

int sq_implicit_loss_heads(const void* raw_heads, int dtype, int batch, int n, double step, double z0,
                           const float* target, long long target_stride_b, const int* row_off, const int* col_off,
                           float tau, float sharpness, double* loss_out, double* per_sample, void* grad_raw,
                           float* depth_out, void* scratch, size_t scratch_bytes, sq_stream_t stream) {
    return implicit_loss_impl(raw_heads, dtype, batch, n, step, z0, target, target_stride_b, row_off, col_off, tau, sharpness,
                              loss_out, per_sample, grad_raw, depth_out, scratch, scratch_bytes, stream, true);
}

// The fwd+bwd pipeline with the upstream pixel as the column weight (implicit_kernel VJP mode): plan (no pixel sum; the
// item classes still let finalize skip proven-empty items, whose columns carry no weight above the cut for any upstream),
// column kernel, finalize with the scale of d depth / d theta alone.  Nothing is read that an earlier call left behind.
int sq_depth_projection_vjp(const void* pred, int pred_dtype, int batch, int n, double step, double z0,
                            float tau, float sharpness, const float* grad_depth, void* grad_pred,
                            void* scratch, size_t scratch_bytes, sq_stream_t stream) {
    Scratch s;
    int rc = check_scratch(batch, n, scratch, scratch_bytes, &s);
    if (rc) return rc;
    if (!grad_depth || !grad_pred) return (int)cudaErrorInvalidValue;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Grid g = make_grid(n, step, z0);
    const Layout L = make_layout(n, SQ_IMPB_CPT);
    // the weight cut of one sample (batch 1): a VJP's gradient of sample b does not depend on the batch
    const ImplicitParams P{sharpness * kLog2e, tau * kLog2e, implicit_cull_bound(sharpness * kLog2e), implicit_active_bits(sharpness * kLog2e, n, 1)};
    rc = launch_plan(pred, nullptr, pred_dtype, batch, true, g, L, P.bound, s, nullptr, s.item_class, nullptr, st, false,
                     SQ_WALK_ESTIMATE ? 32.0f / P.tl : 0.f);
    if (rc) return rc;
    const int items = batch * L.rows_per_sample;
    const int* queue = L.rows_per_sample <= kPlanMaxItems ? s.queue : nullptr;
#ifdef SQ_PDL
    const bool pdl = (t_ev_before == nullptr && t_ev_after == nullptr);
#else
    const bool pdl = false;
#endif
    {
        ColumnKernelTimer timer(st);
        const int blocks = persistent_blocks(items, SQ_IMPB_THREADS / 32, SQ_IMPB_MINB);
        constexpr size_t dyn = kImplicitBwdSmemPerWarp * (SQ_IMPB_THREADS / 32);
        SQ_TRY((opt_in_dyn_smem<implicit_kernel<true, SQ_IMPB_THREADS, SQ_IMPB_MINB, SQ_IMPB_CPT, true>>(dyn)));
        SQ_TRY(launch_dependent(implicit_kernel<true, SQ_IMPB_THREADS, SQ_IMPB_MINB, SQ_IMPB_CPT, true>, blocks, SQ_IMPB_THREADS, dyn,
                                st, pdl, s.pred, g, L, P, items, s.ctl, queue, s.queue_cap, grad_depth, 0LL,
                                static_cast<const int*>(nullptr), static_cast<const int*>(nullptr), s.partials,
                                static_cast<float*>(nullptr)));
    }
    SQ_TRY(cudaGetLastError());
    // d depth / d o_c = (tau / n) S_c and d o / d F = -k o (1 - o): the column sums carry o (1 - o) S_c x upstream
    SQ_TRY(launch_dependent(finalize_kernel<FIN_IMPLICIT>, batch, kFinThreads, 0, st, pdl,
                            s.pred, g, batch, L.rows_per_sample, s.partials, 0.0, -(double)sharpness * (double)tau / (double)n,
                            pred_dtype, grad_pred, s.per_sample, static_cast<double*>(nullptr), static_cast<double*>(nullptr),
                            &s.ctl->ticket, static_cast<const double*>(nullptr), queue ? s.item_class : nullptr));
    SQ_TRY(cudaGetLastError());
    return 0;
}

int sq_explicit_loss(const void* true_params, const void* pred, int params_dtype, int batch, int n, double step,
                     double z0, float sharpness, float mult, double* loss_out, double* per_sample, void* grad_pred,
                     void* scratch, size_t scratch_bytes, sq_stream_t stream) {
    Scratch s;
    int rc = check_scratch(batch, n, scratch, scratch_bytes, &s);
    if (rc) return rc;
    if (!true_params || !pred) return (int)cudaErrorInvalidValue;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Grid g = make_grid(n, step, z0);
    const Layout L = make_layout(n, SQ_EXP_CPT);
    const float kl = sharpness * kLog2e, bound = cull_bound_bits(kl, 24.0f);
    rc = launch_plan(true_params, pred, params_dtype, batch, true, g, L, bound, s, nullptr, s.item_class, nullptr, st);
    if (rc) return rc;
    const int items = batch * L.rows_per_sample;
    const int* queue = L.rows_per_sample <= kPlanMaxItems ? s.queue : nullptr;
    const int blocks = persistent_blocks(items, SQ_EXP_THREADS / 32, SQ_EXP_MINB);
    {
        ColumnKernelTimer timer(st);
        if (grad_pred) explicit_kernel<true><<<blocks, SQ_EXP_THREADS, 0, st>>>(s.tru, s.pred, g, L, kl, bound, items, s.ctl, queue, s.queue_cap, s.partials);
        else explicit_kernel<false><<<blocks, SQ_EXP_THREADS, 0, st>>>(s.tru, s.pred, g, L, kl, bound, items, s.ctl, queue, s.queue_cap, s.partials);
    }
    SQ_TRY(cudaGetLastError());
    const double n3 = (double)n * n * n;
    finalize_kernel<FIN_EXPLICIT><<<batch, kFinThreads, 0, st>>>(
        s.pred, g, batch, L.rows_per_sample, s.partials, (double)mult / n3,
        2.0 * (double)sharpness * (double)mult / (n3 * (double)batch), params_dtype, grad_pred, s.per_sample,
        per_sample, loss_out, &s.ctl->ticket, nullptr, queue ? s.item_class : nullptr);
    SQ_TRY(cudaGetLastError());
    return 0;
}

// plan (the predicted SQ alone, clamped, culled at the VJP's cut: proven-empty items carry no weight above the cut for any
// upstream), the VJP column kernel, finalize with the scale of d o / d F = -k o (1 - o) alone.  Nothing is read that an
// earlier call left behind.
int sq_occupancy_vjp(const void* params, int params_dtype, int batch, int n, double step, double z0,
                     float sharpness, const float* grad_field, void* grad_params,
                     void* scratch, size_t scratch_bytes, sq_stream_t stream) {
    Scratch s;
    int rc = check_scratch(batch, n, scratch, scratch_bytes, &s);
    if (rc) return rc;
    if (!params || !grad_field || !grad_params) return (int)cudaErrorInvalidValue;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Grid g = make_grid(n, step, z0);
    const Layout L = make_layout(n, SQ_EXP_CPT);
    const float kl = sharpness * kLog2e, kact = kExplicitVjpBits, bound = cull_bound_bits(kl, kact);
    rc = launch_plan(params, nullptr, params_dtype, batch, true, g, L, bound, s, nullptr, s.item_class, nullptr, st);
    if (rc) return rc;
    const int items = batch * L.rows_per_sample;
    const int* queue = L.rows_per_sample <= kPlanMaxItems ? s.queue : nullptr;
    const int blocks = persistent_blocks(items, SQ_EXP_THREADS / 32, SQ_EXP_MINB);
    {
        ColumnKernelTimer timer(st);
        explicit_vjp_kernel<<<blocks, SQ_EXP_THREADS, 0, st>>>(s.pred, g, L, kl, bound, kact, grad_field, items, s.ctl, queue,
                                                               s.queue_cap, s.partials);
    }
    SQ_TRY(cudaGetLastError());
    finalize_kernel<FIN_OCC_VJP><<<batch, kFinThreads, 0, st>>>(
        s.pred, g, batch, L.rows_per_sample, s.partials, 0.0, -(double)sharpness, params_dtype, grad_params, s.per_sample,
        nullptr, nullptr, &s.ctl->ticket, nullptr, queue ? s.item_class : nullptr);
    SQ_TRY(cudaGetLastError());
    return 0;
}

// plan (the predicted SQ alone, culled at the VJP's cut), the voxel column kernel, finalize with sq_explicit_loss's scales
// and the VJP's z centre.  Finalize reads every item's row: the column kernel writes one for proven-empty items too.
int sq_voxel_loss(const void* voxels, int voxel_dtype, float voxel_scale,
                  const void* pred, int params_dtype, int batch, int n, double step, double z0,
                  float sharpness, float mult, double* loss_out, double* per_sample, void* grad_pred,
                  void* scratch, size_t scratch_bytes, sq_stream_t stream) {
    Scratch s;
    int rc = check_scratch(batch, n, scratch, scratch_bytes, &s);
    if (rc) return rc;
    if (!voxels || !pred || (voxel_dtype != SQ_F32 && voxel_dtype != SQ_U8)) return (int)cudaErrorInvalidValue;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Grid g = make_grid(n, step, z0);
    const Layout L = make_layout(n, SQ_EXP_CPT);
    const float kl = sharpness * kLog2e, kact = kExplicitVjpBits, bound = cull_bound_bits(kl, kact);
    rc = launch_plan(pred, nullptr, params_dtype, batch, true, g, L, bound, s, nullptr, s.item_class, nullptr, st);
    if (rc) return rc;
    const int items = batch * L.rows_per_sample;
    const int* queue = L.rows_per_sample <= kPlanMaxItems ? s.queue : nullptr;
    const int blocks = persistent_blocks(items, SQ_EXP_THREADS / 32, SQ_EXP_MINB);
    {
        ColumnKernelTimer timer(st);
        const float* vf = static_cast<const float*>(voxels);
        const uint8_t* vb = static_cast<const uint8_t*>(voxels);
        if (voxel_dtype == SQ_U8) {
            if (grad_pred) explicit_vox_kernel<true, uint8_t><<<blocks, SQ_EXP_THREADS, 0, st>>>(
                s.pred, g, L, kl, bound, kact, vb, voxel_scale, items, s.ctl, queue, s.queue_cap, s.partials);
            else explicit_vox_kernel<false, uint8_t><<<blocks, SQ_EXP_THREADS, 0, st>>>(
                s.pred, g, L, kl, bound, kact, vb, voxel_scale, items, s.ctl, queue, s.queue_cap, s.partials);
        } else {
            if (grad_pred) explicit_vox_kernel<true, float><<<blocks, SQ_EXP_THREADS, 0, st>>>(
                s.pred, g, L, kl, bound, kact, vf, voxel_scale, items, s.ctl, queue, s.queue_cap, s.partials);
            else explicit_vox_kernel<false, float><<<blocks, SQ_EXP_THREADS, 0, st>>>(
                s.pred, g, L, kl, bound, kact, vf, voxel_scale, items, s.ctl, queue, s.queue_cap, s.partials);
        }
    }
    SQ_TRY(cudaGetLastError());
    const double n3 = (double)n * n * n;
    finalize_kernel<FIN_OCC_VJP><<<batch, kFinThreads, 0, st>>>(
        s.pred, g, batch, L.rows_per_sample, s.partials, (double)mult / n3,
        2.0 * (double)sharpness * (double)mult / (n3 * (double)batch), params_dtype, grad_pred, s.per_sample,
        per_sample, loss_out, &s.ctl->ticket, nullptr, nullptr);
    SQ_TRY(cudaGetLastError());
    return 0;
}

int sq_iou_counts(const void* true_params, const void* pred, int params_dtype, int batch, int n, double step,
                  double z0, long long* inter, long long* uni, void* scratch, size_t scratch_bytes,
                  sq_stream_t stream) {
    Scratch s;
    int rc = check_scratch(batch, n, scratch, scratch_bytes, &s);
    if (rc) return rc;
    if (!true_params || !pred || !inter || !uni) return (int)cudaErrorInvalidValue;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Grid g = make_grid(n, step, z0);
    const Layout L = make_layout(n, SQ_IOU_CPT);
    rc = launch_plan(true_params, pred, params_dtype, batch, false, g, L, kIoUBound, s, s.counts, nullptr, nullptr, st);
    if (rc) return rc;
    const int items = batch * L.rows_per_sample;
    const int* queue = L.rows_per_sample <= kPlanMaxItems ? s.queue : nullptr;
    const int blocks = persistent_blocks(items, SQ_IOU_THREADS / 32, SQ_IOU_MINB);
    {
        ColumnKernelTimer timer(st);
        iou_kernel<<<blocks, SQ_IOU_THREADS, 0, st>>>(s.tru, s.pred, g, L, items, s.ctl, queue, s.queue_cap, s.counts);
    }
    SQ_TRY(cudaGetLastError());
    iou_export_kernel<<<(batch + 127) / 128, 128, 0, st>>>(s.counts, batch, inter, uni);
    SQ_TRY(cudaGetLastError());
    return 0;
}

int sq_least_squares(const void* pred, int pred_dtype, int batch, int render_size, const float* target,
                     long long target_stride_b, const int* row_off, const int* col_off, double* loss_out,
                     double* per_sample, void* grad_pred, void* scratch, size_t scratch_bytes, sq_stream_t stream) {
    Scratch s;
    int rc = check_scratch(batch, render_size, scratch, scratch_bytes, &s);
    if (rc) return rc;
    if (!target || !row_off || !col_off) return (int)cudaErrorInvalidValue;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Grid g = make_grid(2, 1.0, 0.0);     // the point list carries its own coordinates; the grid is unused
    rc = launch_prep(pred, pred_dtype, batch, true, g, s.pred, s.ctl, st);
    if (rc) return rc;
    const int R = render_size;
    const int ips = (R * R + kThreads * kLsqPix - 1) / (kThreads * kLsqPix);
    if (grad_pred) lsq_kernel<true><<<batch * ips, kThreads, 0, st>>>(s.pred, R, ips, target, target_stride_b, row_off, col_off, s.partials);
    else lsq_kernel<false><<<batch * ips, kThreads, 0, st>>>(s.pred, R, ips, target, target_stride_b, row_off, col_off, s.partials);
    SQ_TRY(cudaGetLastError());
    finalize_kernel<FIN_LSQ><<<batch, kFinThreads, 0, st>>>(s.pred, g, batch, ips, s.partials, 1.0, 2.0 / (double)batch,
                                                   pred_dtype, grad_pred, s.per_sample, per_sample, loss_out, &s.ctl->ticket,
                                                   nullptr, nullptr);
    SQ_TRY(cudaGetLastError());
    return 0;
}

int sq_least_squares_points(const void* pred, int pred_dtype, int batch, const float* points, long long stride,
                            const long long* offsets, long long max_points, double* loss_out, double* per_sample,
                            void* grad_pred, void* scratch, size_t scratch_bytes, sq_stream_t stream) {
    if (!points || !offsets || max_points < 0 || stride < 0 || (stride & 3)) return (int)cudaErrorInvalidValue;
    // scratch rows: one per chunk of kThreads * 4 points; sq_scratch_bytes(batch, n) provides for n * n points per sample
    const long long chunks64 = (max_points + 3 + kThreads * 4 - 1) / (kThreads * 4);
    const int chunks = chunks64 > 0 ? (int)chunks64 : 1;
    int n = 1;
    while ((long long)n * n < (long long)chunks * kThreads) ++n;
    Scratch s;
    int rc = check_scratch(batch, n, scratch, scratch_bytes, &s);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Grid g = make_grid(2, 1.0, 0.0);
    rc = launch_prep(pred, pred_dtype, batch, true, g, s.pred, s.ctl, st);
    if (rc) return rc;
    if (grad_pred) lsq_points_kernel<true><<<batch * chunks, kThreads, 0, st>>>(s.pred, chunks, points, stride, offsets, s.partials);
    else lsq_points_kernel<false><<<batch * chunks, kThreads, 0, st>>>(s.pred, chunks, points, stride, offsets, s.partials);
    SQ_TRY(cudaGetLastError());
    // per-sample energies: the gradient is d per_sample[b] / d pred[b] (no 1 / batch)
    finalize_kernel<FIN_LSQ><<<batch, kFinThreads, 0, st>>>(s.pred, g, batch, chunks, s.partials, 1.0, 2.0, pred_dtype, grad_pred,
                                                   s.per_sample, per_sample, loss_out, &s.ctl->ticket, nullptr, nullptr);
    SQ_TRY(cudaGetLastError());
    return 0;
}

size_t sq_points_scratch_bytes(int batch, long long max_points) {
    if (batch <= 0 || max_points < 0) return 0;
    const long long chunks64 = (max_points + 3 + kThreads * 4 - 1) / (kThreads * 4);
    const int chunks = chunks64 > 0 ? (int)chunks64 : 1;
    int n = 1;
    while ((long long)n * n < (long long)chunks * kThreads) ++n;
    return scratch_layout(batch, n, nullptr, nullptr);
}

int sq_field(const void* params, int params_dtype, int batch, int n, double step, double z0, int mode,
             float sharpness, float* out, void* scratch, size_t scratch_bytes, sq_stream_t stream) {
    Scratch s;
    int rc = check_scratch(batch, n, scratch, scratch_bytes, &s);
    if (rc) return rc;
    if (!out || (mode != 0 && mode != 1)) return (int)cudaErrorInvalidValue;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Grid g = make_grid(n, step, z0);
    rc = launch_prep(params, params_dtype, batch, mode == 1, g, s.pred, nullptr, st);
    if (rc) return rc;
    const size_t total = (size_t)batch * n * n * n;
    field_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(s.pred, g, batch, mode, sharpness * kLog2e, out);
    SQ_TRY(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------ host-buffer API
// An sq_ctx owns kSlots independent slots on one device; a slot = a stream, a device arena (carved per call; the scratch,
// whose Control block is zeroed when the arena is allocated, always sits at its start) and pinned staging.  The blocking
// calls use slot 0.  sq_implicit_loss_host_submit / _wait expose the slots: while slot A's kernels run, slot B's inputs
// cross PCIe.
constexpr int kSlots = SQ_HOST_SLOTS;
struct sq_slot {
    cudaStream_t stream;
    char* dev; size_t dev_bytes;
    char* pin; size_t pin_bytes;
    size_t out_off, out_bytes;           // where the pending call's results sit in `pin`
    const int* tab_dev; int tab_r, tab_h, tab_w;    // the resize offset tables now on the device (sq_implicit_loss_host_submit)
    int pending_batch; bool pending, pending_grad;
};
struct sq_ctx {
    int device;
    sq_slot slot[kSlots];
};

static int slot_reserve(sq_slot* c, size_t dev_bytes, size_t pin_bytes) {
    if (dev_bytes > c->dev_bytes) {
        if (c->dev) { SQ_TRY(cudaStreamSynchronize(c->stream)); SQ_TRY(cudaFree(c->dev)); }
        c->dev = nullptr; c->dev_bytes = 0; c->tab_dev = nullptr;
        SQ_TRY(cudaMalloc(&c->dev, dev_bytes));
        c->dev_bytes = dev_bytes;
        SQ_TRY(cudaMemsetAsync(c->dev, 0, sizeof(Control), c->stream));
    }
    if (pin_bytes > c->pin_bytes) {
        if (c->pin) { SQ_TRY(cudaStreamSynchronize(c->stream)); SQ_TRY(cudaFreeHost(c->pin)); }
        c->pin = nullptr; c->pin_bytes = 0;
        SQ_TRY(cudaMallocHost(&c->pin, pin_bytes));
        c->pin_bytes = pin_bytes;
    }
    return 0;
}

int sq_ctx_create(int device, sq_ctx** out) {
    if (!out) return (int)cudaErrorInvalidValue;
    SQ_TRY(cudaSetDevice(device));
    sq_ctx* c = new (std::nothrow) sq_ctx();
    if (!c) return (int)cudaErrorMemoryAllocation;
    c->device = device;
    for (int i = 0; i < kSlots; ++i) {
        sq_slot& sl = c->slot[i];
        sl.stream = nullptr; sl.dev = nullptr; sl.dev_bytes = 0; sl.pin = nullptr; sl.pin_bytes = 0;
        sl.out_off = sl.out_bytes = 0; sl.pending_batch = 0; sl.pending = sl.pending_grad = false;
        sl.tab_dev = nullptr; sl.tab_r = sl.tab_h = sl.tab_w = 0;
    }
    for (int i = 0; i < kSlots; ++i) {
        cudaError_t e = cudaStreamCreateWithFlags(&c->slot[i].stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            for (int j = 0; j < i; ++j) cudaStreamDestroy(c->slot[j].stream);
            delete c;
            return (int)e;
        }
    }
    *out = c;
    return 0;
}

void sq_ctx_destroy(sq_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    for (int i = 0; i < kSlots; ++i) {
        sq_slot& sl = c->slot[i];
        if (sl.stream) cudaStreamSynchronize(sl.stream);
        if (sl.dev) cudaFree(sl.dev);
        if (sl.pin) cudaFreeHost(sl.pin);
        if (sl.stream) cudaStreamDestroy(sl.stream);
    }
    delete c;
}

// F.interpolate(mode="nearest") source index: min(floor(dst * (float)in / out), in - 1)
static void nearest_offsets(int in, int out, int stride, int* off) {
    const float scale = (float)in / (float)out;
    for (int i = 0; i < out; ++i) {
        int s = (int)floorf((float)i * scale);
        if (s > in - 1) s = in - 1;
        off[i] = s * stride;
    }
}

int sq_implicit_loss_host_submit(sq_ctx* ctx, int slot, const float* pred_host, int batch, int render_size,
                                 const void* images_host, int image_dtype, int height, int width, float image_scale,
                                 float tau, float sharpness, int want_grad) {
    if (!ctx || slot < 0 || slot >= kSlots || !pred_host || !images_host || batch <= 0 || render_size <= 0 ||
        height <= 0 || width <= 0 || (image_dtype != SQ_F32 && image_dtype != SQ_U8))
        return (int)cudaErrorInvalidValue;
    SQ_TRY(cudaSetDevice(ctx->device));
    sq_slot* c = &ctx->slot[slot];
    if (c->pending) return (int)cudaErrorNotReady;          // the previous submit on this slot has not been waited for
    const int R = render_size;
    const size_t px = image_dtype == SQ_U8 ? 1 : sizeof(float);
    // How the pixels cross PCIe.  Images in pinned (or registered) host memory:
    //   kRowsDma     the nearest resize picks every (height/R)-th row and every (width/R)-th pixel of it: the rows are one
    //                strided copy-engine transfer (cudaMemcpy2DAsync) -- it runs beside the kernels of the other slot, which a
    //                zero-copy kernel cannot (the persistent column kernel fills every SM's registers, so a gather kernel
    //                waits for it to retire: 139 us -> 8x us per pipelined config-2 step, tools/pcie_probe.cu);
    //   kRowsMapped  irregular rows but regular columns: whole rows read in place with 16-byte loads;
    //   kPixels      anything else: pixel by pixel through the offset tables.
    // Pageable memory is copied whole first and then sampled on the device (kRowsMapped / kPixels on the copy).
    cudaPointerAttributes attr;
    const void* mapped = nullptr;
    if (cudaPointerGetAttributes(&attr, images_host) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer)
        mapped = attr.devicePointer;
    else
        cudaGetLastError();
    const bool regular = width % R == 0 && ((size_t)width * px) % 16 == 0;
    const bool rows_dma = mapped && regular && height % R == 0;
    const bool rows16 = regular && (rows_dma || !mapped || reinterpret_cast<uintptr_t>(mapped) % 16 == 0);
    const size_t b_off = align_up(sizeof(int) * 5 * (size_t)R, 256);
    const size_t b_pred = align_up(sizeof(float) * 12 * (size_t)batch, 256);
    const size_t b_img = align_up(sizeof(float) * (size_t)batch * R * R, 256);                 // the compact [batch, R, R] fp32 target
    const size_t b_raw = rows_dma ? align_up(px * (size_t)batch * R * width, 256)               // the sampled rows
                       : mapped ? 0 : align_up(px * (size_t)batch * height * width, 256);       // pageable images, copied whole
    const size_t b_out = align_up(sizeof(double) + sizeof(float) * 12 * (size_t)batch, 256);
    const size_t b_scr = sq_scratch_bytes(batch, R);
    int rc = slot_reserve(c, align_up(b_scr, 256) + b_off + b_pred + b_img + b_raw + b_out, b_off + b_pred + b_out);
    if (rc) return rc;
    char* d = c->dev;
    void* d_scr = d; d += align_up(b_scr, 256);
    int* d_off = reinterpret_cast<int*>(d); d += b_off;                                         // [off | pred]: one upload
    float* d_pred = reinterpret_cast<float*>(d); d += b_pred;
    float* d_img = reinterpret_cast<float*>(d); d += b_img;
    void* d_raw = d; d += b_raw;
    double* d_loss = reinterpret_cast<double*>(d);
    float* d_grad = reinterpret_cast<float*>(d + sizeof(double)); d += b_out;
    // offset tables (kept on the device while the shape stays the same) and parameters, staged in pinned memory
    int* h_off = reinterpret_cast<int*>(c->pin);
    const bool same_tables = c->tab_dev == d_off && c->tab_r == R && c->tab_h == height && c->tab_w == width;
    if (!same_tables) {
        nearest_offsets(height, R, width, h_off);
        nearest_offsets(width, R, 1, h_off + R);
        for (int i = 0; i < R; ++i) {
            h_off[2 * R + i] = i * R; h_off[3 * R + i] = i;                                     // identity tables of the compact target
            h_off[4 * R + i] = i * width;                                                       // rows of the kRowsDma staging
        }
    }
    memcpy(c->pin + b_off, pred_host, sizeof(float) * 12 * (size_t)batch);
    if (same_tables) {
        SQ_TRY(cudaMemcpyAsync(d_pred, c->pin + b_off, sizeof(float) * 12 * (size_t)batch, cudaMemcpyHostToDevice, c->stream));
    } else {
        SQ_TRY(cudaMemcpyAsync(d_off, c->pin, b_off + sizeof(float) * 12 * (size_t)batch, cudaMemcpyHostToDevice, c->stream));
        c->tab_dev = d_off; c->tab_r = R; c->tab_h = height; c->tab_w = width;
    }
    const void* src = mapped;
    long long stride_b = (long long)height * width;
    const int* rows_off = d_off;
    if (rows_dma) {
        SQ_TRY(cudaMemcpy2DAsync(d_raw, (size_t)width * px, images_host, (size_t)(height / R) * width * px, (size_t)width * px,
                                 (size_t)batch * R, cudaMemcpyHostToDevice, c->stream));
        src = d_raw; stride_b = (long long)R * width; rows_off = d_off + 4 * R;
    } else if (!mapped) {
        SQ_TRY(cudaMemcpyAsync(d_raw, images_host, px * (size_t)batch * height * width, cudaMemcpyHostToDevice, c->stream));
        src = d_raw;
    }
    const int gblocks = rows_dma ? 592 : 1184;
    if (rows16 && image_dtype == SQ_U8)
        gather_rows_kernel<unsigned char><<<gblocks, 256, 0, c->stream>>>(static_cast<const unsigned char*>(src), stride_b, rows_off, R,
                                                                         width, width / R, batch, image_scale, d_img);
    else if (rows16)
        gather_rows_kernel<float><<<gblocks, 256, 0, c->stream>>>(static_cast<const float*>(src), stride_b, rows_off, R, width, width / R,
                                                                 batch, image_scale, d_img);
    else if (image_dtype == SQ_U8)
        gather_targets_kernel<unsigned char><<<1184, 256, 0, c->stream>>>(static_cast<const unsigned char*>(src), stride_b, d_off, d_off + R,
                                                                         R, batch, image_scale, d_img);
    else
        gather_targets_kernel<float><<<1184, 256, 0, c->stream>>>(static_cast<const float*>(src), stride_b, d_off, d_off + R, R, batch,
                                                                 image_scale, d_img);
    SQ_TRY(cudaGetLastError());
    rc = sq_implicit_loss(d_pred, SQ_F32, batch, R, 1.0 / (double)(R - 1), 1e-4, d_img, (long long)R * R,
                          d_off + 2 * R, d_off + 3 * R, tau, sharpness, d_loss, nullptr, want_grad ? d_grad : nullptr, nullptr,
                          d_scr, b_scr, c->stream);
    if (rc) return rc;
    c->out_off = b_off + b_pred;
    c->out_bytes = sizeof(double) + (want_grad ? sizeof(float) * 12 * (size_t)batch : 0);
    SQ_TRY(cudaMemcpyAsync(c->pin + c->out_off, d_loss, c->out_bytes, cudaMemcpyDeviceToHost, c->stream));
    c->pending = true; c->pending_grad = want_grad != 0; c->pending_batch = batch;
    return 0;
}

int sq_implicit_loss_host_wait(sq_ctx* ctx, int slot, double* loss_host, float* grad_host) {
    if (!ctx || slot < 0 || slot >= kSlots) return (int)cudaErrorInvalidValue;
    sq_slot* c = &ctx->slot[slot];
    if (!c->pending) return (int)cudaErrorInvalidValue;
    if (grad_host && !c->pending_grad) return (int)cudaErrorInvalidValue;
    SQ_TRY(cudaSetDevice(ctx->device));
    c->pending = false;
    SQ_TRY(cudaStreamSynchronize(c->stream));
    const char* h_out = c->pin + c->out_off;
    if (loss_host) memcpy(loss_host, h_out, sizeof(double));
    if (grad_host) memcpy(grad_host, h_out + sizeof(double), sizeof(float) * 12 * (size_t)c->pending_batch);
    return 0;
}

int sq_implicit_loss_host(sq_ctx* c, const float* pred_host, int batch, int render_size, const float* images_host,
                          int height, int width, float tau, float sharpness, double* loss_host, float* grad_host) {
    int rc = sq_implicit_loss_host_submit(c, 0, pred_host, batch, render_size, images_host, SQ_F32, height, width, 1.0f, tau,
                                          sharpness, grad_host ? 1 : 0);
    if (rc) return rc;
    return sq_implicit_loss_host_wait(c, 0, loss_host, grad_host);
}

int sq_explicit_loss_host(sq_ctx* ctx, const float* true_host, const float* pred_host, int batch, int render_size,
                          double* loss_host, float* grad_host) {
    if (!ctx || !true_host || !pred_host || batch <= 0 || render_size <= 0) return (int)cudaErrorInvalidValue;
    SQ_TRY(cudaSetDevice(ctx->device));
    sq_slot* c = &ctx->slot[0];
    if (c->pending) return (int)cudaErrorNotReady;
    // arange(0, 1 + step, step) of the reference: count the entries the way numpy does (ceil((stop-start)/step))
    const double step = 1.0 / (double)render_size;
    const int n = (int)ceil((1.0 + step) / step);
    const size_t b_par = align_up(sizeof(float) * 12 * (size_t)batch, 256);
    const size_t b_out = align_up(sizeof(double) + sizeof(float) * 12 * (size_t)batch, 256);
    const size_t b_scr = sq_scratch_bytes(batch, n);
    int rc = slot_reserve(c, align_up(b_scr, 256) + 2 * b_par + b_out, b_out);
    if (rc) return rc;
    c->tab_dev = nullptr;                                    // this call's arena layout overwrites the resize tables
    char* d = c->dev;
    void* d_scr = d; d += align_up(b_scr, 256);
    float* d_true = reinterpret_cast<float*>(d); d += b_par;
    float* d_pred = reinterpret_cast<float*>(d); d += b_par;
    double* d_loss = reinterpret_cast<double*>(d);
    float* d_grad = reinterpret_cast<float*>(d + sizeof(double)); d += b_out;
    SQ_TRY(cudaMemcpyAsync(d_true, true_host, sizeof(float) * 12 * (size_t)batch, cudaMemcpyHostToDevice, c->stream));
    SQ_TRY(cudaMemcpyAsync(d_pred, pred_host, sizeof(float) * 12 * (size_t)batch, cudaMemcpyHostToDevice, c->stream));
    rc = sq_explicit_loss(d_true, d_pred, SQ_F32, batch, n, step, 1e-4, 5.0f, 100.0f, d_loss, nullptr,
                          grad_host ? d_grad : nullptr, d_scr, b_scr, c->stream);
    if (rc) return rc;
    const size_t out_bytes = sizeof(double) + (grad_host ? sizeof(float) * 12 * (size_t)batch : 0);
    SQ_TRY(cudaMemcpyAsync(c->pin, d_loss, out_bytes, cudaMemcpyDeviceToHost, c->stream));
    SQ_TRY(cudaStreamSynchronize(c->stream));
    if (loss_host) memcpy(loss_host, c->pin, sizeof(double));
    if (grad_host) memcpy(grad_host, c->pin + sizeof(double), sizeof(float) * 12 * (size_t)batch);
    return 0;
}

int sq_iou_counts_host(sq_ctx* ctx, const float* true_host, const float* pred_host, int batch, int render_size,
                       long long* inter_host, long long* uni_host) {
    if (!ctx || !true_host || !pred_host || !inter_host || !uni_host || batch <= 0 || render_size <= 1)
        return (int)cudaErrorInvalidValue;
    SQ_TRY(cudaSetDevice(ctx->device));
    sq_slot* c = &ctx->slot[0];
    if (c->pending) return (int)cudaErrorNotReady;
    const int n = render_size;
    const size_t b_par = align_up(sizeof(float) * 12 * (size_t)batch, 256);
    const size_t b_out = align_up(sizeof(long long) * 2 * (size_t)batch, 256);
    const size_t b_scr = sq_scratch_bytes(batch, n);
    int rc = slot_reserve(c, align_up(b_scr, 256) + 2 * b_par + b_out, b_out);
    if (rc) return rc;
    c->tab_dev = nullptr;                                    // this call's arena layout overwrites the resize tables
    char* d = c->dev;
    void* d_scr = d; d += align_up(b_scr, 256);
    float* d_true = reinterpret_cast<float*>(d); d += b_par;
    float* d_pred = reinterpret_cast<float*>(d); d += b_par;
    long long* d_cnt = reinterpret_cast<long long*>(d); d += b_out;
    SQ_TRY(cudaMemcpyAsync(d_true, true_host, sizeof(float) * 12 * (size_t)batch, cudaMemcpyHostToDevice, c->stream));
    SQ_TRY(cudaMemcpyAsync(d_pred, pred_host, sizeof(float) * 12 * (size_t)batch, cudaMemcpyHostToDevice, c->stream));
    rc = sq_iou_counts(d_true, d_pred, SQ_F32, batch, n, 1.0 / (double)(n - 1), 0.0, d_cnt, d_cnt + batch, d_scr, b_scr, c->stream);
    if (rc) return rc;
    SQ_TRY(cudaMemcpyAsync(c->pin, d_cnt, sizeof(long long) * 2 * (size_t)batch, cudaMemcpyDeviceToHost, c->stream));
    SQ_TRY(cudaStreamSynchronize(c->stream));
    memcpy(inter_host, c->pin, sizeof(long long) * (size_t)batch);
    memcpy(uni_host, c->pin + sizeof(long long) * (size_t)batch, sizeof(long long) * (size_t)batch);
    return 0;
}

}  // extern "C"
