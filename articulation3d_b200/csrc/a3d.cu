// a3d.cu — sm_100a kernels + C ABI (include/a3d.h) of the temporal articulation
// optimizer hot path.  See DESIGN.md for the data layout and per-kernel roofline.
//
// Arithmetic contract (bit-exactness against oracle/): every floating point
// operation that decides a pixel index is written with explicit round-to-nearest
// intrinsics (__fmul_rn/__fadd_rn/__fdiv_rn, __dmul_rn/__dadd_rn/__ddiv_rn) in the
// exact left-to-right order of the reference's matrix products, so nvcc can never
// contract them into FMAs (SURVEY.md §7 hard part 2).  The TU is additionally
// built with -fmad=false.
#include "a3d.h"

#include <cuda.h>
#include <cuda_runtime.h>
#include <time.h>

#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define A3D_CUDA_TRY(expr)                                                              \
    do {                                                                                \
        cudaError_t e__ = (expr);                                                       \
        if (e__ != cudaSuccess)                                                         \
            return fail(A3D_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                        __FILE__, __LINE__);                                            \
    } while (0)

struct Cam {
    double k[9];
    float f, cx, cy;
    int H, W, pitch;
    int sparse;   // kinv has the [[a,0,b],[0,c,d],[0,0,1]] pattern
};

__host__ __device__ inline int pitch_words(int W) { return (((W + 31) >> 5) + 3) & ~3; }

// ---------------------------------------------------------------------------
// pack: dense (n,H,W) -> bits.  One warp per image row, 32 pixels per ballot.
// Pure streaming: 4 B (fp32) or 1 B (u8) read per pixel, 1/8 B written.
// ---------------------------------------------------------------------------
// Programmatic dependent launch (a3d_pass): a kernel launched with the programmatic-serialization
// attribute may start while its predecessor in the stream is still draining; griddepcontrol.wait blocks
// until the predecessor grid has completed and its writes are visible, griddepcontrol.launch_dependents
// lets the successor's CTAs be scheduled as soon as resources free up.  Both are no-ops in a normal launch.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename T>
__global__ void __launch_bounds__(256) k_pack(const T* __restrict__ src, int64_t n_rows, int W,
                                              int pitch, float thresh, uint32_t* __restrict__ gt,
                                              uint32_t* __restrict__ nz) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int wwords = (W + 31) >> 5;
    for (int64_t row = warp0; row < n_rows; row += nwarps) {
        const T* rp = src + row * (int64_t)W;
        for (int j0 = 0; j0 < pitch; j0 += 32) {
            uint32_t mine_gt = 0, mine_nz = 0;
            const int jend = min(32, wwords - j0);
#pragma unroll 4
            for (int j = 0; j < jend; ++j) {
                const int px = ((j0 + j) << 5) + lane;
                float v = 0.f;
                if (px < W) v = (float)rp[px];
                const uint32_t bg = __ballot_sync(0xffffffffu, v > thresh);
                const uint32_t bn = __ballot_sync(0xffffffffu, v != 0.f);
                if (lane == j) { mine_gt = bg; mine_nz = bn; }
            }
            if (j0 + lane < pitch) {
                gt[row * pitch + j0 + lane] = mine_gt;
                if (nz) nz[row * pitch + j0 + lane] = mine_nz;
            }
        }
    }
}

// Vector variant for row strides that are multiples of 16 bytes (W % 4 == 0 for fp32, W % 16 == 0
// for u8): every lane loads 4 pixels per access (LDG.128 / LDG.32), 4 accesses in flight, and the
// 8 lanes of a 32-pixel word combine their nibbles with three shuffles.  128 pixels per warp step.
__device__ __forceinline__ void load4(const float* p, float (&v)[4]) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void load4(const unsigned char* p, float (&v)[4]) {
    const uchar4 t = __ldg(reinterpret_cast<const uchar4*>(p));
    v[0] = (float)t.x; v[1] = (float)t.y; v[2] = (float)t.z; v[3] = (float)t.w;
}

template <typename T>
__global__ void __launch_bounds__(256) k_pack_vec(const T* __restrict__ src, int64_t n_rows, int W, int pitch,
                                                  float thresh, uint32_t* __restrict__ gt,
                                                  uint32_t* __restrict__ nz) {
    constexpr int kUnroll = 4;
    const int lane = threadIdx.x & 31;
    const int segs = (W + 127) >> 7;                         // 128-pixel segments per row
    const int64_t total = n_rows * segs;
    const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t stride = (int64_t)gridDim.x * (blockDim.x >> 5) * kUnroll;
    // (row, seg) of the warp's current item are advanced incrementally: no 64-bit division in the loop
    int64_t it = warp0 * kUnroll;
    int64_t row = it / segs;
    int seg = (int)(it - row * segs);
    const int64_t drow = stride / segs;
    const int dseg = (int)(stride - drow * segs);
    for (; it < total; it += stride) {
        float v[kUnroll][4];
        int64_t r[kUnroll];
        int sg[kUnroll];
        {
            int64_t rr = row;
            int ss = seg;
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                r[u] = rr; sg[u] = ss;
                const int px = ss * 128 + lane * 4;
                if (it + u < total && px < W) load4(src + rr * (int64_t)W + px, v[u]);
                else { v[u][0] = v[u][1] = v[u][2] = v[u][3] = 0.f; }
                if (++ss == segs) { ss = 0; ++rr; }
            }
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            if (it + u >= total) break;
            uint32_t g = 0, z = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                g |= (uint32_t)(v[u][k] > thresh) << k;
                z |= (uint32_t)(v[u][k] != 0.f) << k;
            }
            const int sh = (lane & 7) * 4;
            g <<= sh; z <<= sh;
#pragma unroll
            for (int d = 1; d < 8; d <<= 1) {
                g |= __shfl_xor_sync(0xffffffffu, g, d);
                z |= __shfl_xor_sync(0xffffffffu, z, d);
            }
            const int word = sg[u] * 4 + (lane >> 3);
            if ((lane & 7) == 0 && word < pitch) {
                gt[r[u] * pitch + word] = g;
                if (nz) nz[r[u] * pitch + word] = z;
            }
        }
        row += drow; seg += dseg;
        if (seg >= segs) { seg -= segs; ++row; }
    }
}

// ---------------------------------------------------------------------------
// block-level reduction helpers (popcount sum + bounding box)
// ---------------------------------------------------------------------------
struct MaskStat {
    int popc, rmin, rmax, cmin, cmax;
};

__device__ inline MaskStat stat_identity() { return {0, 0x7fffffff, -1, 0x7fffffff, -1}; }

__device__ inline void stat_add_word(MaskStat& s, uint32_t w, int row, int col) {
    if (w) {
        s.popc += __popc(w);
        s.rmin = min(s.rmin, row);
        s.rmax = max(s.rmax, row);
        s.cmin = min(s.cmin, col);
        s.cmax = max(s.cmax, col);
    }
}

__device__ inline MaskStat stat_warp_reduce(MaskStat s) {
    s.popc = __reduce_add_sync(0xffffffffu, s.popc);
    s.rmin = __reduce_min_sync(0xffffffffu, s.rmin);
    s.rmax = __reduce_max_sync(0xffffffffu, s.rmax);
    s.cmin = __reduce_min_sync(0xffffffffu, s.cmin);
    s.cmax = __reduce_max_sync(0xffffffffu, s.cmax);
    return s;
}

// red points at 5 ints in shared memory initialised to the identity.
__device__ inline void stat_block_accumulate(int* red, MaskStat s) {
    s = stat_warp_reduce(s);
    if ((threadIdx.x & 31) == 0 && s.rmax >= 0) {
        atomicAdd(&red[0], s.popc);
        atomicMin(&red[1], s.rmin);
        atomicMax(&red[2], s.rmax);
        atomicMin(&red[3], s.cmin);
        atomicMax(&red[4], s.cmax);
    }
}

__device__ inline void stat_store(const int* red, int32_t* popc, int32_t* bbox) {
    *popc = red[0];
    if (red[2] < 0) {
        bbox[0] = 0; bbox[1] = -1; bbox[2] = 0; bbox[3] = -1;
    } else {
        bbox[0] = red[1]; bbox[1] = red[2]; bbox[2] = red[3]; bbox[3] = red[4];
    }
}

__global__ void __launch_bounds__(256) k_mask_meta(const uint32_t* __restrict__ bits, int H, int pitch,
                                                   int32_t* __restrict__ popc, int32_t* __restrict__ bbox) {
    __shared__ int red[5];
    if (threadIdx.x == 0) { red[0] = 0; red[1] = 0x7fffffff; red[2] = -1; red[3] = 0x7fffffff; red[4] = -1; }
    __syncthreads();
    const int64_t m = blockIdx.x;
    const uint4* p = reinterpret_cast<const uint4*>(bits + m * (int64_t)H * pitch);
    const int p4 = pitch >> 2, n4 = H * p4;
    MaskStat s = stat_identity();
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
        const uint4 v = __ldg(p + i);
        const int row = i / p4, c = (i - row * p4) << 2;
        stat_add_word(s, v.x, row, c);
        stat_add_word(s, v.y, row, c + 1);
        stat_add_word(s, v.z, row, c + 2);
        stat_add_word(s, v.w, row, c + 3);
    }
    stat_block_accumulate(red, s);
    __syncthreads();
    if (threadIdx.x == 0) stat_store(red, popc + m, bbox + 4 * m);
}

constexpr int kHF = 12;                              // floats per candidate: H (9, recentred), E_cand, exact-only flag, pad

// fp64 set-up of one candidate's homography; m = its 12 floats (R row-major, t), (x0, y0) the centre the
// source coordinates are taken from, (xm, ym) their largest magnitudes.
__device__ __forceinline__ void make_homography(const Cam& cam, const a3d_job_t& job, const float* __restrict__ m, int x0, int y0,
                                float xm, float ym, float* __restrict__ out) {
    const double U = 5.9604644775390625e-8;          // 2^-24
    double A[9], Aa[9], b[3], ba[3];
    const double a[3] = {(double)job.pivot[0], (double)job.pivot[1], (double)job.pivot[2]};
    double rho = 0.0;
    bool bad = false;
    if (job.mode == A3D_MODE_TRANSLATE) {
        for (int i = 0; i < 9; ++i) { A[i] = (i % 4 == 0) ? 1.0 : 0.0; Aa[i] = A[i]; }
    } else {
        for (int i = 0; i < 9; ++i) { A[i] = (double)m[i]; Aa[i] = fabs(A[i]); rho = fmax(rho, Aa[i]); bad |= !(Aa[i] <= 1.001); }
    }
    for (int j = 0; j < 3; ++j) {
        if (job.mode == A3D_MODE_SEQ) {
            b[j] = a[j] - (a[0] * A[j] + a[1] * A[3 + j] + a[2] * A[6 + j]);
            ba[j] = fabs(a[j]) + fabs(a[0]) * Aa[j] + fabs(a[1]) * Aa[3 + j] + fabs(a[2]) * Aa[6 + j];
        } else {
            b[j] = (double)m[9 + j];
            ba[j] = fabs(b[j]);
        }
    }
    const double n[3] = {(double)job.normal[0], (double)job.normal[1], (double)job.normal[2]};
    const double off = (double)job.offset;
    double G[9], Ga[9];                               // G[k][j] = off A[k][j] + n[k] b[j]
    for (int k = 0; k < 3; ++k)
        for (int j = 0; j < 3; ++j) {
            G[3 * k + j] = off * A[3 * k + j] + n[k] * b[j];
            Ga[3 * k + j] = fabs(off) * Aa[3 * k + j] + fabs(n[k]) * ba[j];
        }
    double L[9], La[9];                               // L[mm][j] = sum_k Kinv[k][mm] G[k][j]
    for (int mm = 0; mm < 3; ++mm)
        for (int j = 0; j < 3; ++j) {
            double v = 0.0, va = 0.0;
            for (int k = 0; k < 3; ++k) { v += cam.k[3 * k + mm] * G[3 * k + j]; va += fabs(cam.k[3 * k + mm]) * Ga[3 * k + j]; }
            L[3 * mm + j] = v; La[3 * mm + j] = va;
        }
    const double f = (double)cam.f, cx = (double)cam.cx, cy = (double)cam.cy;
    double H[9], Ha[9];                               // rows u, v, w; columns x, y, 1
    for (int mm = 0; mm < 3; ++mm) {
        H[mm] = f * L[3 * mm] + cx * L[3 * mm + 2];          Ha[mm] = f * La[3 * mm] + fabs(cx) * La[3 * mm + 2];
        H[3 + mm] = f * L[3 * mm + 1] + cy * L[3 * mm + 2];  Ha[3 + mm] = f * La[3 * mm + 1] + fabs(cy) * La[3 * mm + 2];
        H[6 + mm] = L[3 * mm + 2];                           Ha[6 + mm] = La[3 * mm + 2];
    }
    float Hf[9];
    double mag[3], maga[3];
    // rows u and v are stored divided by (W-1) and (H-1): the kernel clamps u/w with a saturating FMA
    const double scale[3] = {(double)(cam.W - 1), (double)(cam.H - 1), 1.0};
    bad |= cam.W < 2 || cam.H < 2;
    for (int r = 0; r < 3; ++r) {                     // recentre on (x0, y0)
        H[3 * r + 2] += H[3 * r] * (double)x0 + H[3 * r + 1] * (double)y0;
        Ha[3 * r + 2] += Ha[3 * r] * fabs((double)x0) + Ha[3 * r + 1] * fabs((double)y0);
        for (int i = 0; i < 3; ++i) {
            Hf[3 * r + i] = (float)(H[3 * r + i] / scale[r]);
            bad |= !(fabsf(Hf[3 * r + i]) <= 3.0e38f);
        }
        mag[r] = scale[r] * (fabs((double)Hf[3 * r]) * xm + fabs((double)Hf[3 * r + 1]) * ym + fabs((double)Hf[3 * r + 2]));
        maga[r] = Ha[3 * r] * xm + Ha[3 * r + 1] * ym + Ha[3 * r + 2];
    }
    const double Dm1 = (double)max(cam.W, cam.H) + 1.0;
    const double ec = 1.25 * (3.0 * U * (fmax(mag[0], mag[1]) + Dm1 * mag[2]) +
                              9.094947017729282e-13 * (fmax(maga[0], maga[1]) + Dm1 * maga[2]));      // 2^-40
    float ecf = __double2float_ru(ec * 1.000001);
    bad |= !(ecf <= 3.0e38f);
    // a candidate that maps the corners of the source box onto themselves in x or in y (rotation by 0,
    // translation along an image axis) leaves that coordinate of EVERY point on an integer boundary:
    // the whole candidate takes the exact chain
    bool fix_x = true, fix_y = true;
    for (int cxs = -1; cxs <= 1; cxs += 2)
        for (int cys = -1; cys <= 1; cys += 2) {
            const double xx = cxs * (double)xm, yy = cys * (double)ym;
            const double w = H[6] * xx + H[7] * yy + H[8];                // |u - x w| < 0.02 |w|: no division
            fix_x &= fabs(H[0] * xx + H[1] * yy + H[2] - (xx + x0) * w) < 0.02 * fabs(w);
            fix_y &= fabs(H[3] * xx + H[4] * yy + H[5] - (yy + y0) * w) < 0.02 * fabs(w);
        }
    bad |= fix_x | fix_y;
    for (int i = 0; i < 9; ++i) out[i] = Hf[i];
    out[9] = ecf;
    out[10] = bad ? 1.f : 0.f;
    out[11] = 0.f;
}

// ---------------------------------------------------------------------------
// unproject: source mask -> compacted fp32 point cloud (get_pcd, vis.py:86-102).
// One CTA per job.  Phase 1: exclusive prefix of the per-word popcounts of the
// source bounding box (row-major = the reference's nonzero() order).  Phase 2:
// one warp per word, one lane per pixel: float64 ray/plane intersection, one
// rounding to fp32, store at prefix + rank.  Output slice of job j:
// X | Y | Z planes of pcd_cap floats each, starting at 3 * pcd_begin.
// ---------------------------------------------------------------------------
constexpr int kUnprojThreads = 256;

template <bool kSparseK>
__global__ void __launch_bounds__(kUnprojThreads)
k_unproject(const Cam cam, const a3d_job_t* __restrict__ jobs, const uint32_t* __restrict__ src_bits,
            const int32_t* __restrict__ src_bbox, const float* __restrict__ xform, float* __restrict__ pcd,
            int32_t* __restrict__ pcd_count, float* __restrict__ hom) {
    extern __shared__ uint32_t prefix[];            // one entry per word of the source box
    __shared__ uint32_t warp_sum[kUnprojThreads / 32];
    __shared__ uint32_t total_s;
    __shared__ int tmax_s;
    pdl_launch_dependents();
    const a3d_job_t job = jobs[blockIdx.x];
    if (threadIdx.x == 0) tmax_s = 0;
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) pcd_count[gridDim.x] = 0;   // work counter of k_project_p
    const int pitch = cam.pitch;
    const int32_t* sb = src_bbox + 4 * (size_t)job.src_mask;
    const int r0 = sb[0], r1 = sb[1], w0 = sb[2], w1 = sb[3];
    if (r1 < r0) {
        if (threadIdx.x == 0 && blockIdx.y == 0) pcd_count[blockIdx.x] = 0;
        return;
    }
    const uint32_t* src = src_bits + (size_t)job.src_mask * cam.H * pitch;
    const int ncols = w1 - w0 + 1, nwords = (r1 - r0 + 1) * ncols;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    // homographies of the job's candidates for the filtered projection, one candidate per thread; source
    // coordinates are taken from the centre of the source box (smaller terms, tighter bound)
    if (hom) {
        const int y0 = (r0 + r1) >> 1, x0 = 16 * (w0 + w1 + 1);
        for (int c = blockIdx.y * kUnprojThreads + threadIdx.x; c < job.n_cand; c += kUnprojThreads * gridDim.y) {
            const size_t g = (size_t)job.cand_begin + c;
            float m[12];
#pragma unroll
            for (int i = 0; i < 12; ++i) m[i] = xform[g * 12 + i];
            make_homography(cam, job, m, x0, y0, (float)(16 * (w1 - w0 + 1)), (float)(r1 - y0), hom + g * kHF);
        }
    }

    // phase 1: block-wide exclusive scan, each thread owns a contiguous chunk of words
    const int chunk = (nwords + kUnprojThreads - 1) / kUnprojThreads;
    const int wb = min(nwords, (int)threadIdx.x * chunk), we = min(nwords, wb + chunk);
    uint32_t mine = 0;
    for (int w = wb; w < we; ++w) {
        const int rr = w / ncols;
        mine += __popc(src[(r0 + rr) * pitch + w0 + (w - rr * ncols)]);
    }
    uint32_t incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    uint32_t base = incl - mine;
    for (int i = 0; i < warp; ++i) base += warp_sum[i];
    if (threadIdx.x == kUnprojThreads - 1) total_s = base + mine;
    for (int w = wb; w < we; ++w) {
        const int rr = w / ncols;
        prefix[w] = base;
        base += __popc(src[(r0 + rr) * pitch + w0 + (w - rr * ncols)]);
    }
    __syncthreads();

    // phase 2
    const int cap = job.pcd_cap;
    float* Xp = pcd + (size_t)A3D_PCD_PLANES * job.pcd_begin;
    float* Yp = Xp + cap;
    float* Zp = Yp + cap;
    uint32_t* XYp = reinterpret_cast<uint32_t*>(Zp + cap);      // (row << 16) | column of the source pixel
    float* Cp = Zp + 2 * (size_t)cap;                           // error-bound coefficient of the point (k_project filter)
    const double n0 = (double)job.normal[0], n1 = (double)job.normal[1], n2 = (double)job.normal[2];
    const double off = (double)job.offset;
    const float NaNf = __int_as_float(0x7fffffff);
    const float INFf = __int_as_float(0x7f800000);
    // filter constants (see "filtered projection" above k_project): the largest |t| over the job's candidates
    // enters the bound of the COMPOSED / TRANSLATE chains, the pivot that of the SEQ chain
    if (job.mode != A3D_MODE_SEQ) {
        int m = 0;
        for (int i = threadIdx.x; i < job.n_cand * 3; i += kUnprojThreads) {
            float v = fabsf(xform[(size_t)(job.cand_begin + i / 3) * 12 + 9 + (i % 3)]);
            if (!(v <= 3.402823466e38f)) v = INFf;               // NaN counts as unbounded
            m = max(m, __float_as_int(v));
        }
        m = __reduce_max_sync(0xffffffffu, m);
        if (lane == 0 && m) atomicMax(&tmax_s, m);
    }
    __syncthreads();
    const double tmax = (double)__int_as_float(tmax_s);
    const double a0 = (double)job.pivot[0], a1 = (double)job.pivot[1], a2 = (double)job.pivot[2];
    const double amax = fmax(fabs(a0), fmax(fabs(a1), fabs(a2)));
    const double K1 = (double)cam.f + fmax(fabs((double)cam.cx), fabs((double)cam.cy));
    const double Dm = (double)max(cam.W, cam.H);
    // the words of the box are dealt round-robin to the warps of the gridDim.y CTAs of this job
    const int wstride = (kUnprojThreads / 32) * gridDim.y;
    for (int w = blockIdx.y * (kUnprojThreads / 32) + warp; w < nwords; w += wstride) {
        const int rr = w / ncols;
        const int row = r0 + rr, wc = w0 + (w - rr * ncols);
        const uint32_t bits = src[row * pitch + wc];
        if (!((bits >> lane) & 1u)) continue;
        const int pos = (int)prefix[w] + __popc(bits & ((1u << lane) - 1u));
        if (pos >= cap) continue;
        const double xd = (double)(wc * 32 + lane), yd = (double)row;
        double rx, ry, rz;
        if (kSparseK) {
            rx = __dadd_rn(__dmul_rn(cam.k[0], xd), cam.k[2]);
            ry = __dadd_rn(__dmul_rn(cam.k[4], yd), cam.k[5]);
            rz = 1.0;
        } else {
            rx = __dadd_rn(__dadd_rn(__dmul_rn(cam.k[0], xd), __dmul_rn(cam.k[1], yd)), cam.k[2]);
            ry = __dadd_rn(__dadd_rn(__dmul_rn(cam.k[3], xd), __dmul_rn(cam.k[4], yd)), cam.k[5]);
            rz = __dadd_rn(__dadd_rn(__dmul_rn(cam.k[6], xd), __dmul_rn(cam.k[7], yd)), cam.k[8]);
        }
        const double dot = __dadd_rn(__dadd_rn(__dmul_rn(n0, rx), __dmul_rn(n1, ry)), __dmul_rn(n2, rz));
        const double depth = __ddiv_rn(off, dot);
        float x = __double2float_rn(__dmul_rn(depth, rx));
        float y = __double2float_rn(__dmul_rn(depth, ry));
        float z = __double2float_rn(__dmul_rn(depth, rz));
        // a point with any non-finite coordinate leaves the first homogeneous transform
        // all-NaN (every output mixes 0*coordinate terms)
        const bool finite = fabsf(x) <= 3.402823466e38f && fabsf(y) <= 3.402823466e38f && fabsf(z) <= 3.402823466e38f;
        if (!finite) {
            x = NaNf; y = NaNf; z = NaNf;
        }
        Xp[pos] = x; Yp[pos] = y; Zp[pos] = z;
        // coefficient C of the point: |q_exact - q_true| <= C * |1/W_h| + c0 for every candidate, W_h the
        // homogeneous w of the plane-induced homography (scaled by n.ray, hence the |dot| factor)
        const double p1 = fabs((double)x) + fabs((double)y) + fabs((double)z);
        double Sig, M;
        if (job.mode == A3D_MODE_SEQ) {
            const double pp1 = fabs((double)x - a0) + fabs((double)y - a1) + fabs((double)z - a2);
            Sig = 1.001 * (1.01 * p1 + 5.0 * pp1) + amax;
            M = 1.001 * pp1 + amax;
        } else {
            Sig = 1.001 * 5.01 * p1 + tmax;
            M = 1.001 * p1 + tmax;
        }
        const double coef = 5.9604644775390625e-8 * 1.25 * fabs(dot) * (K1 * (Sig + 2.0 * M) + Dm * Sig);
        float cf = __double2float_ru(coef * 1.000001);
        const double dmag = fabs(n0 * rx) + fabs(n1 * ry) + fabs(n2 * rz);
        if (!finite || !(fabs(dot) >= 1e-6 * dmag) || !(cf <= 3.402823466e38f)) cf = INFf;
        XYp[pos] = ((uint32_t)row << 16) | (uint32_t)(wc * 32 + lane);
        Cp[pos] = cf;
    }
    if (threadIdx.x == 0 && blockIdx.y == 0) pcd_count[blockIdx.x] = min((int)total_s, cap);
}

// ---------------------------------------------------------------------------
// project: transform -> project -> splat, one CTA per (job, candidate tile); the
// tile's bit-masks live in shared memory.  Each thread takes 8 consecutive points
// of the compacted cloud (mostly one source row, so their images fall into one or
// two destination words) and merges their bits in registers before one atomicOr.
// ---------------------------------------------------------------------------

// emulate `.long()` of an fp32 on x86 followed by the reference's clamp to
// [0, n-1] (opt_utils.py:445-450): truncation toward zero; NaN, +-inf and
// |v| >= 2^63 become INT64_MIN, which clamps to 0.
__device__ __forceinline__ int clamp_index(float v, float n_minus_1) {
    // fmaxf/fminf drop NaN operands: NaN -> 0; negatives -> 0; [n, 2^63) -> n-1.
    float c = fminf(fmaxf(v, 0.f), n_minus_1);
    c = (v < 9.2233720368547758e18f) ? c : 0.f;      // >= 2^63, +inf (and NaN, already 0) -> 0
    return __float2int_rz(c);
}

#ifndef A3D_PROJ_THREADS
#define A3D_PROJ_THREADS 1024
#endif
constexpr int kProjThreads = A3D_PROJ_THREADS;      // 1024: one CTA per SM; 512: two, each with half the candidate slots
constexpr int kProjCtasPerSm = 1024 / kProjThreads;
#ifndef A3D_PROJECT_PERSISTENT_DEFAULT
#define A3D_PROJECT_PERSISTENT_DEFAULT false
#endif
constexpr int kProjPX = 8;

// The reference's fp32 chain for one point and one candidate (kMode is a compile-time constant so the
// code is straight-line): transform, project2D, `.long()`, clamp.  For SEQ the point is already in the
// pivot's frame (p - pivot does not depend on the candidate).
template <int kMode>
__device__ __forceinline__ void exact_pixel(float px, float py, float pz, const float* __restrict__ m,
                                            float ax, float ay, float az, float f, float cx, float cy,
                                            float wmax, float hmax, int& col, int& rw) {
    float sx, sy, sz;
    if (kMode == A3D_MODE_TRANSLATE) {
        sx = __fadd_rn(px, m[9]); sy = __fadd_rn(py, m[10]); sz = __fadd_rn(pz, m[11]);
    } else {
        sx = __fadd_rn(__fadd_rn(__fmul_rn(px, m[0]), __fmul_rn(py, m[3])), __fmul_rn(pz, m[6]));
        sy = __fadd_rn(__fadd_rn(__fmul_rn(px, m[1]), __fmul_rn(py, m[4])), __fmul_rn(pz, m[7]));
        sz = __fadd_rn(__fadd_rn(__fmul_rn(px, m[2]), __fmul_rn(py, m[5])), __fmul_rn(pz, m[8]));
        if (kMode == A3D_MODE_SEQ) {
            sx = __fadd_rn(sx, ax); sy = __fadd_rn(sy, ay); sz = __fadd_rn(sz, az);
        } else {
            sx = __fadd_rn(sx, m[9]); sy = __fadd_rn(sy, m[10]); sz = __fadd_rn(sz, m[11]);
        }
    }
    // project2D (vis.py:72-75): K@p, then /w.  The 0*X, 0*Y terms only matter for
    // non-finite inputs; keeping them in w reproduces those cases exactly.
    const float u = __fadd_rn(__fmul_rn(f, sx), __fmul_rn(cx, sz));
    const float v = __fadd_rn(__fmul_rn(f, sy), __fmul_rn(cy, sz));
    const float w = __fadd_rn(__fmaf_rn(0.f, sx, __fmul_rn(0.f, sy)), sz);   // (0*X + 0*Y) is exactly 0 or NaN
    col = clamp_index(__fdiv_rn(u, w), wmax);
    rw = clamp_index(__fdiv_rn(v, w), hmax);
}

// Hits on the same destination word are merged in registers before one shared-memory atomic.  Words
// are tracked by their 32-bit shared-memory byte address; the flush of the pending word is one
// predicated RED (no branch).
// A3D_ABLATE_* (debug builds of tools/ablate.sh only): leave one part of k_project out to measure what it costs;
// the results are then wrong by construction.
__device__ __forceinline__ void red_or_shared(uint32_t addr, uint32_t bits) {
#ifdef A3D_ABLATE_RED
    asm volatile("" ::"r"(addr), "r"(bits) : "memory");           // operands still computed, no atomic
#else
    asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(addr), "r"(bits) : "memory");
#endif
}

struct WordMerge {
    uint32_t addr, bits;
    __device__ __forceinline__ void first(uint32_t a, uint32_t bm) { addr = a; bits = bm; }
    __device__ __forceinline__ void add(uint32_t a, uint32_t bm) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.u32 p, %2, %0;\n\t"
            "@p red.shared.or.b32 [%0], %1;\n\t"
            "@p mov.b32 %1, 0;\n\t}"
            : "+r"(addr), "+r"(bits) : "r"(a) : "memory");
        addr = a;
        bits |= bm;
    }
    __device__ __forceinline__ void flush() { red_or_shared(addr, bits); }
};

// shared-memory byte address of pixel (rw, col)'s word in the mask at cm; pitch4 = bytes per packed row
__device__ __forceinline__ uint32_t word_addr(uint32_t cm, int rw, int col, int pitch4) {
    return cm + (uint32_t)(rw * pitch4) + (((uint32_t)col >> 5) << 2);
}

// One candidate applied to up to 8 points held in registers.
template <int kMode, bool kFull>
__device__ __forceinline__ void splat_points(const float (&X)[kProjPX], const float (&Y)[kProjPX],
                                             const float (&Z)[kProjPX], int nvalid, const float* __restrict__ m,
                                             float ax, float ay, float az, float f, float cx, float cy,
                                             float wmax, float hmax, int pitch4, uint32_t cm) {
    float mm[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) mm[i] = m[i];
    WordMerge mg;
#pragma unroll
    for (int k = 0; k < kProjPX; ++k) {
        if (!kFull && k >= nvalid) break;
        int col, rw;
        exact_pixel<kMode>(X[k], Y[k], Z[k], mm, ax, ay, az, f, cx, cy, wmax, hmax, col, rw);
        const uint32_t wa = word_addr(cm, rw, col, pitch4), bm = 1u << (col & 31);
        if (k == 0) mg.first(wa, bm); else mg.add(wa, bm);
    }
    mg.flush();
}

template <int kMode, int kStride>
__device__ __forceinline__ void splat_job(const Cam& cam, const a3d_job_t& job, int npts, int nc,
                                          const float* __restrict__ pcd, const float* __restrict__ xf,
                                          uint32_t* __restrict__ masks, int words, int tid) {
    const int cap = job.pcd_cap;
    const float* base = pcd + (size_t)A3D_PCD_PLANES * job.pcd_begin;
    const float4* X4 = reinterpret_cast<const float4*>(base);
    const float4* Y4 = reinterpret_cast<const float4*>(base + cap);
    const float4* Z4 = reinterpret_cast<const float4*>(base + 2 * (size_t)cap);
    const float ax = job.pivot[0], ay = job.pivot[1], az = job.pivot[2];
    const float wmax = (float)(cam.W - 1), hmax = (float)(cam.H - 1);
    const uint32_t masks_s = (uint32_t)__cvta_generic_to_shared(masks);
    const int pitch4 = cam.pitch * 4;
    const int nitems = (npts + kProjPX - 1) / kProjPX;
    auto load_item = [&](int item, float (&X)[kProjPX], float (&Y)[kProjPX], float (&Z)[kProjPX]) {
        const float4 a = __ldg(X4 + 2 * item), b = __ldg(X4 + 2 * item + 1);
        X[0] = a.x; X[1] = a.y; X[2] = a.z; X[3] = a.w; X[4] = b.x; X[5] = b.y; X[6] = b.z; X[7] = b.w;
        const float4 c = __ldg(Y4 + 2 * item), d = __ldg(Y4 + 2 * item + 1);
        Y[0] = c.x; Y[1] = c.y; Y[2] = c.z; Y[3] = c.w; Y[4] = d.x; Y[5] = d.y; Y[6] = d.z; Y[7] = d.w;
        const float4 e = __ldg(Z4 + 2 * item), g = __ldg(Z4 + 2 * item + 1);
        Z[0] = e.x; Z[1] = e.y; Z[2] = e.z; Z[3] = e.w; Z[4] = g.x; Z[5] = g.y; Z[6] = g.z; Z[7] = g.w;
        if (kMode == A3D_MODE_SEQ) {           // first step of the three-step transform, once per point
#pragma unroll
            for (int k = 0; k < kProjPX; ++k) {
                X[k] = __fsub_rn(X[k], ax); Y[k] = __fsub_rn(Y[k], ay); Z[k] = __fsub_rn(Z[k], az);
            }
        }
    };
    // full rounds: every thread owns one 8-point item and applies all candidates of the tile to it; only
    // items of 8 written points take part, so a last item of fewer points always falls in the tail below
    const int nfull = ((npts / kProjPX) / kStride) * kStride;
    for (int item = tid; item < nfull; item += kStride) {
        float X[kProjPX], Y[kProjPX], Z[kProjPX];
        load_item(item, X, Y, Z);
        for (int c = 0; c < nc; ++c)
            splat_points<kMode, true>(X, Y, Z, kProjPX, xf + 12 * c, ax, ay, az, cam.f, cam.cx, cam.cy,
                                      wmax, hmax, pitch4, masks_s + (uint32_t)(c * words) * 4u);
    }
    // last, partial round: its (item, candidate) pairs are dealt out one by one so that all
    // threads finish together (with ~1.5 items per thread the plain loop left half the warps
    // idle for a whole round: 20 % of stall samples sat at the following barrier)
    const int tail = nitems - nfull;
    for (int u = tid; u < tail * nc; u += kStride) {
        const int c = u / tail, item = nfull + (u - c * tail);
        float X[kProjPX], Y[kProjPX], Z[kProjPX];
        load_item(item, X, Y, Z);
        const int nvalid = npts - item * kProjPX;
        if (nvalid >= kProjPX)
            splat_points<kMode, true>(X, Y, Z, kProjPX, xf + 12 * c, ax, ay, az, cam.f, cam.cx, cam.cy,
                                      wmax, hmax, pitch4, masks_s + (uint32_t)(c * words) * 4u);
        else
            splat_points<kMode, false>(X, Y, Z, nvalid, xf + 12 * c, ax, ay, az, cam.f, cam.cx, cam.cy,
                                       wmax, hmax, pitch4, masks_s + (uint32_t)(c * words) * 4u);
    }
}

// ---------------------------------------------------------------------------
// Filtered projection (k_project<true>).  The reference chain costs ~80 instructions per (point,
// candidate), two thirds of them to reproduce its fp32 roundings.  But the map source pixel -> projected
// pixel of a plane under a rigid motion is a homography: with ray = Kinv [x y 1]^T, p = off ray / (n.ray),
// s = p A + b and [u v w] = K s,
//     (n.ray) [u v w]^T = H [x y 1]^T,   H = K (off A + n b^T)^T Kinv      (fp64, once per candidate)
// so q = u/w costs 6 FMA + 1 MUFU.RCP + 2 FMA.  The integer pixel trunc(q) of the cheap value is USED ONLY
// WHEN PROVEN equal to the reference's: a running error bound
//     |q_ref - q_cheap| <= eps = (C_point + E_cand) |1/W_h| + c0
// (C_point: roundings of the reference chain, written by k_unproject; E_cand: roundings of the fp32
// homography evaluation; c0: division / reciprocal terms; derivation in DESIGN.md §4a) must leave the
// cheap value more than eps away from every integer boundary.  Otherwise — 0.3 % of the coordinates on
// the synthetic scenes, plus whole candidates that map pixels onto themselves (angle 0) — the thread
// evaluates the exact chain for that point.  Results are bit-identical by construction; the tests compare
// the two kernels bit for bit.
// ---------------------------------------------------------------------------
#ifdef A3D_FILTER_STATS
// debug build only (tools/filter_stats.py): [0] (point, candidate) pairs, [1] pairs sent to the exact chain,
// [2] of those, pairs of exact-only candidates, [3] warp-iterations of the exact loop
__device__ unsigned long long g_filter_stats[4];
#endif
constexpr float kMagic = 12582912.f;                 // 1.5 * 2^23: x + kMagic holds rint(x) in its low mantissa bits
// Phase A of one (item, candidate): the cheap pixel of up to 8 points; proven ones are splatted, the
// others come back as a bit mask (bit k = point k needs the exact chain).
// The integer-pipe instructions (min/max, select, logic, compares; half rate) bound this loop, so the work
// sits on the FMA pipe wherever it can: u/w is clamped to [0, W-1] by a saturating FMA on rows pre-divided
// by W-1; x + 1.5*2^23 leaves rint(x) in the low mantissa bits and the word address is computed from those
// bits as they are (the constant part is folded into the base); every point issues its own RED, with an
// all-zero operand when it is unproven.
struct FilterConst {
    float wmax, hmax, chx, chy, c0h;                  // chx = -0.5 / wmax; c0h = c0 - 0.5 (rounded up)
    int pitch4;
};

template <bool kFull>
__device__ __forceinline__ uint32_t splat_points_filter(const float (&xs)[kProjPX], const float (&ys)[kProjPX],
                                                        const float C, int nvalid, const float* __restrict__ h,
                                                        const FilterConst& fc, uint32_t cm) {
#ifdef A3D_FILTER_STATS
    atomicAdd(&g_filter_stats[0], (unsigned long long)(kFull ? 8 : nvalid));
    if (h[10] != 0.f) {
        atomicAdd(&g_filter_stats[1], (unsigned long long)(kFull ? 8 : nvalid));
        atomicAdd(&g_filter_stats[2], (unsigned long long)(kFull ? 8 : nvalid));
    }
#endif
    if (h[10] != 0.f) return 0u;                       // exact-only candidate: handled by the straight-line chain
#ifdef A3D_ABLATE_PHASE_A
    return 0u;
#endif
    const float h0 = h[0], h1 = h[1], h2 = h[2], h3 = h[3], h4 = h[4], h5 = h[5], h6 = h[6], h7 = h[7], h8 = h[8];
    const float ce = __fadd_ru(C, h[9]);
    // bits of (kMagic + n) = 0x4B400000 + n: fold the constant out of  row * pitch4 + (col >> 5) * 4
    const uint32_t cmk = cm - 0x4B400000u * (uint32_t)fc.pitch4 - ((0x4B400000u >> 5) << 2);
    uint32_t proven = 0;
#pragma unroll
    for (int k = 0; k < kProjPX; ++k) {
        if (!kFull && k >= nvalid) break;
        const float Uq = fmaf(h0, xs[k], fmaf(h1, ys[k], h2));
        const float Vq = fmaf(h3, xs[k], fmaf(h4, ys[k], h5));
        const float Wq = fmaf(h6, xs[k], fmaf(h7, ys[k], h8));
        float r;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(Wq));
        float sx, sy;                                   // clamp((u/w - 0.5) / (W-1), 0, 1); NaN -> 0
        asm("fma.rn.sat.f32 %0, %1, %2, %3;" : "=f"(sx) : "f"(Uq), "f"(r), "f"(fc.chx));
        asm("fma.rn.sat.f32 %0, %1, %2, %3;" : "=f"(sy) : "f"(Vq), "f"(r), "f"(fc.chy));
        const float tx = fmaf(sx, fc.wmax, kMagic), ty = fmaf(sy, fc.hmax, kMagic);
        const float dx = fmaf(sx, fc.wmax, -__fsub_rn(tx, kMagic)), dy = fmaf(sy, fc.hmax, -__fsub_rn(ty, kMagic));
        const float neg_thr = fmaf(ce, fabsf(r), fc.c0h);         // eps - 0.5
        // proven only if both fractional parts keep more than eps from the integer boundaries (a NaN or
        // infinite eps fails the comparison)
        const uint32_t one = (fabsf(dx) <= -neg_thr && fabsf(dy) <= -neg_thr) ? 1u : 0u;
        const uint32_t txb = __float_as_uint(tx), tyb = __float_as_uint(ty);
        red_or_shared(tyb * (uint32_t)fc.pitch4 + cmk + ((txb >> 5) << 2), one << (txb & 31));
        proven += one << k;
    }
    return ~proven & (kFull ? 0xffu : ((1u << nvalid) - 1u));
}

// Phase B: the exact chain for the (candidate, point) pairs of one item that phase A could not prove.
// bit 8*(c - c_begin) + k of `todo`.
template <int kMode>
__device__ __forceinline__ void splat_exact_list(unsigned long long todo, int c_begin, const float* __restrict__ gX,
                                                 int cap, const float* __restrict__ xf, float ax, float ay, float az,
                                                 float f, float cx, float cy, float wmax, float hmax, int pitch4,
                                                 uint32_t masks_s, int words4) {
#ifdef A3D_FILTER_STATS
    atomicAdd(&g_filter_stats[1], (unsigned long long)__popcll(todo));
#endif
#ifdef A3D_ABLATE_EXACT_LIST
    return;
#endif
    while (todo) {
#ifdef A3D_FILTER_STATS
        if ((threadIdx.x & 31) == (__ffs(__activemask()) - 1)) atomicAdd(&g_filter_stats[3], 1ull);
#endif
        const int b = __ffsll((long long)todo) - 1;
        todo &= todo - 1;
        const int c = c_begin + (b >> 3), k = b & 7;
        float px = __ldg(gX + k), py = __ldg(gX + cap + k), pz = __ldg(gX + 2 * (size_t)cap + k);
        if (kMode == A3D_MODE_SEQ) { px = __fsub_rn(px, ax); py = __fsub_rn(py, ay); pz = __fsub_rn(pz, az); }
        int col, rw;
        exact_pixel<kMode>(px, py, pz, xf + 12 * c, ax, ay, az, f, cx, cy, wmax, hmax, col, rw);
        red_or_shared(word_addr(masks_s + (uint32_t)c * (uint32_t)words4, rw, col, pitch4), 1u << (col & 31));
    }
}

// Phase B for a whole warp: the unproven pairs of the 32 items the warp just ran phase A on, dealt to the lanes
// one pair each.  Left to its owner, a lane with 1-3 unproven pairs (0.6 % of 48) drags the whole warp through
// 2-4 passes of the reference chain with 2-4 lanes active — the ablation build without this list ran 15 %
// faster.  Here the pairs are numbered across the warp (prefix sum of the per-lane counts by shuffles — no
// shared memory is left for a queue), every lane finds the owner of pair number `lane` by binary search over
// the prefix sums, fetches the owner's mask and item by shuffle, and one pass of the chain serves up to 32 pairs.
// All 32 lanes must call it together.
template <int kMode>
__device__ __forceinline__ void splat_exact_list_warp(unsigned long long todo, int item, int c_begin,
                                                      const float* __restrict__ base, int cap, const float* __restrict__ xf,
                                                      float ax, float ay, float az, float f, float cx, float cy, float wmax,
                                                      float hmax, int pitch4, uint32_t masks_s, int words4) {
    const unsigned kAll = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int cnt = __popcll(todo);
    if (!__any_sync(kAll, cnt != 0)) return;
#ifdef A3D_FILTER_STATS
    atomicAdd(&g_filter_stats[1], (unsigned long long)cnt);
#endif
#ifdef A3D_ABLATE_EXACT_LIST
    return;
#endif
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(kAll, incl, d);
        if (lane >= d) incl += v;
    }
    const int excl = incl - cnt;
    const int total = __shfl_sync(kAll, incl, 31);
    for (int b0 = 0; b0 < total; b0 += 32) {
#ifdef A3D_FILTER_STATS
        if (lane == 0) atomicAdd(&g_filter_stats[3], 1ull);
#endif
        const int idx = b0 + lane;
        int src = 0;                                    // lanes whose pairs all come before pair idx
#pragma unroll
        for (int step = 16; step > 0; step >>= 1) {
            const int v = __shfl_sync(kAll, incl, src + step - 1);
            if (v <= idx) src += step;
        }
        src = min(src, 31);
        const unsigned lo = __shfl_sync(kAll, (unsigned)todo, src), hi = __shfl_sync(kAll, (unsigned)(todo >> 32), src);
        const int sitem = __shfl_sync(kAll, item, src);
        const int sexcl = __shfl_sync(kAll, excl, src);
        const int scb = c_begin;
        if (idx < total) {
            unsigned long long t = ((unsigned long long)hi << 32) | lo;
            for (int r = idx - sexcl; r > 0; --r) t &= t - 1;     // the (idx - sexcl)-th set bit of the owner's mask
            const int b = __ffsll((long long)t) - 1;
            const int c = scb + (b >> 3), k = b & 7;
            const float* gX = base + (size_t)sitem * kProjPX;
            float px = __ldg(gX + k), py = __ldg(gX + cap + k), pz = __ldg(gX + 2 * (size_t)cap + k);
            if (kMode == A3D_MODE_SEQ) { px = __fsub_rn(px, ax); py = __fsub_rn(py, ay); pz = __fsub_rn(pz, az); }
            int col, rw;
            exact_pixel<kMode>(px, py, pz, xf + 12 * c, ax, ay, az, f, cx, cy, wmax, hmax, col, rw);
            red_or_shared(word_addr(masks_s + (uint32_t)c * (uint32_t)words4, rw, col, pitch4), 1u << (col & 31));
        }
    }
}

template <int kMode, int kStride>
__device__ __forceinline__ void splat_job_filter(const Cam& cam, const a3d_job_t& job, int npts, int nc,
                                                 const float* __restrict__ pcd, const float* __restrict__ xf,
                                                 const float* __restrict__ hf, int x0, int y0,
                                                 uint32_t* __restrict__ masks, int words, int tid) {
    const int cap = job.pcd_cap;
    const float* base = pcd + (size_t)A3D_PCD_PLANES * job.pcd_begin;
    const uint4* XY4 = reinterpret_cast<const uint4*>(base + 3 * (size_t)cap);
    const float4* C4 = reinterpret_cast<const float4*>(base + 4 * (size_t)cap);
    const float ax = job.pivot[0], ay = job.pivot[1], az = job.pivot[2];
    const float wmax = (float)(cam.W - 1), hmax = (float)(cam.H - 1);
    const float Dm = (float)max(cam.W, cam.H);
    const int pitch4 = cam.pitch * 4, words4 = words * 4;
    FilterConst fc;
    fc.wmax = wmax; fc.hmax = hmax; fc.pitch4 = pitch4;
    fc.chx = -0.5f / wmax; fc.chy = -0.5f / hmax;
    // (Dm + 1) (2^-22 + 6 * 2^-24) + 2^-24 Dm, rounded up: reciprocal, scaled clamp and division terms
    fc.c0h = __fadd_ru(__fmul_ru(__fadd_ru(__fmul_ru(__fadd_ru(Dm, 1.f), 5.9604645e-7f), __fmul_ru(Dm, 5.9604645e-8f)), 1.0001f), -0.5f);
    const uint32_t masks_s = (uint32_t)__cvta_generic_to_shared(masks);
    const int nitems = (npts + kProjPX - 1) / kProjPX;
    // C: the largest coefficient of the item's points (neighbouring pixels: nearly equal); unwritten slots of
    // the last item are ignored
    auto load_item = [&](int item, float (&xs)[kProjPX], float (&ys)[kProjPX], float& C, int nvalid) {
        const uint4 a = __ldg(XY4 + 2 * item), b = __ldg(XY4 + 2 * item + 1);
        const uint32_t xy[kProjPX] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int k = 0; k < kProjPX; ++k) {
            xs[k] = (float)((int)(xy[k] & 0xffffu) - x0);
            ys[k] = (float)((int)(xy[k] >> 16) - y0);
        }
        const float4 c = __ldg(C4 + 2 * item), d = __ldg(C4 + 2 * item + 1);
        const float cc[kProjPX] = {c.x, c.y, c.z, c.w, d.x, d.y, d.z, d.w};
        C = 0.f;
#pragma unroll
        for (int k = 0; k < kProjPX; ++k)
            if (k < nvalid) C = (cc[k] >= C) ? cc[k] : C;         // +inf propagates (a written C is never NaN)
    };
    // full rounds: every thread owns one 8-point item and applies the candidates of the tile to it, 8 at a
    // time (the unproven pairs of 8 candidates x 8 points fit one 64-bit mask); only items of 8 written points
    const int nfull = ((npts / kProjPX) / kStride) * kStride;
    for (int item = tid; item < nfull; item += kStride) {
        float xs[kProjPX], ys[kProjPX], C;
        load_item(item, xs, ys, C, kProjPX);
        for (int cb = 0; cb < nc; cb += 8) {
            unsigned long long todo = 0;
            const int ce = min(nc, cb + 8);
            for (int c = cb; c < ce; ++c) {
                const uint32_t unc = splat_points_filter<true>(xs, ys, C, kProjPX, hf + kHF * c, fc,
                                                               masks_s + (uint32_t)(c * words4));
                todo |= (unsigned long long)unc << (8 * (c - cb));
            }
#ifdef A3D_NO_WARP_LIST               // A/B build: every lane walks its own list
            splat_exact_list<kMode>(todo, cb, base + (size_t)item * kProjPX, cap, xf, ax, ay, az, cam.f, cam.cx, cam.cy,
                                    wmax, hmax, pitch4, masks_s, words4);
#else
            // (every thread of the warp is here: nfull is a multiple of the stride)
            splat_exact_list_warp<kMode>(todo, item, cb, base, cap, xf, ax, ay, az, cam.f, cam.cx, cam.cy, wmax, hmax,
                                         pitch4, masks_s, words4);
#endif
        }
    }
    // last, partial round: its items are dealt out in (item, group of g candidates) units so that all threads
    // finish together; g is the largest group size that does not lengthen the round (a group shares one
    // load of the item and one exact list)
    const int tail = nitems - nfull;
    if (tail > 0) {
        int g = 1, best = 0x7fffffff;
        for (int t = 1; t <= min(nc, 8); ++t) {
            const int rounds = (tail * ((nc + t - 1) / t) + kStride - 1) / kStride;
            if (rounds * t <= best) { best = rounds * t; g = t; }
        }
        const int ngroups = (nc + g - 1) / g;
        // (the lanes of a warp leave this loop at different times, so every lane walks its own list here; a
        // warp-uniform form of the loop with the shared list was measured 3 % slower: spills)
        for (int u = tid; u < tail * ngroups; u += kStride) {
            const int grp = u / tail, item = nfull + (u - grp * tail);
            const int cb = grp * g, ce = min(nc, cb + g);
            float xs[kProjPX], ys[kProjPX], C;
            const int nvalid = min(kProjPX, npts - item * kProjPX);
            load_item(item, xs, ys, C, nvalid);
            unsigned long long todo = 0;
            for (int c = cb; c < ce; ++c) {
                const uint32_t unc = splat_points_filter<false>(xs, ys, C, nvalid, hf + kHF * c, fc,
                                                                masks_s + (uint32_t)(c * words4));
                todo |= (unsigned long long)unc << (8 * (c - cb));
            }
            splat_exact_list<kMode>(todo, cb, base + (size_t)item * kProjPX, cap, xf, ax, ay, az, cam.f, cam.cx, cam.cy,
                                    wmax, hmax, pitch4, masks_s, words4);
        }
    }
}

// CTA roles.  k_project<false>: a worker = (job, tile of <= tile_cand candidates), the reference chain for
// every point.  k_project<true>: the same tiles run the filter on their candidates; candidates flagged
// exact-only by k_unproject (rotation by 0: every pixel maps onto an integer boundary) cost 3x a filtered
// one, so they are taken out of the tiles and given to one EXTRA worker per job, which runs the
// straight-line reference chain on them — unless the job has more of them than one worker holds, in which
// case every tile keeps its own.
//
// A worker is kStride threads with their own candidate slots in shared memory and their own barrier:
// the whole CTA (k_project: 1024 threads, one tile per CTA) or half of it (k_project_p: two groups of 512
// threads that fetch tiles from a global counter until none is left — while one group sits in the load
// latencies of its prologue, the barrier at the end of its splat or its write-out, the other one computes).
struct ProjSmem {
    uint32_t* masks;   // [slots][words]
    float* xf;         // [slots][12]
    int* red;          // [slots][5]
    float* hf;         // [slots][kHF]   (filter only)
    int* gid;          // [slots] candidate of the slot, -1 = not mine
    int* ctl;          // [2] nflag, nlist
};

template <int kStride>
__device__ __forceinline__ void worker_sync(int barrier_id) {
    if (kStride == kProjThreads) __syncthreads();
    else if (barrier_id == 1) asm volatile("bar.sync 1, %0;" ::"n"(kStride) : "memory");
    else asm volatile("bar.sync 2, %0;" ::"n"(kStride) : "memory");
}

// Streams a worker's tile out of shared memory, with popcount + bounding box per candidate.
// (row, uint4 column) of a thread's elements advance by constants: no division in the loop; the occupied word
// columns are collected as a bit mask (pitch <= 32 words).
// kRows = false (A3D_OUT_FULL): every word is written.  kRows = true (A3D_OUT_BBOX_ROWS): the slot's image in
// proj_bits is zero outside the rows of proj_bbox[slot] (the caller's promise on entry, this kernel's on exit),
// so a 16-byte piece is written only if it lies in a row of the slot's OLD box (whatever it holds now, zeros
// included) or is non-zero — one pass, no box needed in advance.  A door-sized mask occupies an eighth of the
// frame's rows; the zeros around it were 85 % of the pass's DRAM writes.
template <bool kRows, int kStride>
__device__ __forceinline__ void write_tile(const a3d_job_t& job, int nc, int H, int pitch, int words,
                                           const uint32_t* __restrict__ masks, const int* __restrict__ gid,
                                           int* __restrict__ red, uint32_t* __restrict__ proj_bits,
                                           int32_t* __restrict__ proj_popc, int32_t* __restrict__ proj_bbox, int tid,
                                           int bar) {
    const int p4 = pitch >> 2, n4 = H * p4;
    const int row0 = tid / p4, col0 = tid - row0 * p4;
    const int drow = kStride / p4, dcol = kStride - drow * p4;
    for (int c = 0; c < nc; ++c) {
        if (gid[c] < 0) continue;
        const size_t g = (size_t)job.cand_begin + gid[c];
        const uint4* s4 = reinterpret_cast<const uint4*>(masks + (size_t)c * words);
        uint4* d4 = reinterpret_cast<uint4*>(proj_bits + g * words);
        int wlo = 0, whi = -1;                       // rows of the old box: always written
        if (kRows) { wlo = proj_bbox[4 * g]; whi = proj_bbox[4 * g + 1]; }
        MaskStat s = stat_identity();
        if (pitch <= 32) {
            uint32_t colmask = 0;
            int row = row0, col = col0;
            for (int i = tid; i < n4; i += kStride) {
                const uint4 v = s4[i];
                const bool nzv = (v.x | v.y | v.z | v.w) != 0u;
                if (!kRows || nzv || (row >= wlo && row <= whi)) d4[i] = v;
                if (nzv) {
                    s.popc += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
                    s.rmin = min(s.rmin, row);
                    s.rmax = max(s.rmax, row);
                    const uint32_t nz = (v.x ? 1u : 0u) | (v.y ? 2u : 0u) | (v.z ? 4u : 0u) | (v.w ? 8u : 0u);
                    colmask |= nz << (4 * col);
                }
                row += drow; col += dcol;
                if (col >= p4) { col -= p4; ++row; }
            }
            colmask = __reduce_or_sync(0xffffffffu, colmask);
            if (colmask) { s.cmin = __ffs(colmask) - 1; s.cmax = 31 - __clz(colmask); }
        } else {
            for (int i = tid; i < n4; i += kStride) {
                const uint4 v = s4[i];
                const int row = i / p4;
                const bool nzv = (v.x | v.y | v.z | v.w) != 0u;
                if (!kRows || nzv || (row >= wlo && row <= whi)) d4[i] = v;
                if (nzv) {
                    const int cc = (i - row * p4) << 2;
                    stat_add_word(s, v.x, row, cc);
                    stat_add_word(s, v.y, row, cc + 1);
                    stat_add_word(s, v.z, row, cc + 2);
                    stat_add_word(s, v.w, row, cc + 3);
                }
            }
        }
        stat_block_accumulate(red + 5 * c, s);
    }
    worker_sync<kStride>(bar);                     // (the old boxes are all read before any is replaced)
    for (int c = tid; c < nc; c += kStride) {
        if (gid[c] < 0) continue;
        const size_t g = (size_t)job.cand_begin + gid[c];
        stat_store(red + 5 * c, proj_popc + g, proj_bbox + 4 * g);
    }
}

template <bool kFilter, int kStride>
__device__ __forceinline__ void project_tile(const Cam& cam, const a3d_job_t& job, int jid, int c0, int want, bool extra,
                                             int slots, const float* __restrict__ xform,
                                             const int32_t* __restrict__ src_bbox, const float* __restrict__ pcd,
                                             const int32_t* __restrict__ pcd_count, const float* __restrict__ hom,
                                             uint32_t* __restrict__ proj_bits, int32_t* __restrict__ proj_popc,
                                             int32_t* __restrict__ proj_bbox, const ProjSmem& sm, int tid, int bar,
                                             bool first, bool rows_only) {
    if (extra) c0 = 0;
    int nc = extra ? min(slots, job.n_cand) : min(want, job.n_cand - c0);   // slots in use
    if (nc <= 0 || c0 < 0) {
        if (first) { pdl_wait(); pdl_launch_dependents(); }
        return;
    }
    const int H = cam.H, pitch = cam.pitch;
    const int words = H * pitch;
    uint32_t* masks = sm.masks;
    float* xf = sm.xf;
    int* red = sm.red;
    float* hf = sm.hf;
    int* gid = sm.gid;
    {
        uint4* m4 = reinterpret_cast<uint4*>(masks);
        const int n4 = (nc * words) >> 2;
        for (int i = tid; i < n4; i += kStride) m4[i] = make_uint4(0, 0, 0, 0);
        if (!extra) {
            const float* gx = xform + (size_t)(job.cand_begin + c0) * 12;
            for (int i = tid; i < nc * 12; i += kStride) xf[i] = gx[i];
        }
        for (int i = tid; i < nc; i += kStride) {
            red[5 * i + 0] = 0; red[5 * i + 1] = 0x7fffffff; red[5 * i + 2] = -1;
            red[5 * i + 3] = 0x7fffffff; red[5 * i + 4] = -1;
            gid[i] = extra ? -1 : c0 + i;
        }
        if (tid == 0) { sm.ctl[0] = 0; sm.ctl[1] = 0; }
    }
    worker_sync<kStride>(bar);
    if (first) {
        pdl_wait();                   // the point clouds of k_unproject (the shared-memory tile is already zeroed)
        pdl_launch_dependents();
    }
    const int npts = pcd_count[jid];
    int x0 = 0, y0 = 0;
    bool moved = false;               // exact-only candidates of this job live in the extra worker
    if (kFilter) {
        const int32_t* sb = src_bbox + 4 * (size_t)job.src_mask;
        y0 = (sb[0] + sb[1]) >> 1;
        x0 = 16 * (sb[2] + sb[3] + 1);
        const float* gh = hom + (size_t)job.cand_begin * kHF;                 // written by k_unproject
        int mine = 0;
        for (int c = tid; c < job.n_cand; c += kStride) mine += (npts > 0 && gh[(size_t)c * kHF + 10] != 0.f) ? 1 : 0;
        mine = __reduce_add_sync(0xffffffffu, mine);
        if ((tid & 31) == 0 && mine) atomicAdd(&sm.ctl[0], mine);
        if (!extra)
            for (int i = tid; i < nc * kHF; i += kStride) hf[i] = gh[(size_t)c0 * kHF + i];
        worker_sync<kStride>(bar);
        const int nflag = sm.ctl[0];
        moved = nflag > 0 && nflag <= slots;
        if (extra) {
            if (!moved) return;
            for (int c = tid; c < job.n_cand; c += kStride)
                if (gh[(size_t)c * kHF + 10] != 0.f) {
                    const int slot = atomicAdd(&sm.ctl[1], 1);
                    gid[slot] = c;
                    for (int i = 0; i < 12; ++i) xf[12 * slot + i] = xform[(size_t)(job.cand_begin + c) * 12 + i];
                }
            nc = nflag;
            worker_sync<kStride>(bar);          // the slots' transforms and candidate ids
        } else if (moved) {
            // (read again only after the barrier that ends the splat)
            for (int i = tid; i < nc; i += kStride)
                if (hf[kHF * i + 10] != 0.f) gid[i] = -1;
        }
    } else if (extra) {
        return;
    }
    if (npts > 0) {
        if (kFilter && !extra) {
            if (job.mode == A3D_MODE_SEQ) splat_job_filter<A3D_MODE_SEQ, kStride>(cam, job, npts, nc, pcd, xf, hf, x0, y0, masks, words, tid);
            else if (job.mode == A3D_MODE_COMPOSED) splat_job_filter<A3D_MODE_COMPOSED, kStride>(cam, job, npts, nc, pcd, xf, hf, x0, y0, masks, words, tid);
            else splat_job_filter<A3D_MODE_TRANSLATE, kStride>(cam, job, npts, nc, pcd, xf, hf, x0, y0, masks, words, tid);
            if (!moved && sm.ctl[0] > 0) {
                // more exact-only candidates than the extra worker holds: each tile runs its own
                for (int c = 0; c < nc; ++c) {
                    if (hf[kHF * c + 10] == 0.f) continue;
                    if (job.mode == A3D_MODE_SEQ) splat_job<A3D_MODE_SEQ, kStride>(cam, job, npts, 1, pcd, xf + 12 * c, masks + (size_t)c * words, words, tid);
                    else if (job.mode == A3D_MODE_COMPOSED) splat_job<A3D_MODE_COMPOSED, kStride>(cam, job, npts, 1, pcd, xf + 12 * c, masks + (size_t)c * words, words, tid);
                    else splat_job<A3D_MODE_TRANSLATE, kStride>(cam, job, npts, 1, pcd, xf + 12 * c, masks + (size_t)c * words, words, tid);
                }
            }
        } else {
            if (job.mode == A3D_MODE_SEQ) splat_job<A3D_MODE_SEQ, kStride>(cam, job, npts, nc, pcd, xf, masks, words, tid);
            else if (job.mode == A3D_MODE_COMPOSED) splat_job<A3D_MODE_COMPOSED, kStride>(cam, job, npts, nc, pcd, xf, masks, words, tid);
            else splat_job<A3D_MODE_TRANSLATE, kStride>(cam, job, npts, nc, pcd, xf, masks, words, tid);
        }
    }
    worker_sync<kStride>(bar);

#ifdef A3D_ABLATE_WRITE
    return;
#endif
    if (rows_only) write_tile<true, kStride>(job, nc, H, pitch, words, masks, gid, red, proj_bits, proj_popc, proj_bbox, tid, bar);
    else write_tile<false, kStride>(job, nc, H, pitch, words, masks, gid, red, proj_bits, proj_popc, proj_bbox, tid, bar);
}

// worker id -> (job, first candidate, candidates, extra): from the caller's tile map, else uniform tiles
template <bool kFilter>
__device__ __forceinline__ void decode_work(int w, const int4* __restrict__ tile_map, int tile_cand, int tiles_per_job,
                                            int& jid, int& c0, int& want, bool& extra) {
    if (tile_map) {                   // caller-planned tiles: {job, first candidate, count, 1 = the job's extra worker}
        const int4 t = tile_map[w];
        jid = t.x; c0 = t.y; want = min(t.z, tile_cand); extra = t.w != 0;
    } else {
        const int per_job = tiles_per_job + (kFilter ? 1 : 0);
        jid = w / per_job;
        const int tile_id = w - jid * per_job;
        extra = kFilter && tile_id == tiles_per_job;
        c0 = tile_id * tile_cand; want = tile_cand;
    }
}

template <bool kFilter>
__global__ void __launch_bounds__(kProjThreads, kProjCtasPerSm)
k_project(const Cam cam, const a3d_job_t* __restrict__ jobs, int tile_cand, int tiles_per_job,
          const float* __restrict__ xform, const int32_t* __restrict__ src_bbox, const float* __restrict__ pcd,
          const int32_t* __restrict__ pcd_count, const float* __restrict__ hom, const int4* __restrict__ tile_map,
          uint32_t* __restrict__ proj_bits, int32_t* __restrict__ proj_popc, int32_t* __restrict__ proj_bbox,
          bool rows_only) {
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ int ctl[2];
    int jid, c0, want;
    bool extra;
    decode_work<kFilter>(blockIdx.x, tile_map, tile_cand, tiles_per_job, jid, c0, want, extra);
    const a3d_job_t job = jobs[jid];
    const int words = cam.H * cam.pitch;
    ProjSmem sm;
    sm.masks = smem;
    sm.xf = reinterpret_cast<float*>(smem + (size_t)tile_cand * words);
    sm.red = reinterpret_cast<int*>(sm.xf + tile_cand * 12);
    sm.hf = reinterpret_cast<float*>(sm.red + tile_cand * 5);
    sm.gid = reinterpret_cast<int*>(sm.hf + tile_cand * kHF);
    sm.ctl = ctl;
    project_tile<kFilter, kProjThreads>(cam, job, jid, c0, want, extra, tile_cand, xform, src_bbox, pcd, pcd_count, hom,
                                        proj_bits, proj_popc, proj_bbox, sm, threadIdx.x, 0, true, rows_only);
}

// Persistent variant: gridDim.x <= SM count CTAs of two 512-thread groups; each group owns tile_cand
// candidate slots and takes the next tile from *work_counter (zeroed by k_unproject) until n_work are done.
constexpr int kGroupThreads = kProjThreads / 2;

template <bool kFilter>
__global__ void __launch_bounds__(kProjThreads, 1)
k_project_p(const Cam cam, const a3d_job_t* __restrict__ jobs, int tile_cand, int tiles_per_job, int n_work,
            int* __restrict__ work_counter, const float* __restrict__ xform, const int32_t* __restrict__ src_bbox,
            const float* __restrict__ pcd, const int32_t* __restrict__ pcd_count, const float* __restrict__ hom,
            const int4* __restrict__ tile_map, uint32_t* __restrict__ proj_bits, int32_t* __restrict__ proj_popc,
            int32_t* __restrict__ proj_bbox, bool rows_only) {
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ int ctl[2][2];
    __shared__ int next_work[2];
    const int g = threadIdx.x / kGroupThreads, tid = threadIdx.x - g * kGroupThreads;
    const int words = cam.H * cam.pitch;
    // per group: masks | xf | red | hf | gid, laid out as in k_project with tile_cand slots
    const size_t group_words = ((size_t)tile_cand * (words + 12 + 5 + kHF + 1) + 3) & ~(size_t)3;
    uint32_t* base = smem + (size_t)g * group_words;
    ProjSmem sm;
    sm.masks = base;
    sm.xf = reinterpret_cast<float*>(base + (size_t)tile_cand * words);
    sm.red = reinterpret_cast<int*>(sm.xf + tile_cand * 12);
    sm.hf = reinterpret_cast<float*>(sm.red + tile_cand * 5);
    sm.gid = reinterpret_cast<int*>(sm.hf + tile_cand * kHF);
    sm.ctl = ctl[g];
    const int bar = 1 + g;
    pdl_wait();                       // the work counter and the point clouds of k_unproject
    pdl_launch_dependents();
    for (;;) {
        if (tid == 0) next_work[g] = atomicAdd(work_counter, 1);
        worker_sync<kGroupThreads>(bar);
        const int w = next_work[g];
        if (w >= n_work) break;
        int jid, c0, want;
        bool extra;
        decode_work<kFilter>(w, tile_map, tile_cand, tiles_per_job, jid, c0, want, extra);
        const a3d_job_t job = jobs[jid];
        project_tile<kFilter, kGroupThreads>(cam, job, jid, c0, want, extra, tile_cand, xform, src_bbox, pcd, pcd_count,
                                             hom, proj_bits, proj_popc, proj_bbox, sm, tid, bar, false, rows_only);
        worker_sync<kGroupThreads>(bar);        // the slots and next_work are free again
    }
}

// ---------------------------------------------------------------------------
// score: inter[t][c] = popc(T_t & P_c) over the overlap of the bounding boxes;
// union = |T_t| + |P_c| - inter; iou = fp32 divide; arg-max over candidates is
// fused through a 64-bit atomicMax key  (iou bits << 32) | ~candidate
// (first maximum wins; NaN = 0/0 orders above every finite value, as in torch).
// CTA = 8 warps = (2 target groups) x (4 candidate groups); each warp owns a
// 4x4 register tile of (target, candidate) pairs and strides its lanes over the
// words of the region, two words per step folded by a carry-save adder so that
// one POPC (quarter-rate pipe) serves two words.  CTAs are ordered job-major so
// one job's masks stay L2-resident while its tiles run.
// ---------------------------------------------------------------------------
// arg-max key: IoU bits in the high word (IoU >= 0 or NaN, so unsigned order = float order with
// NaN on top, as torch.argmax), then the candidate index inverted so the FIRST maximum wins.
// When candidates < 4096 and the mask has < 2^20 pixels the intersection count rides in the low
// 20 bits ("packed"), so the winner's counts need no recomputation.
__device__ __forceinline__ unsigned long long make_key(float iou, int cand, int inter, int packed) {
    const unsigned lo = packed ? (((0xfffu - (unsigned)cand) << 20) | (unsigned)inter) : ~(unsigned)cand;
    return ((unsigned long long)__float_as_uint(iou) << 32) | lo;
}

// one carry-save step of the popcount accumulation: a, b are two AND-ed words, o the pending
// weight-1 bits.  Explicit LOP3s (xor3 = 0x96, majority = 0xE8) keep it at 4 logic ops per pair;
// left to the compiler the 5-input majority is re-derived from the un-ANDed words in 6.
__device__ __forceinline__ void csa_step(uint32_t a, uint32_t b, uint32_t& ones, int& acc2) {
    uint32_t s, c;
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(s) : "r"(ones), "r"(a), "r"(b));
    asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(c) : "r"(ones), "r"(a), "r"(b));
    ones = s;
    acc2 += __popc(c);
}

constexpr int kScoreTT = 8;    // targets per CTA

// kNarrow: every mask of the target pool / of the projected masks starts less than 2^32 words from its base,
// so a load address is base + 32-bit word offset (one IMAD.WIDE) instead of a 64-bit pointer per mask —
// without it half of the loop's instructions were address arithmetic.
// kWC: candidates per warp (warp tile = 4 targets x kWC candidates; CTA = 8 targets x 4*kWC candidates).
template <bool kNarrow, int kWC, bool kPipe>
__global__ void __launch_bounds__(256, (kWC == 4 || kPipe) ? 3 : 4)
k_score(const a3d_job_t* __restrict__ jobs, int H, int pitch, int tt_tiles, int ct_tiles,
        const uint32_t* __restrict__ tgt_bits, const int32_t* __restrict__ tgt_popc,
        const int32_t* __restrict__ tgt_bbox, const int32_t* __restrict__ tgt_index,
        const uint32_t* __restrict__ proj_bits, const int32_t* __restrict__ proj_popc,
        const int32_t* __restrict__ proj_bbox, unsigned long long* __restrict__ key_ws,
        int32_t* __restrict__ inter_tab, int packed) {
    const int per_job = tt_tiles * ct_tiles;
    const int jid = blockIdx.x / per_job;
    const int rem = blockIdx.x - jid * per_job;
    const a3d_job_t job = jobs[jid];
    const int tb = (rem / ct_tiles) * kScoreTT;
    const int cb = (rem % ct_tiles) * (4 * kWC);
    if (tb >= job.n_tgt || cb >= job.n_cand) return;
    pdl_wait();                       // the projected masks of k_project
    pdl_launch_dependents();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t0 = tb + (warp >> 2) * 4;
    const int c0 = cb + (warp & 3) * kWC;
    if (t0 >= job.n_tgt || c0 >= job.n_cand) return;
    const int nt = min(4, job.n_tgt - t0), ncd = min(kWC, job.n_cand - c0);
    const size_t words = (size_t)H * pitch;

    const uint32_t* tp[4];          // wide addressing: one pointer per mask
    const uint32_t* pp[kWC];
    unsigned toff[4], poff[kWC];    // narrow addressing: 32-bit word offsets from tgt_bits / proj_bits
    int tmask[4];
    // region = (union of candidate boxes) ∩ (union of target boxes)
    int pr0 = 0x7fffffff, pr1 = -1, pc0 = 0x7fffffff, pc1 = -1;
    int qr0 = 0x7fffffff, qr1 = -1, qc0 = 0x7fffffff, qc1 = -1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int ti = min(i, nt - 1);
        tmask[i] = tgt_index[job.tgt_begin + t0 + ti];
        tp[i] = tgt_bits + (size_t)tmask[i] * words;
        toff[i] = (unsigned)tmask[i] * (unsigned)words;
        const int32_t* b = tgt_bbox + 4 * (size_t)tmask[i];
        if (b[1] >= b[0]) { qr0 = min(qr0, b[0]); qr1 = max(qr1, b[1]); qc0 = min(qc0, b[2]); qc1 = max(qc1, b[3]); }
    }
#pragma unroll
    for (int k = 0; k < kWC; ++k) {
        const int ci = min(k, ncd - 1);
        const size_t g = (size_t)job.cand_begin + c0 + ci;
        pp[k] = proj_bits + g * words;
        poff[k] = (unsigned)g * (unsigned)words;
        const int32_t* pb = proj_bbox + 4 * g;
        if (pb[1] >= pb[0]) { pr0 = min(pr0, pb[0]); pr1 = max(pr1, pb[1]); pc0 = min(pc0, pb[2]); pc1 = max(pc1, pb[3]); }
    }
    const int ra = max(pr0, qr0), rb = min(pr1, qr1), ca = max(pc0, qc0), cbw = min(pc1, qc1);

    int acc2[4][kWC];           // number of carries (weight 2)
    uint32_t ones[4][kWC];      // pending weight-1 bits
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int k = 0; k < kWC; ++k) { acc2[i][k] = 0; ones[i][k] = 0u; }

    if (rb >= ra && cbw >= ca) {
        const int ncols = cbw - ca + 1;
        const int total = (rb - ra + 1) * ncols;
        // two word positions per step: idx and idx + 32, both advance by 64
        const int dr = 64 / ncols, dc = 64 - dr * ncols;
        int rA = lane / ncols, cA = lane - rA * ncols;
        int rB = (lane + 32) / ncols, cB = (lane + 32) - rB * ncols;
        struct Step { uint32_t tA[4], tB[4], pA[kWC], pB[kWC]; };
        auto load = [&](int idx, Step& w) {                       // the loads of step idx, and advance the cursor
            const unsigned oA = (unsigned)((ra + rA) * pitch + ca + cA);
            const bool hasB = idx + 32 < total;
            const unsigned oB = hasB ? (unsigned)((ra + rB) * pitch + ca + cB) : oA;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                w.tA[i] = kNarrow ? __ldg(tgt_bits + (toff[i] + oA)) : __ldg(tp[i] + oA);
                w.tB[i] = kNarrow ? __ldg(tgt_bits + (toff[i] + oB)) : __ldg(tp[i] + oB);
            }
#pragma unroll
            for (int k = 0; k < kWC; ++k) {
                w.pA[k] = kNarrow ? __ldg(proj_bits + (poff[k] + oA)) : __ldg(pp[k] + oA);
                w.pB[k] = kNarrow ? __ldg(proj_bits + (poff[k] + oB)) : __ldg(pp[k] + oB);
            }
            if (!hasB) {
#pragma unroll
                for (int i = 0; i < 4; ++i) w.tB[i] = 0u;
            }
            rA += dr; cA += dc;
            if (cA >= ncols) { cA -= ncols; ++rA; }
            rB += dr; cB += dc;
            if (cB >= ncols) { cB -= ncols; ++rB; }
        };
        auto fold = [&](const Step& w) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int k = 0; k < kWC; ++k) csa_step(w.tA[i] & w.pA[k], w.tB[i] & w.pB[k], ones[i][k], acc2[i][k]);
        };
        if (kPipe) {
            // small grids are bound by the chain of load latencies of a warp's few steps (C2: ~7 steps, every
            // first touch a DRAM miss): the next step's loads are in flight while this one is folded
            Step a, b;
            int idx = lane;
            if (idx < total) load(idx, a);
            while (idx < total) {
                if (idx + 64 < total) load(idx + 64, b);
                fold(a);
                idx += 64;
                if (idx >= total) break;
                if (idx + 64 < total) load(idx + 64, a);
                fold(b);
                idx += 64;
            }
        } else {
            for (int idx = lane; idx < total; idx += 64) {
                Step w;
                load(idx, w);
                fold(w);
            }
        }
    }
    int acc[4][kWC];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int k = 0; k < kWC; ++k)
            acc[i][k] = __reduce_add_sync(0xffffffffu, 2 * acc2[i][k] + __popc(ones[i][k]));

    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (i >= nt) break;
            const int pt = tgt_popc[tmask[i]];
            unsigned long long best = 0ull;
#pragma unroll
            for (int k = 0; k < kWC; ++k) {
                if (k >= ncd) break;
                const int inter = acc[i][k];
                const int uni = pt + proj_popc[(size_t)job.cand_begin + c0 + k] - inter;
                const float iou = __fdiv_rn((float)inter, (float)uni);
                const unsigned long long key = make_key(iou, c0 + k, inter, packed);
                best = key > best ? key : best;
                if (inter_tab) inter_tab[job.tab_begin + (int64_t)(t0 + i) * job.n_cand + c0 + k] = inter;
            }
            atomicMax(key_ws + job.tgt_begin + t0 + i, best);
        }
    }
}

// ---------------------------------------------------------------------------
// score, TMA-staged.  Same arithmetic as k_score above; CTA = (job, 16 targets,
// 8 candidates), 8 warps = 4 target groups x 2 candidate groups, each warp a
// 4x4 register tile.  The CTA walks the overlap box of its masks in chunks of
// R rows x bw words (R*bw <= 256 words = 1 KB per mask); warp 0 stages the 24
// mask tiles of the NEXT chunk with cp.async.bulk.tensor.2d (TMA, completion on
// an mbarrier) while all warps AND/POPC the current one out of shared memory.
// Tensor maps: uint32 [n_masks*H][pitch] with boxes {bw, R}; out-of-range
// columns are zero-filled by the TMA unit.
// ---------------------------------------------------------------------------
constexpr int kTmaTT = 8, kTmaCT = 16, kTmaMasks = kTmaTT + kTmaCT;
constexpr int kTmaTileWords = 256;
constexpr int kTmaStages = 2;
constexpr size_t kTmaSmemBytes = (size_t)kTmaStages * kTmaMasks * kTmaTileWords * 4 + 64;

struct TmaMaps {
    CUtensorMap t[4];     // target pool, box widths bw[0..3]
    CUtensorMap p[4];     // projected masks
    int bw[4];            // words per box row
    int rows[4];          // rows per box
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar) : "memory");
}

__global__ void __launch_bounds__(256, 3)
k_score_tma(const __grid_constant__ TmaMaps maps, const a3d_job_t* __restrict__ jobs, int H, int pitch,
            int tt_tiles, int ct_tiles, const int32_t* __restrict__ tgt_popc,
            const int32_t* __restrict__ tgt_bbox, const int32_t* __restrict__ tgt_index,
            const int32_t* __restrict__ proj_popc, const int32_t* __restrict__ proj_bbox,
            unsigned long long* __restrict__ key_ws, int32_t* __restrict__ inter_tab, int packed) {
    extern __shared__ __align__(1024) uint32_t tiles[];      // [stage][mask][256 words]
    __shared__ int s_mask_row0[kTmaMasks];                   // first tensor row of every mask of the tile
    __shared__ int s_mbox[kTmaMasks][4];                     // bounding box of every mask of the tile
    __shared__ int s_wbox[8][4];                             // per-warp region
    uint64_t* bars = reinterpret_cast<uint64_t*>(tiles + kTmaStages * kTmaMasks * kTmaTileWords);

    const int per_job = tt_tiles * ct_tiles;
    const int jid = blockIdx.x / per_job;
    const int rem = blockIdx.x - jid * per_job;
    const a3d_job_t job = jobs[jid];
    const int tb = (rem / ct_tiles) * kTmaTT;
    const int cb = (rem % ct_tiles) * kTmaCT;
    if (tb >= job.n_tgt || cb >= job.n_cand) return;           // whole CTA leaves together
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ntile_t = min(kTmaTT, job.n_tgt - tb), ntile_c = min(kTmaCT, job.n_cand - cb);
    pdl_wait();
    pdl_launch_dependents();

    if (threadIdx.x == 0) {
        mbar_init(smem_u32(&bars[0]), 1);
        mbar_init(smem_u32(&bars[1]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x < kTmaMasks) {
        const int m = threadIdx.x;
        const int32_t* b;
        if (m < kTmaTT) {
            const int ti = tgt_index[job.tgt_begin + tb + min(m, ntile_t - 1)];
            s_mask_row0[m] = ti * H;
            b = tgt_bbox + 4 * (size_t)ti;
        } else {
            const int g = job.cand_begin + cb + min(m - kTmaTT, ntile_c - 1);
            s_mask_row0[m] = g * H;
            b = proj_bbox + 4 * (size_t)g;
        }
        s_mbox[m][0] = b[0]; s_mbox[m][1] = b[1]; s_mbox[m][2] = b[2]; s_mbox[m][3] = b[3];
    }
    __syncthreads();

    // this warp's 4 targets x 4 candidates inside the tile, and its own overlap box:
    // (union of its candidate boxes) ∩ (union of its target boxes)
    const int tw = (warp >> 2) * 4, cw = (warp & 3) * 4;
    const bool active = tw < ntile_t && cw < ntile_c;
    int wra = 0, wrb = -1, wca = 0, wcb = -1;
    if (active) {
        int pr0 = 0x7fffffff, pr1 = -1, pc0 = 0x7fffffff, pc1 = -1;
        int qr0 = 0x7fffffff, qr1 = -1, qc0 = 0x7fffffff, qc1 = -1;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int* t = s_mbox[min(tw + i, ntile_t - 1)];
            if (t[1] >= t[0]) { qr0 = min(qr0, t[0]); qr1 = max(qr1, t[1]); qc0 = min(qc0, t[2]); qc1 = max(qc1, t[3]); }
            const int* c = s_mbox[kTmaTT + min(cw + i, ntile_c - 1)];
            if (c[1] >= c[0]) { pr0 = min(pr0, c[0]); pr1 = max(pr1, c[1]); pc0 = min(pc0, c[2]); pc1 = max(pc1, c[3]); }
        }
        wra = max(pr0, qr0); wrb = min(pr1, qr1); wca = max(pc0, qc0); wcb = min(pc1, qc1);
        if (wrb < wra || wcb < wca) { wra = 0; wrb = -1; wca = 0; wcb = -1; }
    }
    if (lane == 0) { s_wbox[warp][0] = wra; s_wbox[warp][1] = wrb; s_wbox[warp][2] = wca; s_wbox[warp][3] = wcb; }
    __syncthreads();
    // staged box of the CTA = hull of the warps' regions
    int ra = 0x7fffffff, rb = -1, ca = 0x7fffffff, cbw = -1;
#pragma unroll
    for (int i = 0; i < 8; ++i)
        if (s_wbox[i][1] >= s_wbox[i][0]) {
            ra = min(ra, s_wbox[i][0]); rb = max(rb, s_wbox[i][1]);
            ca = min(ca, s_wbox[i][2]); cbw = max(cbw, s_wbox[i][3]);
        }
    // TMA needs the box to start on a 16-byte boundary in global memory (measured on B200:
    // an inner coordinate that is not a multiple of 4 words raises an illegal instruction)
    ca &= ~3;

    int acc2[4][4];
    uint32_t ones[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int k = 0; k < 4; ++k) { acc2[i][k] = 0; ones[i][k] = 0u; }

    if (rb >= ra) {
        const int ncols = cbw - ca + 1;
        const int sel = ncols <= maps.bw[0] ? 0 : (ncols <= maps.bw[1] ? 1 : (ncols <= maps.bw[2] ? 2 : 3));
        const int bw = maps.bw[sel], R = maps.rows[sel];
        const int ncb = (ncols + bw - 1) / bw;                 // column blocks (1 unless pitch > 32 words)
        const int nrc = (rb - ra + R) / R;                     // row chunks
        const int nchunks = ncb * nrc;
        const uint32_t tile_bytes = (uint32_t)(R * bw * 4);
        const CUtensorMap* mt = &maps.t[sel];
        const CUtensorMap* mp = &maps.p[sel];
        const uint32_t tiles_s = smem_u32(tiles);

        auto issue = [&](int chunk) {                           // executed by warp 0
            const int st = chunk & 1;
            const int r = ra + (chunk / ncb) * R, c = ca + (chunk % ncb) * bw;
            const uint32_t bar = smem_u32(&bars[st]);
            if (lane == 0) {
                mbar_expect_tx(bar, tile_bytes * kTmaMasks);
                for (int m = 0; m < kTmaTT; ++m)
                    tma_load_2d(tiles_s + (uint32_t)((st * kTmaMasks + m) * kTmaTileWords * 4), mt, c,
                                s_mask_row0[m] + r, bar);
                for (int m = kTmaTT; m < kTmaMasks; ++m)
                    tma_load_2d(tiles_s + (uint32_t)((st * kTmaMasks + m) * kTmaTileWords * 4), mp, c,
                                s_mask_row0[m] + r, bar);
            }
            __syncwarp();
        };

        if (warp == 0) issue(0);
        for (int chunk = 0; chunk < nchunks; ++chunk) {
            if (warp == 0 && chunk + 1 < nchunks) issue(chunk + 1);
            mbar_wait(smem_u32(&bars[chunk & 1]), (uint32_t)((chunk >> 1) & 1));
            // this warp's rows / columns inside the staged box (rows past the image belong to another mask)
            const int r0 = ra + (chunk / ncb) * R, c0 = ca + (chunk % ncb) * bw;
            const int ya = max(wra, r0), yb = min(min(wrb, r0 + R - 1), H - 1);
            const int xa = max(wca, c0), xb = min(wcb, c0 + bw - 1);
            if (yb >= ya && xb >= xa) {
                const int ncw = xb - xa + 1;
                const int total = (yb - ya + 1) * ncw;
                const uint32_t* st = tiles + (size_t)(chunk & 1) * kTmaMasks * kTmaTileWords;
                const uint32_t* tbase = st + (size_t)tw * kTmaTileWords + (ya - r0) * bw + (xa - c0);
                const uint32_t* pbase = st + (size_t)(kTmaTT + cw) * kTmaTileWords + (ya - r0) * bw + (xa - c0);
                const int dr = 64 / ncw, dc = 64 - dr * ncw;
                int rA = lane / ncw, cA = lane - rA * ncw;
                int rB = (lane + 32) / ncw, cB = (lane + 32) - rB * ncw;
                for (int idx = lane; idx < total; idx += 64) {
                    const int oA = rA * bw + cA;
                    const bool hasB = idx + 32 < total;
                    const int oB = hasB ? rB * bw + cB : oA;
                    uint32_t tA[4], pA[4], tB[4], pB[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        tA[i] = tbase[i * kTmaTileWords + oA]; pA[i] = pbase[i * kTmaTileWords + oA];
                        tB[i] = tbase[i * kTmaTileWords + oB]; pB[i] = pbase[i * kTmaTileWords + oB];
                    }
                    if (!hasB) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) tB[i] = 0u;
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int k = 0; k < 4; ++k) csa_step(tA[i] & pA[k], tB[i] & pB[k], ones[i][k], acc2[i][k]);
                    rA += dr; cA += dc;
                    if (cA >= ncw) { cA -= ncw; ++rA; }
                    rB += dr; cB += dc;
                    if (cB >= ncw) { cB -= ncw; ++rB; }
                }
            }
            __syncthreads();                                    // stage may be refilled by the next issue
        }
    }
    if (!active) return;

    int acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int k = 0; k < 4; ++k)
            acc[i][k] = __reduce_add_sync(0xffffffffu, 2 * acc2[i][k] + __popc(ones[i][k]));

    if (lane == 0) {
        const int t0 = tb + tw, c0 = cb + cw;
        const int nt = min(4, job.n_tgt - t0), ncd = min(4, job.n_cand - c0);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (i >= nt) break;
            const int pt = tgt_popc[tgt_index[job.tgt_begin + t0 + i]];
            unsigned long long best = 0ull;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (k >= ncd) break;
                const int inter = acc[i][k];
                const int uni = pt + proj_popc[(size_t)job.cand_begin + c0 + k] - inter;
                const float iou = __fdiv_rn((float)inter, (float)uni);
                const unsigned long long key = make_key(iou, c0 + k, inter, packed);
                best = key > best ? key : best;
                if (inter_tab) inter_tab[job.tab_begin + (int64_t)(t0 + i) * job.n_cand + c0 + k] = inter;
            }
            atomicMax(key_ws + job.tgt_begin + t0 + i, best);
        }
    }
}

// ---------------------------------------------------------------------------
// score on the tensor cores.  inter[t][c] = sum over pixels of T_t[p] * P_c[p] is a dense
// contraction with 1-bit operands: a (targets x pixels) . (pixels x candidates) product.  Blackwell
// has no 1-bit MMA (mma.sync .b1 is emulated with IMMA on sm_100a), so the words of the overlap
// region are expanded to 4-bit e2m1 values (bit -> 0x2 = 1.0) in shared memory and fed to
// tcgen05.mma kind::mxf4 with every UE8M0 block scale 1.0: each product is exactly 0 or 1 and the
// f32 accumulator of the 128 x N tile in tensor memory holds every count below 2^24 exactly
// (tools/mma_probe.cu checks this past 2^21; a3d_score takes k_score for frames over 2^24 pixels).
//   * CTA = (job, 128 targets, N <= 240 candidates); region = (hull of its target boxes) ∩ (hull of
//     its candidate boxes), walked as one row-major sequence of word positions, 16 per step.
//   * 24 producer warps: thread -> (word of the step, up to 8 masks).  One 4-byte load per word, issued
//     2 steps ahead of its use (register ring, static indices through unrolling); 4 shift+mask ops turn
//     the word into 16 bytes of nibbles (nibble i of register j = bit 4i+j — any permutation serves as
//     long as both operands use it); one 16-byte store into the no-swizzle K-major core-matrix layout
//     [word position][row][16 B]; fence.proxy.async; arrive on the stage's full barrier.
//   * one thread issues one MMA (K = 64 = two word positions: LBO = the position slot, SBO = 128;
//     tools/mma_probe.cu pins the fields) per position pair of the step and commits the stage back to
//     the producers (2 stages of 16 positions).  An odd last position is paired with zeros.
//   * block scales: 0x7F (2^0) in every byte of TMEM columns 256..511, written once per CTA.
//   * epilogue: warps 0-3 read their 32 TMEM lanes (= targets) with tcgen05.ld, and every thread
//     scans its target's candidates: union, fp32 divide, arg-max key, one atomicMax per target.
// Bound (DESIGN.md §4): shared-memory bandwidth — every mask bit crosses shared memory as a nibble
// twice (producer store, tensor-core operand read: 2 x 5 KB per word position at N = 192).
// ---------------------------------------------------------------------------
#ifndef A3D_MMA_WARPS
#define A3D_MMA_WARPS 24
#endif
#ifndef A3D_MMA_AHEAD
#define A3D_MMA_AHEAD 2
#endif
#ifndef A3D_MMA_POS
#define A3D_MMA_POS 16
#endif
#ifndef A3D_MMA_STAGES
#define A3D_MMA_STAGES 2
#endif
constexpr int kMmaProducerWarps = A3D_MMA_WARPS;
constexpr int kMmaProducers = 32 * kMmaProducerWarps;
constexpr int kMmaThreads = kMmaProducers + 32;   // + the issuing warp
constexpr int kMmaM = 128;                    // targets per CTA (TMEM lanes)
constexpr int kMmaNMax = 240;                 // candidates per CTA (TMEM columns), multiple of 16
constexpr int kMmaStages = A3D_MMA_STAGES;
constexpr int kMmaPos = A3D_MMA_POS;          // word positions per stage (two per MMA)
constexpr int kMmaItems = ((kMmaM + kMmaNMax) * kMmaPos + kMmaProducers - 1) / kMmaProducers;   // words per producer thread per step
constexpr int kMmaTmemCols = 512;             // accumulator in columns 0..255, block scales in 256..511
constexpr int kMmaSfCol = 256;
constexpr int kMmaAhead = A3D_MMA_AHEAD;                  // steps between a producer's loads and its stores
static_assert(kMmaPos >= 2 && (kMmaPos & (kMmaPos - 1)) == 0 && kMmaProducers % kMmaPos == 0,
              "positions of a step pair up into MMAs; a thread's word is tid & (kMmaPos - 1)");

// position slots of one stage are padded so that the 16-byte stores of a quarter-warp (8 positions
// of one mask, or 4 positions of two masks) hit distinct banks
constexpr int kMmaPad = kMmaPos >= 8 ? 16 : 32;
__host__ __device__ constexpr size_t mma_stage_bytes(int nb) {
    return (size_t)kMmaPos * (kMmaM * 16 + kMmaPad) + (size_t)kMmaPos * (nb * 16 + kMmaPad);
}

// bounded wait: a broken pipeline traps (launch error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait_bounded(uint32_t bar, uint32_t parity) {
    uint32_t ok, spins = 0;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (!ok && ++spins > (1u << 24)) __trap();
    } while (!ok);
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes) {
    // K-major, no swizzle: start >> 4 | LBO >> 4 (K-chunk stride) | SBO >> 4 = 8 (8-row group stride 128 B) | version 1
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)8 << 32) | (1ull << 46);
}
__device__ __forceinline__ void expand_store(uint32_t w, uint32_t dst) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"((w << 1) & 0x22222222u), "r"(w & 0x22222222u),
                 "r"((w >> 1) & 0x22222222u), "r"((w >> 2) & 0x22222222u) : "memory");
}

__global__ void __launch_bounds__(kMmaThreads, 1)
k_score_mma(const a3d_job_t* __restrict__ jobs, int H, int pitch, int tt_tiles, int ct_tiles, int ctile,
            const uint32_t* __restrict__ tgt_bits, const int32_t* __restrict__ tgt_popc,
            const int32_t* __restrict__ tgt_bbox, const int32_t* __restrict__ tgt_index,
            const uint32_t* __restrict__ proj_bits, const int32_t* __restrict__ proj_popc,
            const int32_t* __restrict__ proj_bbox, unsigned long long* __restrict__ key_ws,
            int32_t* __restrict__ inter_tab, int packed) {
    extern __shared__ __align__(1024) uint8_t stage_mem[];
    __shared__ const uint32_t* s_ptr[kMmaM + kMmaNMax];       // first word of every mask of the tile
    __shared__ int s_pc[kMmaNMax];                            // pixel counts of the candidates
    __shared__ int s_box[8];                                  // target hull, candidate hull
    __shared__ __align__(8) uint64_t s_bar[2 * kMmaStages + 1];
    __shared__ uint32_t s_tmem;

    const int per_job = tt_tiles * ct_tiles;
    const int jid = blockIdx.x / per_job;
    const int rem = blockIdx.x - jid * per_job;
    const a3d_job_t job = jobs[jid];
    const int tb = (rem / ct_tiles) * kMmaM;
    const int cb = (rem % ct_tiles) * ctile;
    if (tb >= job.n_tgt || cb >= job.n_cand) return;           // whole CTA leaves together
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nt = min(kMmaM, job.n_tgt - tb), nc = min(ctile, job.n_cand - cb);
    pdl_wait();
    pdl_launch_dependents();
    const int nb = (nc + 15) & ~15;                            // MMA N
    const size_t words = (size_t)H * pitch;

    if (tid < 8) s_box[tid] = (tid & 1) ? -1 : 0x7fffffff;     // {r0, r1, c0, c1} x {targets, candidates}
    if (tid == 0) {
        for (int i = 0; i < kMmaStages; ++i) {
#ifdef A3D_MMA_WARP_ARRIVE
            mbar_init(smem_u32(&s_bar[i]), kMmaProducerWarps);             // full: one arrive per producer warp
#else
            mbar_init(smem_u32(&s_bar[i]), kMmaProducers);                 // full: every producer thread arrives
#endif
            mbar_init(smem_u32(&s_bar[kMmaStages + i]), 1);                // empty: one tcgen05.commit
        }
        mbar_init(smem_u32(&s_bar[2 * kMmaStages]), 1);                    // accumulator complete
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kMmaProducerWarps) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "r"(kMmaTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (warp < 4) {
        // block scales: every byte of columns kMmaSfCol.. of the warp's 32 lanes = 0x7F (UE8M0 2^0)
        const uint32_t one = 0x7F7F7F7Fu;
#pragma unroll
        for (int c = kMmaSfCol; c < kMmaTmemCols; c += 8)
            asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};"
                         ::"r"(s_tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c), "r"(one) : "memory");
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    for (int m = tid; m < nt + nc; m += kMmaThreads) {
        const int32_t* b;
        if (m < nt) {
            const int ti = tgt_index[job.tgt_begin + tb + m];
            s_ptr[m] = tgt_bits + (size_t)ti * words;
            b = tgt_bbox + 4 * (size_t)ti;
        } else {
            const size_t g = (size_t)job.cand_begin + cb + (m - nt);
            s_ptr[m] = proj_bits + g * words;
            s_pc[m - nt] = proj_popc[g];
            b = proj_bbox + 4 * g;
        }
        if (b[1] >= b[0]) {
            int* box = s_box + (m < nt ? 0 : 4);
            atomicMin(box + 0, b[0]); atomicMax(box + 1, b[1]); atomicMin(box + 2, b[2]); atomicMax(box + 3, b[3]);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = s_tmem;

    // region = (hull of the target boxes) ∩ (hull of the candidate boxes), walked as one row-major
    // sequence of word positions; a step = kMmaPos consecutive positions = kMmaPos / 2 MMAs
    const int ra = max(s_box[0], s_box[4]), rb = min(s_box[1], s_box[5]);
    const int ca = max(s_box[2], s_box[6]), ce = min(s_box[3], s_box[7]);
    int npos = 0, ncols = 1;
    if (rb >= ra && ce >= ca) {
        ncols = ce - ca + 1;
        npos = (rb - ra + 1) * ncols;
    }
    const int nsteps = (npos + kMmaPos - 1) / kMmaPos;
    const uint32_t stage0 = smem_u32(stage_mem);
    const uint32_t stage_bytes = (uint32_t)mma_stage_bytes(nb);
    const uint32_t a_slot = (uint32_t)(kMmaM * 16 + kMmaPad), b_slot = (uint32_t)(nb * 16 + kMmaPad);
    const uint32_t b_off = (uint32_t)kMmaPos * a_slot;
    const uint32_t bar0 = smem_u32(&s_bar[0]);

    if (warp < kMmaProducerWarps) {
        // ===== producers =====
        // thread -> word q of the step, for the masks tid / kMmaPos + (kMmaProducers / kMmaPos) u: one
        // position cursor per thread, a constant stage slot per (thread, u).  Loads run kMmaAhead steps
        // ahead of the stores in a register ring (static indices through full unrolling).  Positions past
        // the region load as zeros, so an odd last position pairs with a zero chunk.
        const int nmask = nt + nc;
        const int npos2 = (npos + 1) & ~1;
        const int q = tid & (kMmaPos - 1);
        const uint32_t* src[kMmaItems];             // word (ra, ca) of this thread's masks
        uint32_t dst[kMmaItems];                    // byte offset of the mask's 16-byte row slot inside a stage
        bool act[kMmaItems];
#pragma unroll
        for (int u = 0; u < kMmaItems; ++u) {
            const int m = tid / kMmaPos + u * (kMmaProducers / kMmaPos);
            act[u] = m < nmask;
            src[u] = act[u] ? s_ptr[m] + (size_t)ra * pitch + ca : nullptr;
            dst[u] = m < nt ? (uint32_t)q * a_slot + (uint32_t)m * 16u
                            : b_off + (uint32_t)q * b_slot + (uint32_t)(m - nt) * 16u;
        }
        // position of this thread's word in the step the load cursor is at: p = kMmaPos k + q = row * ncols + col
        const int dr = kMmaPos / ncols, dc = kMmaPos - dr * ncols;
        int p_ld = q, col = q % ncols;
        unsigned rowoff = (unsigned)((q / ncols) * pitch);
        auto load_step = [&](uint32_t (&w)[kMmaItems]) {
            const unsigned o = rowoff + (unsigned)col;
            const bool in = p_ld < npos;
#pragma unroll
            for (int u = 0; u < kMmaItems; ++u)
                if (act[u]) w[u] = in ? __ldg(src[u] + o) : 0u;
            p_ld += kMmaPos;
            col += dc;
            rowoff += (unsigned)(dr * pitch);
            if (col >= ncols) { col -= ncols; rowoff += (unsigned)pitch; }
        };
        int p_st = q;
        auto store_step = [&](int st, uint32_t parity, const uint32_t (&w)[kMmaItems]) {
            const uint32_t sa = stage0 + (uint32_t)st * stage_bytes;
            mbar_wait_bounded(bar0 + 8u * (uint32_t)(kMmaStages + st), parity ^ 1u);
            if (p_st < npos2) {
#pragma unroll
                for (int u = 0; u < kMmaItems; ++u)
                    if (act[u]) expand_store(w[u], sa + dst[u]);
            }
            p_st += kMmaPos;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy stores -> async-proxy (MMA) reads
#ifdef A3D_MMA_WARP_ARRIVE
            __syncwarp();
            if (lane == 0) mbar_arrive(bar0 + 8u * (uint32_t)st);
#else
            mbar_arrive(bar0 + 8u * (uint32_t)st);
#endif
        };
        static_assert(kMmaAhead % kMmaStages == 0, "the stage of a step must be static in the unrolled loop");
        uint32_t ring[kMmaAhead][kMmaItems];
#pragma unroll
        for (int d = 0; d < kMmaAhead - 1; ++d)
            if (d < nsteps) load_step(ring[d]);
        for (int k0 = 0; k0 < nsteps; k0 += kMmaAhead) {
#pragma unroll
            for (int d = 0; d < kMmaAhead; ++d) {
                const int k = k0 + d;
                if (k < nsteps) {
                    if (k + kMmaAhead - 1 < nsteps) load_step(ring[(d + kMmaAhead - 1) % kMmaAhead]);
                    store_step(d % kMmaStages, (uint32_t)((k / kMmaStages) & 1), ring[d]);
                }
            }
        }
    } else if (lane == 0) {
        // ===== MMA issuer (one thread) =====
        // e2m1 x e2m1 -> f32, UE8M0 block scales, K-major
        const uint32_t idesc = (1u << 7) | (1u << 10) | ((uint32_t)(nb >> 3) << 17) | (1u << 23) | ((uint32_t)(kMmaM >> 4) << 24);
        const uint32_t sfa = tmem + (uint32_t)kMmaSfCol, sfb = sfa + 128u;
        for (int k = 0; k < nsteps; ++k) {
            const int st = k % kMmaStages;
            const int nmma = (min(kMmaPos, npos - k * kMmaPos) + 1) >> 1;
            const uint32_t sa = stage0 + (uint32_t)st * stage_bytes, sb = sa + b_off;
            mbar_wait_bounded(bar0 + 8u * (uint32_t)st, (uint32_t)((k / kMmaStages) & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            for (int j = 0; j < nmma; ++j) {
                const uint64_t da = umma_desc(sa + (uint32_t)(2 * j) * a_slot, a_slot);
                const uint64_t db = umma_desc(sb + (uint32_t)(2 * j) * b_slot, b_slot);
                const uint32_t acc = (k > 0 || j > 0) ? 1u : 0u;
                asm volatile(
                    "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %6, 0;\n\t"
                    "tcgen05.mma.cta_group::1.kind::mxf4.block_scale.scale_vec::2X [%0], %1, %2, %3, [%4], [%5], p;\n\t}"
                    ::"r"(tmem), "l"(da), "l"(db), "r"(idesc), "r"(sfa), "r"(sfb), "r"(acc) : "memory");
            }
            // arrives on the stage's empty barrier once these MMAs have read shared memory
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                         ::"r"(bar0 + 8u * (uint32_t)(kMmaStages + st)) : "memory");
        }
        if (nsteps > 0)
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                         ::"r"(bar0 + 8u * (uint32_t)(2 * kMmaStages)) : "memory");
    }

    if (warp < 4) {
        // ===== epilogue: TMEM lane = target, column = candidate =====
        if (nsteps > 0) {
            mbar_wait_bounded(bar0 + 8u * (uint32_t)(2 * kMmaStages), 0u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        const int m = warp * 32 + lane;
        const bool valid = m < nt;
        const int pt = valid ? tgt_popc[tgt_index[job.tgt_begin + tb + m]] : 0;
        unsigned long long best = 0ull;
        for (int c0 = 0; c0 < nb; c0 += 16) {
            uint32_t v[16];
            if (nsteps > 0) {
                const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0;
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                    : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                      "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                    : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = 0u;
            }
            if (valid) {
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int c = c0 + j;
                    if (c < nc) {
                        const int inter = __float2int_rn(__uint_as_float(v[j]));   // an integer, at most 2^24
                        const int uni = pt + s_pc[c] - inter;
                        const float iou = __fdiv_rn((float)inter, (float)uni);
                        const unsigned long long key = make_key(iou, cb + c, inter, packed);
                        best = key > best ? key : best;
                        if (inter_tab) inter_tab[job.tab_begin + (int64_t)(tb + m) * job.n_cand + cb + c] = inter;
                    }
                }
            }
        }
        if (valid) atomicMax(key_ws + job.tgt_begin + tb + m, best);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == kMmaProducerWarps) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kMmaTmemCols));
}

// decode the winning candidate of every target.  Packed keys carry the intersection count
// (one thread per target); otherwise one warp per target recomputes it over the candidate's box.
__global__ void __launch_bounds__(256)
k_finalize(const a3d_job_t* __restrict__ jobs, int H, int pitch,
           const uint32_t* __restrict__ tgt_bits, const int32_t* __restrict__ tgt_popc,
           const int32_t* __restrict__ tgt_index, const uint32_t* __restrict__ proj_bits,
           const int32_t* __restrict__ proj_popc, const int32_t* __restrict__ proj_bbox,
           const unsigned long long* __restrict__ key_ws, int32_t* __restrict__ best_cand,
           int32_t* __restrict__ best_inter, int32_t* __restrict__ best_union,
           float* __restrict__ best_iou, int packed) {
    const a3d_job_t job = jobs[blockIdx.x];
    pdl_wait();                       // the arg-max keys of the scoring kernel
    if (packed) {
        for (int t = blockIdx.y * blockDim.x + threadIdx.x; t < job.n_tgt; t += gridDim.y * blockDim.x) {
            const size_t slot = (size_t)job.tgt_begin + t;
            const unsigned lo = (unsigned)(key_ws[slot] & 0xffffffffull);
            const int cand = (int)(0xfffu - (lo >> 20)), inter = (int)(lo & 0xfffffu);
            const int uni = tgt_popc[tgt_index[slot]] + proj_popc[(size_t)job.cand_begin + cand] - inter;
            best_cand[slot] = cand;
            best_inter[slot] = inter;
            best_union[slot] = uni;
            best_iou[slot] = __fdiv_rn((float)inter, (float)uni);
        }
        return;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const size_t words = (size_t)H * pitch;
    for (int t = blockIdx.y * nw + warp; t < job.n_tgt; t += gridDim.y * nw) {
        const size_t slot = (size_t)job.tgt_begin + t;
        const unsigned long long key = key_ws[slot];
        const int cand = (int)(~(unsigned)(key & 0xffffffffull));
        const size_t g = (size_t)job.cand_begin + cand;
        const int tm = tgt_index[slot];
        const uint32_t* tp = tgt_bits + (size_t)tm * words;
        const uint32_t* pp = proj_bits + g * words;
        const int32_t* pb = proj_bbox + 4 * g;
        int inter = 0;
        if (pb[1] >= pb[0]) {
            const int ncols = pb[3] - pb[2] + 1;
            const int total = (pb[1] - pb[0] + 1) * ncols;
            for (int idx = lane; idx < total; idx += 32) {
                const int r = idx / ncols, c = idx - r * ncols;
                const int o = (pb[0] + r) * pitch + pb[2] + c;
                inter += __popc(__ldg(tp + o) & __ldg(pp + o));
            }
        }
        inter = __reduce_add_sync(0xffffffffu, inter);
        if (lane == 0) {
            const int uni = tgt_popc[tm] + proj_popc[g] - inter;
            best_cand[slot] = cand;
            best_inter[slot] = inter;
            best_union[slot] = uni;
            best_iou[slot] = __fdiv_rn((float)inter, (float)uni);
        }
    }
}

// ---------------------------------------------------------------------------
// rle_to_bits: COCO run-length masks (column-major runs, alternating 0/1, starting
// with 0) -> row-major bit-packed masks, one CTA per mask.  The packed image is
// assembled in shared memory: runs are taken 256 at a time (block prefix sum of the
// lengths), each warp then paints whole runs, one lane per pixel.
// Replaces pycocotools' mask_util.decode in create_instances (utils/arti_vis.py:182).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_rle_to_bits(const uint32_t* __restrict__ counts, const int64_t* __restrict__ begin, int H, int W, int pitch,
              uint32_t* __restrict__ bits) {
    extern __shared__ __align__(16) uint32_t img[];          // [H][pitch]
    __shared__ unsigned long long s_start[256];
    __shared__ uint32_t s_len[256];
    __shared__ unsigned long long s_warp[8];
    __shared__ unsigned long long s_base;
    const int words = H * pitch;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < words; i += 256) img[i] = 0u;
    if (threadIdx.x == 0) s_base = 0ull;
    __syncthreads();
    const int64_t b0 = begin[blockIdx.x], nruns = begin[blockIdx.x + 1] - b0;
    const unsigned long long npix = (unsigned long long)H * W;
    for (int64_t c0 = 0; c0 < nruns; c0 += 256) {
        const int64_t r = c0 + threadIdx.x;
        const uint32_t len = r < nruns ? counts[b0 + r] : 0u;
        unsigned long long incl = len;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += v;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        unsigned long long off = s_base;
        for (int i = 0; i < warp; ++i) off += s_warp[i];
        s_start[threadIdx.x] = off + incl - len;
        s_len[threadIdx.x] = (r & 1) ? len : 0u;             // odd runs are the ones
        __syncthreads();
        for (int k = warp; k < 256; k += 8) {
            const uint32_t L = s_len[k];
            if (L == 0) continue;
            const unsigned long long st = s_start[k];
            for (unsigned long long i = st + lane; i < st + L && i < npix; i += 32) {
                const int x = (int)(i / (unsigned)H), y = (int)(i - (unsigned long long)x * H);
                atomicOr(&img[y * pitch + (x >> 5)], 1u << (x & 31));
            }
        }
        __syncthreads();
        if (threadIdx.x == 255) s_base = off + incl;
        __syncthreads();
    }
    uint32_t* out = bits + (size_t)blockIdx.x * words;
    for (int i = threadIdx.x; i < words; i += 256) out[i] = img[i];
}

// ---------------------------------------------------------------------------
// plane_offsets: per instance, mean over the mask of n . (ray * depth) — the plane
// offset the detector's depth map implies (override_depth, utils/arti_vis.py:125-149).
// One CTA per instance walks the mask's bounding box, one warp per packed word, one
// lane per pixel; X = ray_x*depth etc. are fp32 products as in depth2XYZ (:90-99),
// the dot product is separately rounded fp32, the sum is carried in fp64.
// Streams depth (4 B/px) + the ray table (12 B/px, L2-resident) once per instance.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_plane_offsets(const float* __restrict__ depth, const float* __restrict__ rays, int H, int W, int pitch,
                const uint32_t* __restrict__ bits, const int32_t* __restrict__ bbox,
                const int32_t* __restrict__ inst_mask, const int32_t* __restrict__ inst_frame,
                const float* __restrict__ normals, float* __restrict__ offset_out, int32_t* __restrict__ count_out) {
    __shared__ double s_sum[8];
    __shared__ int s_cnt[8];
    const int inst = blockIdx.x;
    const int m = inst_mask[inst];
    const int32_t* b = bbox + 4 * (size_t)m;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double sum = 0.0;
    int cnt = 0;
    if (b[1] >= b[0]) {
        const uint32_t* mb = bits + (size_t)m * H * pitch;
        const size_t plane = (size_t)H * W;
        const float* d = depth ? depth + (size_t)inst_frame[inst] * plane : nullptr;
        const float n0 = normals[3 * inst], n1 = normals[3 * inst + 1], n2 = normals[3 * inst + 2];
        const int ncols = b[3] - b[2] + 1, nwords = (b[1] - b[0] + 1) * ncols;
        for (int w = warp; w < nwords; w += 8) {
            const int rr = w / ncols;
            const int row = b[0] + rr, wc = b[2] + (w - rr * ncols);
            const uint32_t word = mb[row * pitch + wc];
            const int x = wc * 32 + lane;
            if (((word >> lane) & 1u) && x < W) {
                const size_t o = (size_t)row * W + x;
                const float dz = d ? d[o] : 1.0f;
                const float X = __fmul_rn(rays[o], dz), Y = __fmul_rn(rays[plane + o], dz),
                            Z = __fmul_rn(rays[2 * plane + o], dz);
                sum += (double)__fadd_rn(__fadd_rn(__fmul_rn(n0, X), __fmul_rn(n1, Y)), __fmul_rn(n2, Z));
                ++cnt;
            }
        }
    }
#pragma unroll
    for (int dlt = 16; dlt > 0; dlt >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, dlt);
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) { s_sum[warp] = sum; s_cnt[warp] = cnt; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        int c = 0;
        for (int i = 0; i < 8; ++i) { t += s_sum[i]; c += s_cnt[i]; }
        count_out[inst] = c;
        offset_out[inst] = c > 0 ? (float)(t / (double)c) : 0.f;
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
k_emit(const uint32_t* __restrict__ bits, const int32_t* __restrict__ index, int H, int W, int pitch,
       T* __restrict__ out) {
    const int64_t i = blockIdx.y;
    const int64_t m = index ? index[i] : i;
    const uint32_t* b = bits + m * (int64_t)H * pitch;
    T* o = out + i * (int64_t)H * W;
    const int npx = H * W;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < npx; p += gridDim.x * blockDim.x) {
        const int r = p / W, x = p - r * W;
        o[p] = (T)((b[r * pitch + (x >> 5)] >> (x & 31)) & 1u);
    }
}

// ---------------------------------------------------------------------------
// bits -> COCO RLE (column-major runs, alternating 0/1, starting with 0s).
// A run boundary sits at flat position p = x*H + y wherever pixel (y, x) differs from its column-major
// predecessor: (y-1, x) for y >= 1, (H-1, x-1) for y == 0, a virtual 0 for (0, 0) (a set first pixel opens
// with an empty 0-run).  As packed words that is the transition row D[y] = R[y] ^ R[y-1], and for row 0
// D[0] = R[0] ^ (R[H-1] shifted up by one pixel, bit 31 of word j-1 carried into bit 0 of word j, a 0 into
// pixel 0); only the W valid bits of every row are read or kept.  A mask has popc(D) + 1 runs; the runs are
// the differences of consecutive boundary positions, with 0 as the first bound and H*W as the last.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t rle_valid(int j, int W) {
    const int left = W - 32 * j;
    return left >= 32 ? 0xffffffffu : ((1u << left) - 1u);
}

// transition word D[y][j] of one packed mask
__device__ __forceinline__ uint32_t rle_transitions(const uint32_t* __restrict__ b, int H, int W, int pitch, int y, int j) {
    const uint32_t valid = rle_valid(j, W);
    const uint32_t r = b[(int64_t)y * pitch + j] & valid;
    uint32_t prev;
    if (y > 0) {
        prev = b[(int64_t)(y - 1) * pitch + j] & valid;
    } else {
        const uint32_t* last = b + (int64_t)(H - 1) * pitch;
        prev = ((last[j] & valid) << 1) | (j > 0 ? last[j - 1] >> 31 : 0u);
    }
    return (r ^ prev) & valid;
}

// runs_out[i] = popc(D) + 1 of mask index[i]; one CTA per mask (grid-stride), coalesced over the mask's words
__global__ void __launch_bounds__(256)
k_rle_count(const uint32_t* __restrict__ bits, const int32_t* __restrict__ index, int64_t n, int H, int W, int pitch,
            int64_t* __restrict__ runs_out) {
    __shared__ int64_t s_sum[8];
    const int nw = (W + 31) >> 5;
    const int64_t words = (int64_t)H * nw;
    for (int64_t i = blockIdx.x; i < n; i += gridDim.x) {
        const uint32_t* b = bits + (index ? (int64_t)index[i] : i) * H * pitch;
        int64_t c = 0;
        for (int64_t w = threadIdx.x; w < words; w += blockDim.x) {
            const int y = (int)(w / nw), j = (int)(w - (int64_t)y * nw);
            c += __popc(rle_transitions(b, H, W, pitch, y, j));
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
        if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = c;
        __syncthreads();
        if (threadIdx.x == 0) {
            int64_t t = 1;
            for (int k = 0; k < 8; ++k) t += s_sum[k];
            runs_out[i] = t;
        }
        __syncthreads();
    }
}

// The 32x32 tile of D at word column j, rows y0..y0+31, transposed: lane c gets the transition bits of pixel
// column 32j + c, bit r = row y0 + r.  One ballot per column; tiles without a transition return 0 at once.
__device__ __forceinline__ uint32_t rle_tile_column(const uint32_t* __restrict__ b, int H, int W, int pitch, int y0,
                                                    int j, int lane) {
    const int y = y0 + lane;
    const uint32_t d = y < H ? rle_transitions(b, H, W, pitch, y, j) : 0u;
    if (!__any_sync(0xffffffffu, d != 0u)) return 0u;
    uint32_t mine = 0;
#pragma unroll
    for (int c = 0; c < 32; ++c) {
        const uint32_t t = __ballot_sync(0xffffffffu, (d >> c) & 1u);
        if (lane == c) mine = t;
    }
    return mine;
}

// counts_out[begin[i] ..] = runs of mask index[i].  One CTA per mask (grid-stride), one warp per word column;
// the word columns are taken in groups of 8 (one per warp) so that no per-column state needs shared memory
// whatever W is.  Per group: pass 1 counts every pixel column's transitions and finds its last one; a scan
// over lanes, over the group's warps and the carry of the earlier groups gives each lane the rank of its
// first transition and the position of the transition before it; pass 2 re-walks the column and writes the
// differences.  The transposed tiles are re-read rather than kept (L1 / L2 hits: a 640x480 mask is 38 KB).
constexpr int kRleWarps = 8;
__global__ void __launch_bounds__(kRleWarps * 32)
k_bits_to_rle(const uint32_t* __restrict__ bits, const int32_t* __restrict__ index, int64_t n, int H, int W,
              int pitch, const int64_t* __restrict__ begin, uint32_t* __restrict__ counts_out) {
    __shared__ int64_t s_cnt[kRleWarps];
    __shared__ int64_t s_last[kRleWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nw = (W + 31) >> 5;
    for (int64_t i = blockIdx.x; i < n; i += gridDim.x) {
        const uint32_t* b = bits + (index ? (int64_t)index[i] : i) * H * pitch;
        const int64_t out0 = begin[i], n_runs = begin[i + 1] - out0;
        uint32_t* out = counts_out + out0;
        int64_t carry_cnt = 0, carry_last = 0;          // transitions of the earlier groups; position of the last
        for (int g = 0; g < nw; g += kRleWarps) {
            const int j = g + warp;
            const int64_t col0 = (int64_t)(32 * j + lane) * H;     // this lane's pixel column starts here
            // pass 1: transitions of column x and the position of its last one (-1: none)
            int64_t cnt = 0, last = -1;
            if (j < nw) {
                for (int y0 = 0; y0 < H; y0 += 32) {
                    const uint32_t t = rle_tile_column(b, H, W, pitch, y0, j, lane);
                    if (t) {
                        cnt += __popc(t);
                        last = col0 + y0 + 31 - __clz(t);
                    }
                }
            }
            // scans over lanes: transitions before this column, last transition before it
            int64_t incl = cnt, mx = last;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int64_t a = __shfl_up_sync(0xffffffffu, incl, d);
                const int64_t m = __shfl_up_sync(0xffffffffu, mx, d);
                if (lane >= d) { incl += a; mx = m > mx ? m : mx; }
            }
            const int64_t excl = incl - cnt;
            int64_t prev_in_warp = __shfl_up_sync(0xffffffffu, mx, 1);
            if (lane == 0) prev_in_warp = -1;
            if (lane == 31) { s_cnt[warp] = incl; s_last[warp] = mx; }
            __syncthreads();
            int64_t rank = carry_cnt + excl, prev = carry_last;
            for (int k = 0; k < warp; ++k) {
                rank += s_cnt[k];
                prev = s_last[k] > prev ? s_last[k] : prev;
            }
            prev = prev_in_warp > prev ? prev_in_warp : prev;
            // pass 2 (the whole warp, for its ballots): the runs that end at this column's transitions
            if (j < nw && __any_sync(0xffffffffu, cnt > 0)) {
                for (int y0 = 0; y0 < H; y0 += 32) {
                    uint32_t t = rle_tile_column(b, H, W, pitch, y0, j, lane);
                    while (t) {
                        const int r = __ffs(t) - 1;
                        t &= t - 1;
                        const int64_t pos = col0 + y0 + r;
                        if (rank < n_runs - 1) out[rank] = (uint32_t)(pos - prev);
                        prev = pos;
                        ++rank;
                    }
                }
            }
            for (int k = 0; k < kRleWarps; ++k) {
                carry_cnt += s_cnt[k];
                carry_last = s_last[k] > carry_last ? s_last[k] : carry_last;
            }
            __syncthreads();
        }
        if (threadIdx.x == 0 && carry_cnt == n_runs - 1) out[carry_cnt] = (uint32_t)((int64_t)H * W - carry_last);
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// uint32 [rows][pitch] tensor with a {bw, box_rows} box
int encode_mask_map(CUtensorMap* map, const void* base, uint64_t rows, int pitch, int bw, int box_rows) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return fail(A3D_ECUDA, "cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t dims[2] = {(cuuint64_t)pitch, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)pitch * 4};
    const cuuint32_t box[2] = {(cuuint32_t)bw, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(A3D_ECUDA, "cuTensorMapEncodeTiled failed (%d) rows=%llu pitch=%d box=%dx%d", (int)r,
                    (unsigned long long)rows, pitch, bw, box_rows);
    return A3D_OK;
}

int device_smem_optin() {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return 0;
    return v;
}

int device_sm_count() {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
    return v;
}

// A3D_PROJECT_SCHED = cta | persistent: one tile per 1024-thread CTA, or persistent CTAs of two 512-thread
// groups that fetch tiles from a counter (each group holds `tile` candidate slots)
bool project_persistent() {
    const char* e = getenv("A3D_PROJECT_SCHED");
    return e ? !strcmp(e, "persistent") : A3D_PROJECT_PERSISTENT_DEFAULT;
}

size_t project_smem_bytes(int H, int pitch, int tile) {
    const size_t group_words = ((size_t)tile * ((size_t)H * pitch + 12 + 5 + kHF + 1) + 3) & ~(size_t)3;
    return group_words * 4 * (project_persistent() ? 2 : 1);
}

}  // namespace

// ===========================================================================
// C ABI
// ===========================================================================
// kernel launch, optionally as a programmatic dependent of the previous kernel in the stream
template <typename... KArgs, typename... Args>
static cudaError_t launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl,
                          Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

static int project_impl(const a3d_camera_t* cam, const a3d_job_t* jobs, int n_jobs, int max_cand,
                        int tile_cand, const uint32_t* src_bits, const int32_t* src_bbox,
                        const float* xform, float* pcd_ws, int32_t* pcd_count, float* hom_ws,
                        const int32_t* tile_map, int n_tiles,
                        uint32_t* proj_bits, int32_t* proj_popc, int32_t* proj_bbox, void* stream, bool pdl,
                        bool rows_only);
static int score_impl(int H, int W, const a3d_job_t* jobs, int n_jobs, int max_tgt, int max_cand,
                      int64_t n_tgt_total, int64_t n_pool_masks, int64_t n_cand_total,
                      const uint32_t* tgt_bits, const int32_t* tgt_popc, const int32_t* tgt_bbox,
                      const int32_t* tgt_index,
                      const uint32_t* proj_bits, const int32_t* proj_popc, const int32_t* proj_bbox,
                      uint64_t* key_ws, int32_t* inter_tab,
                      int32_t* best_cand, int32_t* best_inter, int32_t* best_union, float* best_iou,
                      void* stream, bool zero_keys, bool pdl);

// a3d_fetch_host_block: grid-stride copy of 16-byte pieces, four independent loads in flight per thread (the
// source is host memory: every load is a PCIe round trip)
__global__ void __launch_bounds__(256) k_fetch_block(uint4* __restrict__ dst, const uint4* __restrict__ src, int64_t n16) {
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n16; i += 4 * stride) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (i + u * stride < n16) v[u] = src[i + u * stride];
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (i + u * stride < n16) dst[i + u * stride] = v[u];
    }
}

extern "C" {

int a3d_version(void) { return A3D_VERSION; }

#ifdef A3D_FILTER_STATS
int a3d_debug_filter_stats(unsigned long long* out4, int reset) {
    if (out4) cudaMemcpyFromSymbol(out4, g_filter_stats, sizeof(unsigned long long) * 4);
    if (reset) { unsigned long long z[4] = {0, 0, 0, 0}; cudaMemcpyToSymbol(g_filter_stats, z, sizeof(z)); }
    return 0;
}
#endif

const char* a3d_last_error_string(void) { return g_err; }

int a3d_pitch_words(int W) { return W > 0 ? pitch_words(W) : 0; }

// Host-side planner of projection CTAs for grids of about one wave (see include/a3d.h).  Cost model in
// point units, from the ncu instruction counts of k_project<filter>: a CTA costs
// kPlanFixed + tile * (kPlanPerCand + points); the job's extra CTA kPlanFixed + kPlanPerCand + 2.5 points.
// HOST helper: unit quaternions -> candidate transforms.  The host builds the candidates of a pass in float64
// exactly as the reference does (pytorch3d axis_angle_to_matrix via quaternions, utils/opt_utils.py:428-431):
// norms, sin / cos and the quaternion come from the same torch calls; what is left — nine entries of ~4
// multiplications and additions each — is IEEE arithmetic that is bit-identical in any order-preserving
// implementation, and as ~40 separate array operations over (sources x candidates) elements it was the largest
// single piece of host time of the public API (30 ms per 8-track video).  One fused pass here, every operation
// rounded separately in the order of the reference expression, the result rounded once to fp32 (what Rotate
// stores) into rows of 12 floats (entries 9..11 left as they are).
int a3d_host_quat_to_xform(const double* q, const double* two_s, int64_t n, float* xform_out) {
    if (n < 0 || (n > 0 && (!q || !two_s || !xform_out))) return fail(A3D_EINVAL, "a3d_host_quat_to_xform: bad argument");
    for (int64_t e = 0; e < n; ++e) {
        const volatile double r = q[4 * e], i = q[4 * e + 1], j = q[4 * e + 2], k = q[4 * e + 3], s = two_s[e];
        const double ii = i * i, jj = j * j, kk = k * k;
        const double ij = i * j, ik = i * k, jk = j * k;
        const double ir = i * r, jr = j * r, kr = k * r;
        float* o = xform_out + 12 * e;
        double t;
        t = jj + kk; t = s * t; o[0] = (float)(1.0 - t);
        t = ij - kr; o[1] = (float)(s * t);
        t = ik + jr; o[2] = (float)(s * t);
        t = ij + kr; o[3] = (float)(s * t);
        t = ii + kk; t = s * t; o[4] = (float)(1.0 - t);
        t = jk - ir; o[5] = (float)(s * t);
        t = ik - jr; o[6] = (float)(s * t);
        t = jk + ir; o[7] = (float)(s * t);
        t = ii + jj; t = s * t; o[8] = (float)(1.0 - t);
    }
    return A3D_OK;
}

// COCO compressed RLE strings -> run lengths (see include/a3d.h; format restated in articulation3d_b200/rle.py).
// The per-mask Python loop this replaces cost 40 us per simple mask — 39 ms per 960-mask clip, more than the
// dense upload of the same clip.
int64_t a3d_host_rle_counts(const uint8_t* chars, const int64_t* begin, int64_t n, uint32_t* counts_out, int64_t cap,
                            int64_t* count_begin_out, int64_t* run_sum_out) {
    if (n < 0 || (n > 0 && (!chars || !begin))) return fail(A3D_EINVAL, "a3d_host_rle_counts: bad argument");
    int64_t total = 0;
    for (int64_t i = 0; i < n; ++i) {
        int64_t p = begin[i];
        const int64_t end = begin[i + 1];
        if (p < 0 || end < p) return fail(A3D_EINVAL, "a3d_host_rle_counts: string %lld: bad offsets", (long long)i);
        if (count_begin_out) count_begin_out[i] = total;
        int64_t m = 0, sum = 0;
        long long prev1 = 0, prev2 = 0;                 // counts m-1 and m-2 (before the cast to uint32)
        while (p < end) {
            unsigned long long x = 0;
            int k = 0;
            for (;;) {
                if (p >= end || k > 12) return fail(A3D_EINVAL, "a3d_host_rle_counts: string %lld is truncated or malformed", (long long)i);
                const unsigned c = (unsigned)chars[p++] - 48u;
                x |= (unsigned long long)(c & 0x1Fu) << (5 * k);
                ++k;
                if (!(c & 0x20u)) {
                    if (c & 0x10u) x |= ~0ULL << (5 * k);        // sign extension from bit 4 of the last group
                    break;
                }
            }
            long long v = (long long)x;
            if (m > 2) v += prev2;                      // counts beyond the third are differences to the count two back
            prev2 = prev1;
            prev1 = v;
            if (counts_out) {
                if (total >= cap) return fail(A3D_EINVAL, "a3d_host_rle_counts: counts_out holds %lld, more are needed", (long long)cap);
                counts_out[total] = (uint32_t)v;
            }
            sum += (int64_t)(uint32_t)v;
            ++total;
            ++m;
        }
        if (run_sum_out) run_sum_out[i] = sum;
    }
    if (count_begin_out) count_begin_out[n] = total;
    return total;
}

// Run lengths -> COCO compressed strings (the inverse of a3d_host_rle_counts; rle.counts_to_string restated):
// from the fourth count of a mask on, the count is stored as its difference to the count two places back (signed,
// 64-bit), each
// value as 5-bit groups, least significant first, 0x20 = more groups follow, +48; the last group's bit 4 is the
// sign.
int64_t a3d_host_rle_strings(const uint32_t* counts, const int64_t* begin, int64_t n, uint8_t* chars_out,
                             int64_t cap, int64_t* char_begin_out) {
    if (n < 0 || cap < 0 || (n > 0 && (!counts || !begin)) || (cap > 0 && !chars_out))
        return fail(A3D_EINVAL, "a3d_host_rle_strings: bad argument");
    int64_t p = 0;
    for (int64_t i = 0; i < n; ++i) {
        const int64_t b = begin[i], e = begin[i + 1];
        if (b < 0 || e < b) return fail(A3D_EINVAL, "a3d_host_rle_strings: mask %lld: bad offsets", (long long)i);
        if (char_begin_out) char_begin_out[i] = p;
        for (int64_t k = b; k < e; ++k) {
            int64_t x = (int64_t)counts[k];
            if (k - b > 2) x -= (int64_t)counts[k - 2];
            for (bool more = true; more;) {
                unsigned c = (unsigned)(x & 0x1f);
                x >>= 5;                                    // arithmetic: the sign is kept
                more = (c & 0x10u) ? x != -1 : x != 0;
                if (more) c |= 0x20u;
                if (p >= cap) return fail(A3D_EINVAL, "a3d_host_rle_strings: chars_out holds %lld bytes, more are needed", (long long)cap);
                chars_out[p++] = (uint8_t)(c + 48);
            }
        }
    }
    if (char_begin_out) char_begin_out[n] = p;
    return p;
}

int a3d_plan_tiles(const a3d_job_t* jobs_host, int n_jobs, int tile_max, int sm_count, int32_t* tile_map_out,
                   int cap_tiles, int* tile_cand_out) {
    const double kPlanFixed = 21500.0, kPlanPerCand = 3000.0;
    if (n_jobs < 0 || tile_max < 1 || sm_count < 1 || !tile_cand_out || (n_jobs > 0 && !jobs_host))
        return fail(A3D_EINVAL, "a3d_plan_tiles: bad argument");
    *tile_cand_out = tile_max;
    if (n_jobs == 0) return 0;
    long long min_ctas = 0;
    for (int j = 0; j < n_jobs; ++j) {
        if (jobs_host[j].n_cand < 0) return fail(A3D_EINVAL, "a3d_plan_tiles: job %d has n_cand < 0", j);
        min_ctas += (jobs_host[j].n_cand + tile_max - 1) / tile_max;
    }
    const int waves = (min_ctas + n_jobs <= sm_count) ? 1 : 2;
    if (min_ctas + n_jobs > (long long)waves * sm_count) return 0;           // several waves anyway: uniform tiles
    const long long cap = (long long)waves * sm_count - n_jobs;
    if (!tile_map_out || cap_tiles < waves * sm_count) return fail(A3D_EINVAL, "a3d_plan_tiles: tile_map_out too small");
    auto cost = [&](int j) { return (double)jobs_host[j].pcd_cap + kPlanPerCand; };
    auto tile_of = [&](int j, double w) {
        const double t = floor(w / cost(j));
        return t < 1.0 ? 1 : (t > tile_max ? tile_max : (int)t);
    };
    double lo = cost(0), hi = cost(0);
    for (int j = 1; j < n_jobs; ++j) { lo = cost(j) < lo ? cost(j) : lo; hi = cost(j) > hi ? cost(j) : hi; }
    hi *= tile_max;
    for (int it = 0; it < 40; ++it) {                  // smallest per-CTA budget whose CTAs fit the wave(s)
        const double mid = 0.5 * (lo + hi);
        long long ctas = 0;
        for (int j = 0; j < n_jobs; ++j) {
            const int t = tile_of(j, mid);
            ctas += (jobs_host[j].n_cand + t - 1) / t;
        }
        if (ctas <= cap) hi = mid; else lo = mid;
    }
    struct Row { double c; int32_t v[4]; };
    Row* rows = (Row*)malloc(sizeof(Row) * (size_t)(cap + n_jobs));
    if (!rows) return fail(A3D_EINVAL, "a3d_plan_tiles: out of memory");
    int n = 0, tile_used = 1;
    for (int j = 0; j < n_jobs; ++j) {
        const int nc = jobs_host[j].n_cand;
        if (nc == 0) continue;
        const int t = tile_of(j, hi), k = (nc + t - 1) / t, base = nc / k, rem = nc % k;
        int c = 0;
        for (int i = 0; i < k; ++i) {
            const int sz = base + (i < rem ? 1 : 0);
            rows[n++] = {kPlanFixed + sz * cost(j), {j, c, sz, 0}};
            c += sz;
            tile_used = sz > tile_used ? sz : tile_used;
        }
    }
    for (int j = 0; j < n_jobs; ++j)
        rows[n++] = {kPlanFixed + kPlanPerCand + 2.5 * (double)jobs_host[j].pcd_cap, {j, 0, 0, 1}};
    // most expensive first (stable: ties keep job / candidate order)
    for (int i = 1; i < n; ++i) {
        const Row r = rows[i];
        int k = i - 1;
        while (k >= 0 && rows[k].c < r.c) { rows[k + 1] = rows[k]; --k; }
        rows[k + 1] = r;
    }
    for (int i = 0; i < n; ++i) memcpy(tile_map_out + 4 * (size_t)i, rows[i].v, sizeof(int32_t) * 4);
    free(rows);
    *tile_cand_out = tile_used;
    return n;
}

int a3d_project_max_tile(int H, int W) {
    if (H <= 0 || W <= 0) return fail(A3D_EINVAL, "a3d_project_max_tile: bad shape %dx%d", H, W);
    const int optin = device_smem_optin();
    if (optin <= 0) return fail(A3D_ECUDA, "a3d_project_max_tile: no CUDA device");
    const int pitch = pitch_words(W);
    int tile = 0;
    while (project_smem_bytes(H, pitch, tile + 1) <= (size_t)optin) ++tile;
    if (tile < 1)
        return fail(A3D_ELIMIT, "a3d_project: a %dx%d mask (%zu B packed) does not fit the %d B of shared memory",
                    H, W, (size_t)H * pitch * 4, optin);
    return tile;
}

// Pinned host block -> device block by SM loads over PCIe (see include/a3d.h): the pass descriptors of a
// pipeline must not queue on the H2D copy engine behind a gigabyte of mask uploads.
int a3d_fetch_host_block(void* dst_dev, const void* src_host_pinned, int64_t nbytes, void* stream) {
    if (nbytes < 0) return fail(A3D_EINVAL, "a3d_fetch_host_block: nbytes < 0");
    if (nbytes == 0) return A3D_OK;
    if (!dst_dev || !src_host_pinned) return fail(A3D_EINVAL, "a3d_fetch_host_block: null pointer");
    if (((uintptr_t)dst_dev | (uintptr_t)src_host_pinned) & 15) return fail(A3D_EINVAL, "a3d_fetch_host_block: blocks must be 16-byte aligned");
    void* src_dev = nullptr;
    if (cudaHostGetDevicePointer(&src_dev, const_cast<void*>(src_host_pinned), 0) != cudaSuccess || !src_dev) {
        cudaGetLastError();
        return fail(A3D_EINVAL, "a3d_fetch_host_block: the source is not pinned (device-mapped) host memory");
    }
    const int64_t n16 = (nbytes + 15) / 16;
    const int64_t want = (n16 + 4 * 256 - 1) / (4 * 256);
    const int cap = device_sm_count();
    k_fetch_block<<<(unsigned)(want < cap ? want : cap), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<uint4*>(dst_dev), reinterpret_cast<const uint4*>(src_dev), n16);
    A3D_CUDA_TRY(cudaGetLastError());
    return A3D_OK;
}

int a3d_pack_masks(const void* src, int dtype, int64_t n, int H, int W, float thresh,
                   uint32_t* bits_gt, uint32_t* bits_nz, void* stream) {
    if (n < 0 || H <= 0 || W <= 0) return fail(A3D_EINVAL, "a3d_pack_masks: bad shape");
    if (n == 0) return A3D_OK;
    if (!src || !bits_gt) return fail(A3D_EINVAL, "a3d_pack_masks: null pointer");
    const int pitch = pitch_words(W);
    const int64_t rows = n * H;
    const int64_t want = (rows + 7) / 8;
    const int cap_ctas = device_sm_count() * 16;
    const int grid = (int)(want < cap_ctas ? want : cap_ctas);
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype != A3D_F32 && dtype != A3D_U8) return fail(A3D_EINVAL, "a3d_pack_masks: unknown dtype %d", dtype);
    const size_t esz = dtype == A3D_F32 ? 4 : 1;
    const bool vec = ((size_t)W * esz) % 16 == 0 && ((uintptr_t)src % 16) == 0;
    if (vec) {
        // words past ceil(W/32) up to the pitch are padding: the vector kernel writes every word it owns,
        // the remainder (pitch not a multiple of 4 segments) is cleared here
        const int64_t segs = (W + 127) / 128;
        if (segs * 4 < pitch) {
            A3D_CUDA_TRY(cudaMemsetAsync(bits_gt, 0, (size_t)rows * pitch * 4, s));
            if (bits_nz) A3D_CUDA_TRY(cudaMemsetAsync(bits_nz, 0, (size_t)rows * pitch * 4, s));
        }
        const int64_t wantv = (rows * segs + 31) / 32;
        const int gridv = (int)(wantv < cap_ctas ? (wantv > 0 ? wantv : 1) : cap_ctas);
        if (dtype == A3D_F32)
            k_pack_vec<float><<<gridv, 256, 0, s>>>((const float*)src, rows, W, pitch, thresh, bits_gt, bits_nz);
        else
            k_pack_vec<unsigned char><<<gridv, 256, 0, s>>>((const unsigned char*)src, rows, W, pitch, thresh, bits_gt, bits_nz);
    } else if (dtype == A3D_F32) {
        k_pack<float><<<grid, 256, 0, s>>>((const float*)src, rows, W, pitch, thresh, bits_gt, bits_nz);
    } else {
        k_pack<unsigned char><<<grid, 256, 0, s>>>((const unsigned char*)src, rows, W, pitch, thresh, bits_gt, bits_nz);
    }
    A3D_CUDA_TRY(cudaGetLastError());
    return A3D_OK;
}

// The whole upload of a clip's dense masks in one call (see include/a3d.h): frame copies into a device
// staging block with a bounded number in flight, a pack launch whenever the block is full.  Called from a
// helper thread through ctypes, i.e. WITHOUT the interpreter lock: driven from Python, every one of the
// ~120 frame copies per clip needed the lock back after waiting for its predecessor, and lost the copy
// engine's slack whenever another thread held it.
int a3d_upload_masks(const void* const* chunks, const int64_t* chunk_masks, int n_chunks, int dtype, int H, int W,
                     float thresh, void* stage_dev, int64_t stage_cap_masks, uint32_t* bits_gt, uint32_t* bits_nz,
                     int depth, void* stream) {
    if (n_chunks < 0 || H <= 0 || W <= 0 || stage_cap_masks <= 0) return fail(A3D_EINVAL, "a3d_upload_masks: bad shape");
    if (n_chunks == 0) return A3D_OK;
    if (!chunks || !chunk_masks || !stage_dev || !bits_gt) return fail(A3D_EINVAL, "a3d_upload_masks: null pointer");
    if (dtype != A3D_F32 && dtype != A3D_U8) return fail(A3D_EINVAL, "a3d_upload_masks: unknown dtype %d", dtype);
    const size_t per_mask = (size_t)H * W * (dtype == A3D_F32 ? 4 : 1);
    const size_t words = (size_t)H * pitch_words(W);
    cudaStream_t s = (cudaStream_t)stream;
    if (depth > 64) depth = 64;
    cudaEvent_t ev[64];
    for (int i = 0; i < depth; ++i)
        if (cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming) != cudaSuccess) {
            for (int j = 0; j < i; ++j) cudaEventDestroy(ev[j]);
            return fail(A3D_ECUDA, "a3d_upload_masks: cudaEventCreate: %s", cudaGetErrorString(cudaGetLastError()));
        }
    int rc = A3D_OK;
    cudaError_t ce = cudaSuccess;
    int64_t fill = 0, done = 0;                       // masks in the staging block / masks packed so far
    auto flush = [&]() {
        if (fill == 0 || rc != A3D_OK) return;
        rc = a3d_pack_masks(stage_dev, dtype, fill, H, W, thresh, bits_gt + (size_t)done * words,
                            bits_nz ? bits_nz + (size_t)done * words : nullptr, stream);
        done += fill;
        fill = 0;
    };
    for (int i = 0; i < n_chunks && rc == A3D_OK; ++i) {
        const int64_t k = chunk_masks[i];
        if (k < 0 || k > stage_cap_masks || (k > 0 && !chunks[i])) { rc = fail(A3D_EINVAL, "a3d_upload_masks: chunk %d: bad size or pointer", i); break; }
        if (k == 0) continue;
        if (fill + k > stage_cap_masks) flush();      // (the copies that follow are ordered after the pack by the stream)
        if (rc != A3D_OK) break;
        if (depth > 0 && i >= depth) {
            // polled with short sleeps: cudaEventSynchronize either spins on a core for the whole upload (eight
            // ranks of a node share its cores with their hosts' work) or, as a blocking-sync event, wakes up
            // late enough to drain the copies in flight (measured: 181 against 165 ms per 6 clips)
            while ((ce = cudaEventQuery(ev[i % depth])) == cudaErrorNotReady) {
                struct timespec ts = {0, 20000};
                nanosleep(&ts, nullptr);
                cudaGetLastError();                   // (not-ready is recorded as the thread's last error)
            }
            if (ce != cudaSuccess) break;
        }
        ce = cudaMemcpyAsync((char*)stage_dev + (size_t)fill * per_mask, chunks[i], (size_t)k * per_mask,
                             cudaMemcpyHostToDevice, s);
        if (ce != cudaSuccess) break;
        if (depth > 0 && (ce = cudaEventRecord(ev[i % depth], s)) != cudaSuccess) break;
        fill += k;
    }
    if (ce == cudaSuccess) flush();
    for (int i = 0; i < depth; ++i) cudaEventDestroy(ev[i]);
    if (ce != cudaSuccess) return fail(A3D_ECUDA, "a3d_upload_masks: %s", cudaGetErrorString(ce));
    return rc;
}

int a3d_mask_meta(const uint32_t* bits, int64_t n, int H, int W, int32_t* popc, int32_t* bbox,
                  void* stream) {
    if (n < 0 || H <= 0 || W <= 0) return fail(A3D_EINVAL, "a3d_mask_meta: bad shape");
    if (n == 0) return A3D_OK;
    if (!bits || !popc || !bbox) return fail(A3D_EINVAL, "a3d_mask_meta: null pointer");
    if (n > 0x7fffffff) return fail(A3D_ELIMIT, "a3d_mask_meta: n too large");
    k_mask_meta<<<(unsigned)n, 256, 0, (cudaStream_t)stream>>>(bits, H, pitch_words(W), popc, bbox);
    A3D_CUDA_TRY(cudaGetLastError());
    return A3D_OK;
}

int a3d_project(const a3d_camera_t* cam, const a3d_job_t* jobs, int n_jobs, int max_cand,
                int tile_cand, const uint32_t* src_bits, const int32_t* src_bbox,
                const float* xform, float* pcd_ws, int32_t* pcd_count, float* hom_ws,
                const int32_t* tile_map, int n_tiles,
                uint32_t* proj_bits, int32_t* proj_popc, int32_t* proj_bbox, int out_mode, void* stream) {
    if (out_mode != A3D_OUT_FULL && out_mode != A3D_OUT_BBOX_ROWS) return fail(A3D_EINVAL, "a3d_project: unknown out_mode %d", out_mode);
    return project_impl(cam, jobs, n_jobs, max_cand, tile_cand, src_bits, src_bbox, xform, pcd_ws, pcd_count, hom_ws,
                        tile_map, n_tiles, proj_bits, proj_popc, proj_bbox, stream, false, out_mode == A3D_OUT_BBOX_ROWS);
}

int a3d_pass(const a3d_camera_t* cam, const a3d_job_t* jobs, int n_jobs, int max_tgt, int max_cand,
             int tile_cand, int64_t n_tgt_total, int64_t n_pool_masks, int64_t n_cand_total,
             const uint32_t* pool_bits, const int32_t* pool_popc, const int32_t* pool_bbox,
             const uint32_t* src_bits, const int32_t* src_bbox, const float* xform, const int32_t* tgt_index,
             float* pcd_ws, int32_t* pcd_count, float* hom_ws, const int32_t* tile_map, int n_tiles,
             uint32_t* proj_bits, int32_t* proj_popc, int32_t* proj_bbox,
             uint64_t* key_ws, int32_t* inter_tab,
             int32_t* best_cand, int32_t* best_inter, int32_t* best_union, float* best_iou,
             int out_mode, void* stream) {
    if (!cam) return fail(A3D_EINVAL, "a3d_pass: null camera");
    if (out_mode != A3D_OUT_FULL && out_mode != A3D_OUT_BBOX_ROWS) return fail(A3D_EINVAL, "a3d_pass: unknown out_mode %d", out_mode);
    const bool score = n_jobs > 0 && max_tgt > 0 && n_tgt_total > 0;
    if (score) {
        // the keys are cleared FIRST so that no memset node sits between the kernels: k_project, the scoring
        // kernel and k_finalize are then launched as programmatic dependents of their predecessors
        if (!key_ws) return fail(A3D_EINVAL, "a3d_pass: null pointer");
        A3D_CUDA_TRY(cudaMemsetAsync(key_ws, 0, sizeof(uint64_t) * (size_t)n_tgt_total, (cudaStream_t)stream));
    }
    // Dependent launches pay when a pass is a handful of short kernels (C2: 80.9 -> 72.8 us); on the
    // 256-job shard they measured 7 % slower than plain stream order (2.82 vs 2.63 ms), so only passes whose
    // projection grid fits about two waves use them (A3D_PDL=0 | 1 forces).
    const char* env_pdl = getenv("A3D_PDL");
    const bool pdl = env_pdl ? env_pdl[0] == '1' : (long long)n_jobs * (max_cand > 0 ? max_cand : 1) <= 12LL * device_sm_count();
    int rc = project_impl(cam, jobs, n_jobs, max_cand, tile_cand, src_bits ? src_bits : pool_bits,
                          src_bits ? src_bbox : pool_bbox, xform, pcd_ws, pcd_count, hom_ws, tile_map, n_tiles,
                          proj_bits, proj_popc, proj_bbox, stream, pdl, out_mode == A3D_OUT_BBOX_ROWS);
    if (rc != A3D_OK || !score) return rc;
    return score_impl(cam->H, cam->W, jobs, n_jobs, max_tgt, max_cand, n_tgt_total, n_pool_masks, n_cand_total,
                      pool_bits, pool_popc, pool_bbox, tgt_index, proj_bits, proj_popc, proj_bbox, key_ws, inter_tab,
                      best_cand, best_inter, best_union, best_iou, stream, false, pdl);
}

}  // extern "C"

static int project_impl(const a3d_camera_t* cam, const a3d_job_t* jobs, int n_jobs, int max_cand,
                        int tile_cand, const uint32_t* src_bits, const int32_t* src_bbox,
                        const float* xform, float* pcd_ws, int32_t* pcd_count, float* hom_ws,
                        const int32_t* tile_map, int n_tiles,
                        uint32_t* proj_bits, int32_t* proj_popc, int32_t* proj_bbox, void* stream, bool pdl,
                        bool rows_only) {
    if (!cam || n_jobs < 0 || max_cand < 0) return fail(A3D_EINVAL, "a3d_project: bad argument");
    if (n_jobs == 0 || max_cand == 0) return A3D_OK;
    if (!jobs || !src_bits || !src_bbox || !xform || !pcd_ws || !pcd_count || !proj_bits || !proj_popc ||
        !proj_bbox)
        return fail(A3D_EINVAL, "a3d_project: null pointer");
    // A3D_PROJECT_KERNEL = exact | filter (default filter: homography + proven truncation, exact chain on
    // demand; identical results).  The filter packs source coordinates in 16 bits and needs hom_ws.
    // Default: the filter kernel when the grid is more than two waves of CTAs; on smaller grids the per-CTA
    // fixed work and the extra CTAs outweigh the cheaper pixels (C2, 124-148 CTAs: 46 us against 42 us).
    const char* env_proj = getenv("A3D_PROJECT_KERNEL");
    const bool force_filter = env_proj && !strcmp(env_proj, "filter"), force_exact = env_proj && !strcmp(env_proj, "exact");
    if (force_filter && !hom_ws) return fail(A3D_EINVAL, "a3d_project: A3D_PROJECT_KERNEL=filter needs hom_ws");
    bool filter = !force_exact && cam->H <= 32768 && cam->W <= 32768 && hom_ws;
    if (filter && !force_filter) {
        const int mt = a3d_project_max_tile(cam->H, cam->W);
        const int t = tile_cand > 0 ? tile_cand : (mt > 0 ? mt : 1);
        const long long grid = tile_map ? n_tiles : (long long)n_jobs * ((max_cand + t - 1) / t);
        filter = grid > 2LL * device_sm_count();
    }
    const int max_tile = a3d_project_max_tile(cam->H, cam->W);
    if (max_tile < 0) return max_tile;
    if (tile_cand <= 0) tile_cand = max_tile;
    if (tile_cand > max_tile)
        return fail(A3D_EINVAL, "a3d_project: tile_cand %d > max %d for %dx%d", tile_cand, max_tile, cam->H, cam->W);
    if (tile_cand > max_cand) tile_cand = max_cand;

    Cam c;
    memcpy(c.k, cam->kinv, sizeof(c.k));
    c.f = cam->f; c.cx = cam->cx; c.cy = cam->cy;
    c.H = cam->H; c.W = cam->W; c.pitch = pitch_words(cam->W);
    c.sparse = (c.k[1] == 0.0 && c.k[3] == 0.0 && c.k[6] == 0.0 && c.k[7] == 0.0 && c.k[8] == 1.0);
    cudaStream_t s = (cudaStream_t)stream;

    // 1. source pixels -> compacted point clouds
    const size_t usmem = (size_t)c.H * c.pitch * sizeof(uint32_t);
    if (usmem > (size_t)device_smem_optin())
        return fail(A3D_ELIMIT, "a3d_project: %dx%d mask does not fit shared memory", c.H, c.W);
    // few jobs: spread each job's phase 2 over several CTAs so all SMs have work
    int usplit = (2 * device_sm_count() + n_jobs - 1) / n_jobs;
    usplit = usplit < 1 ? 1 : (usplit > 32 ? 32 : usplit);
    const dim3 ugrid((unsigned)n_jobs, (unsigned)usplit);
    if (c.sparse) {
        A3D_CUDA_TRY(cudaFuncSetAttribute(k_unproject<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)usmem));
        A3D_CUDA_TRY(launch(k_unproject<true>, ugrid, dim3(kUnprojThreads), usmem, s, false, c, jobs, src_bits, src_bbox,
                            xform, pcd_ws, pcd_count, filter ? hom_ws : (float*)nullptr));
    } else {
        A3D_CUDA_TRY(cudaFuncSetAttribute(k_unproject<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)usmem));
        A3D_CUDA_TRY(launch(k_unproject<false>, ugrid, dim3(kUnprojThreads), usmem, s, false, c, jobs, src_bits, src_bbox,
                            xform, pcd_ws, pcd_count, filter ? hom_ws : (float*)nullptr));
    }
    A3D_CUDA_TRY(cudaGetLastError());

    // 2. candidates
    const size_t smem = project_smem_bytes(c.H, c.pitch, tile_cand);
    const int tiles_per_job = (max_cand + tile_cand - 1) / tile_cand;
    long long nblocks = (long long)n_jobs * tiles_per_job;
    if (nblocks > 0x7fffffffLL) return fail(A3D_ELIMIT, "a3d_project: too many (job, tile) blocks");
    const int4* tmap = nullptr;
    if (tile_map) {                   // caller-planned tiles (their extra CTAs included)
        if (n_tiles <= 0) return fail(A3D_EINVAL, "a3d_project: tile_map with n_tiles %d", n_tiles);
        if ((uintptr_t)tile_map % 16) return fail(A3D_EINVAL, "a3d_project: tile_map must be 16-byte aligned");
        tmap = reinterpret_cast<const int4*>(tile_map);
        nblocks = n_tiles;
    } else if (filter) {
        nblocks += n_jobs;            // one extra CTA per job for its exact-only candidates
        if (nblocks > 0x7fffffffLL) return fail(A3D_ELIMIT, "a3d_project: too many (job, tile) blocks");
    }
    if (project_persistent()) {
        int* counter = pcd_count + n_jobs;           // zeroed by k_unproject
        const int sms = device_sm_count();
        const long long want_ctas = (nblocks + 1) / 2;
        const unsigned grid = (unsigned)(want_ctas < sms ? want_ctas : sms);
        if (filter) {
            A3D_CUDA_TRY(cudaFuncSetAttribute(k_project_p<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            A3D_CUDA_TRY(launch(k_project_p<true>, dim3(grid), dim3(kProjThreads), smem, s, pdl, c, jobs, tile_cand,
                                tiles_per_job, (int)nblocks, counter, xform, src_bbox, (const float*)pcd_ws,
                                (const int32_t*)pcd_count, (const float*)hom_ws, tmap, proj_bits, proj_popc, proj_bbox, rows_only));
        } else {
            A3D_CUDA_TRY(cudaFuncSetAttribute(k_project_p<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            A3D_CUDA_TRY(launch(k_project_p<false>, dim3(grid), dim3(kProjThreads), smem, s, pdl, c, jobs, tile_cand,
                                tiles_per_job, (int)nblocks, counter, xform, src_bbox, (const float*)pcd_ws,
                                (const int32_t*)pcd_count, (const float*)hom_ws, tmap, proj_bits, proj_popc, proj_bbox, rows_only));
        }
        return A3D_OK;
    }
    if (filter) {
        A3D_CUDA_TRY(cudaFuncSetAttribute(k_project<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        A3D_CUDA_TRY(launch(k_project<true>, dim3((unsigned)nblocks), dim3(kProjThreads), smem, s, pdl, c, jobs, tile_cand,
                            tiles_per_job, xform, src_bbox, (const float*)pcd_ws, (const int32_t*)pcd_count,
                            (const float*)hom_ws, tmap, proj_bits, proj_popc, proj_bbox, rows_only));
    } else {
        A3D_CUDA_TRY(cudaFuncSetAttribute(k_project<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        A3D_CUDA_TRY(launch(k_project<false>, dim3((unsigned)nblocks), dim3(kProjThreads), smem, s, pdl, c, jobs, tile_cand,
                            tiles_per_job, xform, src_bbox, (const float*)pcd_ws, (const int32_t*)pcd_count,
                            (const float*)hom_ws, tmap, proj_bits, proj_popc, proj_bbox, rows_only));
    }
    return A3D_OK;
}

extern "C" {

int a3d_score(int H, int W, const a3d_job_t* jobs, int n_jobs, int max_tgt, int max_cand,
              int64_t n_tgt_total, int64_t n_pool_masks, int64_t n_cand_total,
              const uint32_t* tgt_bits, const int32_t* tgt_popc, const int32_t* tgt_bbox,
              const int32_t* tgt_index,
              const uint32_t* proj_bits, const int32_t* proj_popc, const int32_t* proj_bbox,
              uint64_t* key_ws, int32_t* inter_tab,
              int32_t* best_cand, int32_t* best_inter, int32_t* best_union, float* best_iou,
              void* stream) {
    return score_impl(H, W, jobs, n_jobs, max_tgt, max_cand, n_tgt_total, n_pool_masks, n_cand_total, tgt_bits,
                      tgt_popc, tgt_bbox, tgt_index, proj_bits, proj_popc, proj_bbox, key_ws, inter_tab, best_cand,
                      best_inter, best_union, best_iou, stream, true, false);
}

}  // extern "C"

static int score_impl(int H, int W, const a3d_job_t* jobs, int n_jobs, int max_tgt, int max_cand,
                      int64_t n_tgt_total, int64_t n_pool_masks, int64_t n_cand_total,
                      const uint32_t* tgt_bits, const int32_t* tgt_popc, const int32_t* tgt_bbox,
                      const int32_t* tgt_index,
                      const uint32_t* proj_bits, const int32_t* proj_popc, const int32_t* proj_bbox,
                      uint64_t* key_ws, int32_t* inter_tab,
                      int32_t* best_cand, int32_t* best_inter, int32_t* best_union, float* best_iou,
                      void* stream, bool zero_keys, bool pdl) {
    if (H <= 0 || W <= 0 || n_jobs < 0 || max_tgt < 0 || max_cand < 0 || n_tgt_total < 0 || n_pool_masks < 0 ||
        n_cand_total < 0)
        return fail(A3D_EINVAL, "a3d_score: bad argument");
    if (n_jobs == 0 || max_tgt == 0 || n_tgt_total == 0) return A3D_OK;
    if (max_cand == 0) return fail(A3D_EINVAL, "a3d_score: jobs need at least one candidate");
    if (!jobs || !tgt_bits || !tgt_popc || !tgt_bbox || !tgt_index || !proj_bits || !proj_popc ||
        !proj_bbox || !key_ws || !best_cand || !best_inter || !best_union || !best_iou)
        return fail(A3D_EINVAL, "a3d_score: null pointer");
    const int pitch = pitch_words(W);
    cudaStream_t s = (cudaStream_t)stream;
    if (zero_keys) A3D_CUDA_TRY(cudaMemsetAsync(key_ws, 0, sizeof(uint64_t) * (size_t)n_tgt_total, s));
    // the winner's intersection count fits the key when candidates < 4096 and pixels < 2^20
    const char* env_key = getenv("A3D_SCORE_KEY");
    const int packed = (max_cand <= 4096 && (long long)H * W < (1 << 20) && !(env_key && !strcmp(env_key, "wide"))) ? 1 : 0;

    // Three scoring kernels with identical results (A3D_SCORE_KERNEL = ldg | tma | mma forces one):
    //  * k_score ("ldg"): AND + popcount on the integer pipes, direct loads, per-warp regions — every SM
    //    works on every job, so it is the one for few or small jobs;
    //  * k_score_mma ("mma"): tensor cores (tcgen05 kind::mxf4 on bit-expanded masks), one CTA per
    //    (job, 128 targets, <= 240 candidates); its time is ~245 us per wave of CTAs almost regardless of
    //    the candidate count.  Measured on B200 (tools/score_ab.py) with the earlier kind::i8 kernel (the
    //    kind::mxf4 one is faster: 308 vs 1237 us on the first shape), 120 targets per job:
    //    180 candidates x 256 jobs 440 us vs 1232 us; x 64 jobs 251 vs 322; x 48 jobs 249 vs 245;
    //    720 candidates x 64 jobs 421 vs 1138; but 60 x 90 x 256 jobs 339 vs 355 and 60 x 45: 323 vs 204
    //    — hence the automatic choice below: enough CTAs to fill the SMs and big (target, candidate) tiles;
    //  * k_score_tma ("tma"): TMA-staged variant of k_score, measured slower than direct loads.
    const char* env_kernel = getenv("A3D_SCORE_KERNEL");
    const bool use_tma = env_kernel && !strcmp(env_kernel, "tma");
    const bool tma_ok = use_tma && (n_pool_masks * H < 0x7fffffffLL) && (n_cand_total * H < 0x7fffffffLL);
    int mma_ctile = (max_cand + 15) & ~15;
    if (mma_ctile > kMmaNMax) mma_ctile = kMmaNMax;
    const long long mma_blocks = (long long)n_jobs * ((max_tgt + kMmaM - 1) / kMmaM) * ((max_cand + mma_ctile - 1) / mma_ctile);
    const bool mma_auto = mma_blocks >= 60 && (long long)(max_tgt < kMmaM ? max_tgt : kMmaM) * mma_ctile >= 16384;
    // its f32 accumulators count exactly up to 2^24: larger frames always take k_score
    const bool mma_exact = (long long)H * W <= (1LL << 24);
    const bool use_mma = mma_exact && (env_kernel ? !strcmp(env_kernel, "mma") : mma_auto);
    if (use_mma) {
        // tensor-core scoring: CTA = (job, 128 targets, <= 240 candidates)
        const int ctile = mma_ctile;
        const int tt_tiles = (max_tgt + kMmaM - 1) / kMmaM, ct_tiles = (max_cand + ctile - 1) / ctile;
        const long long nblocks = (long long)n_jobs * tt_tiles * ct_tiles;
        if (nblocks > 0x7fffffffLL) return fail(A3D_ELIMIT, "a3d_score: too many (job, tile) blocks");
        const size_t smem = (size_t)kMmaStages * mma_stage_bytes(ctile);
        A3D_CUDA_TRY(cudaFuncSetAttribute(k_score_mma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        A3D_CUDA_TRY(launch(k_score_mma, dim3((unsigned)nblocks), dim3(kMmaThreads), smem, s, pdl, jobs, H, pitch, tt_tiles,
                            ct_tiles, ctile, tgt_bits, tgt_popc, tgt_bbox, tgt_index, proj_bits, proj_popc, proj_bbox,
                            (unsigned long long*)key_ws, inter_tab, packed));
    } else if (tma_ok) {
        // mask tiles staged by TMA: one tensor map per (array, box width)
        TmaMaps maps;
        const int widths[4] = {4, 8, 16, 32};
        for (int i = 0; i < 4; ++i) {
            const int bw = widths[i] < pitch ? widths[i] : pitch;
            const int rows = kTmaTileWords / bw;
            maps.bw[i] = bw;
            maps.rows[i] = rows;
            int rc = encode_mask_map(&maps.t[i], tgt_bits, (uint64_t)n_pool_masks * H, pitch, bw, rows);
            if (rc) return rc;
            rc = encode_mask_map(&maps.p[i], proj_bits, (uint64_t)n_cand_total * H, pitch, bw, rows);
            if (rc) return rc;
        }
        const int tt_tiles = (max_tgt + kTmaTT - 1) / kTmaTT, ct_tiles = (max_cand + kTmaCT - 1) / kTmaCT;
        const long long nblocks = (long long)n_jobs * tt_tiles * ct_tiles;
        if (nblocks > 0x7fffffffLL) return fail(A3D_ELIMIT, "a3d_score: too many (job, tile) blocks");
        A3D_CUDA_TRY(cudaFuncSetAttribute(k_score_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTmaSmemBytes));
        A3D_CUDA_TRY(launch(k_score_tma, dim3((unsigned)nblocks), dim3(256), kTmaSmemBytes, s, pdl, maps, jobs, H, pitch,
                            tt_tiles, ct_tiles, tgt_popc, tgt_bbox, tgt_index, proj_popc, proj_bbox,
                            (unsigned long long*)key_ws, inter_tab, packed));
    } else {
        // candidates per warp: 4x4 register tiles (3 CTAs/SM) are fastest on full grids (1.23 vs 1.39 ms on the
        // C3 shard); 4x2 tiles (4 CTAs/SM, twice the CTAs) win when the 4x4 grid cannot fill the SMs
        // (26.9 vs 30.7 us on C2).  A3D_SCORE_WC overrides for A/B runs.
        const char* env_wc = getenv("A3D_SCORE_WC");
        const long long blocks44 = (long long)n_jobs * ((max_tgt + kScoreTT - 1) / kScoreTT) * ((max_cand + 15) / 16);
        int wc = blocks44 < 6LL * device_sm_count() ? 2 : 4;
        if (env_wc && (env_wc[0] == '2' || env_wc[0] == '4')) wc = env_wc[0] - '0';
        const int tt_tiles = (max_tgt + kScoreTT - 1) / kScoreTT, ct_tiles = (max_cand + 4 * wc - 1) / (4 * wc);
        const long long nblocks = (long long)n_jobs * tt_tiles * ct_tiles;
        if (nblocks > 0x7fffffffLL) return fail(A3D_ELIMIT, "a3d_score: too many (job, tile) blocks");
        // A3D_SCORE_ADDR=wide forces 64-bit mask addressing, which only pools or candidate buffers of
        // 2^32 words and more need, so that it can be checked on small inputs
        const char* env_addr = getenv("A3D_SCORE_ADDR");
        const unsigned long long words = (unsigned long long)H * pitch;
        const bool narrow = (unsigned long long)n_pool_masks * words < (1ull << 32) &&
                            (unsigned long long)n_cand_total * words < (1ull << 32) &&
                            !(env_addr && !strcmp(env_addr, "wide"));
#define A3D_LAUNCH_SCORE(N, WC)                                                                                    \
    A3D_CUDA_TRY(launch(k_score<N, WC, WC == 2>, dim3((unsigned)nblocks), dim3(256), 0, s, pdl, jobs, H, pitch, tt_tiles, \
                        ct_tiles, tgt_bits, tgt_popc, tgt_bbox, tgt_index, proj_bits, proj_popc, proj_bbox,         \
                        (unsigned long long*)key_ws, inter_tab, packed))
        if (narrow && wc == 4) A3D_LAUNCH_SCORE(true, 4);
        else if (narrow) A3D_LAUNCH_SCORE(true, 2);
        else if (wc == 4) A3D_LAUNCH_SCORE(false, 4);
        else A3D_LAUNCH_SCORE(false, 2);
#undef A3D_LAUNCH_SCORE
    }
    A3D_CUDA_TRY(cudaGetLastError());
    const int fy = packed ? (max_tgt + 255) / 256 : ((max_tgt + 7) / 8 < 64 ? (max_tgt + 7) / 8 : 64);
    const dim3 fgrid((unsigned)n_jobs, (unsigned)fy);
    A3D_CUDA_TRY(launch(k_finalize, fgrid, dim3(256), 0, s, pdl, jobs, H, pitch, tgt_bits, tgt_popc, tgt_index, proj_bits,
                        proj_popc, proj_bbox, (const unsigned long long*)key_ws, best_cand, best_inter, best_union,
                        best_iou, packed));
    return A3D_OK;
}

extern "C" {

int a3d_emit_masks(const uint32_t* bits, const int32_t* index, int64_t n, int H, int W,
                   int out_dtype, void* out, void* stream) {
    if (n < 0 || H <= 0 || W <= 0) return fail(A3D_EINVAL, "a3d_emit_masks: bad shape");
    if (n == 0) return A3D_OK;
    if (!bits || !out) return fail(A3D_EINVAL, "a3d_emit_masks: null pointer");
    if (n > 65535) return fail(A3D_ELIMIT, "a3d_emit_masks: at most 65535 masks per call");
    const int pitch = pitch_words(W);
    const int bx = (H * W + 255) / 256;
    const dim3 grid((unsigned)(bx < 64 ? bx : 64), (unsigned)n);
    cudaStream_t s = (cudaStream_t)stream;
    if (out_dtype == A3D_F32)
        k_emit<float><<<grid, 256, 0, s>>>(bits, index, H, W, pitch, (float*)out);
    else if (out_dtype == A3D_U8)
        k_emit<unsigned char><<<grid, 256, 0, s>>>(bits, index, H, W, pitch, (unsigned char*)out);
    else
        return fail(A3D_EINVAL, "a3d_emit_masks: unknown dtype %d", out_dtype);
    A3D_CUDA_TRY(cudaGetLastError());
    return A3D_OK;
}

// shape checks shared by the two encoder calls; 1 = nothing to do, 0 = go on, < 0 = error
static int rle_encode_args(const char* what, const uint32_t* bits, int64_t n, int H, int W, const void* a,
                           const void* b) {
    if (n < 0 || H <= 0 || W <= 0) return fail(A3D_EINVAL, "%s: bad shape n=%lld %dx%d", what, (long long)n, H, W);
    if ((int64_t)H * W > 0x7fffffffLL)
        return fail(A3D_ELIMIT, "%s: a %dx%d mask has more than 2^31 - 1 pixels", what, H, W);
    if (n == 0) return 1;
    if (!bits || !a || !b) return fail(A3D_EINVAL, "%s: null pointer", what);
    return 0;
}

static unsigned rle_grid(int64_t n) {
    const int sms = device_sm_count();
    const int64_t cap = (int64_t)(sms > 0 ? sms : 1) * 16;
    return (unsigned)(n < cap ? n : cap);
}

int a3d_rle_count_runs(const uint32_t* bits, const int32_t* index, int64_t n, int H, int W, int64_t* runs_out,
                       void* stream) {
    const int rc = rle_encode_args("a3d_rle_count_runs", bits, n, H, W, runs_out, runs_out);
    if (rc) return rc < 0 ? rc : A3D_OK;
    k_rle_count<<<rle_grid(n), 256, 0, (cudaStream_t)stream>>>(bits, index, n, H, W, pitch_words(W), runs_out);
    A3D_CUDA_TRY(cudaGetLastError());
    return A3D_OK;
}

int a3d_bits_to_rle(const uint32_t* bits, const int32_t* index, int64_t n, int H, int W, const int64_t* begin,
                    uint32_t* counts_out, void* stream) {
    const int rc = rle_encode_args("a3d_bits_to_rle", bits, n, H, W, begin, counts_out);
    if (rc) return rc < 0 ? rc : A3D_OK;
    k_bits_to_rle<<<rle_grid(n), kRleWarps * 32, 0, (cudaStream_t)stream>>>(bits, index, n, H, W, pitch_words(W),
                                                                             begin, counts_out);
    A3D_CUDA_TRY(cudaGetLastError());
    return A3D_OK;
}

int a3d_rle_to_bits(const uint32_t* counts, const int64_t* begin, int64_t n, int H, int W, uint32_t* bits,
                    void* stream) {
    if (n < 0 || H <= 0 || W <= 0) return fail(A3D_EINVAL, "a3d_rle_to_bits: bad shape");
    if (n == 0) return A3D_OK;
    if (!counts || !begin || !bits) return fail(A3D_EINVAL, "a3d_rle_to_bits: null pointer");
    if (n > 0x7fffffff) return fail(A3D_ELIMIT, "a3d_rle_to_bits: n too large");
    const int pitch = pitch_words(W);
    const size_t smem = (size_t)H * pitch * 4;
    if (smem > (size_t)device_smem_optin() - 8192)
        return fail(A3D_ELIMIT, "a3d_rle_to_bits: %dx%d mask does not fit shared memory", H, W);
    A3D_CUDA_TRY(cudaFuncSetAttribute(k_rle_to_bits, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_rle_to_bits<<<(unsigned)n, 256, smem, (cudaStream_t)stream>>>(counts, begin, H, W, pitch, bits);
    A3D_CUDA_TRY(cudaGetLastError());
    return A3D_OK;
}

int a3d_plane_offsets(const float* depth, const float* rays, int H, int W, const uint32_t* bits,
                      const int32_t* bbox, const int32_t* inst_mask, const int32_t* inst_frame,
                      const float* normals, int64_t n_inst, float* offset_out, int32_t* count_out,
                      void* stream) {
    if (n_inst < 0 || H <= 0 || W <= 0) return fail(A3D_EINVAL, "a3d_plane_offsets: bad shape");
    if (n_inst == 0) return A3D_OK;
    if (!rays || !bits || !bbox || !inst_mask || !normals || !offset_out || !count_out || (depth && !inst_frame))
        return fail(A3D_EINVAL, "a3d_plane_offsets: null pointer");
    if (n_inst > 0x7fffffff) return fail(A3D_ELIMIT, "a3d_plane_offsets: too many instances");
    k_plane_offsets<<<(unsigned)n_inst, 256, 0, (cudaStream_t)stream>>>(depth, rays, H, W, pitch_words(W), bits, bbox,
                                                                         inst_mask, inst_frame, normals, offset_out,
                                                                         count_out);
    A3D_CUDA_TRY(cudaGetLastError());
    return A3D_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------
// render (a3d_render): masks and segments composited over the frames' backgrounds into RGB frames.
// One CTA per (frame, band of rows).  The band's bytes are contiguous in the background and in `out`,
// so they are staged in shared memory with 16-byte copies (bytes where the two addresses disagree modulo
// 16), the frame's list entries that touch the band are culled into shared memory (a pass of up to
// kRenderCap layers, then segments, at a time, in list order), and every thread composites whole packed
// words: 32 pixels of one row per work item.  HBM traffic: the band's background bytes, its output bytes
// and the words of the layers inside their boxes.
// ---------------------------------------------------------------------------
constexpr int kRenderThreads = 256;
constexpr int kRenderCap = kRenderThreads;      // list entries culled per pass: one per thread
constexpr int kRenderStageBytes = 32768;        // target size of a band's RGB staging

struct RenderSeg {                              // a culled segment with its box clipped to the band
    int x0, y0, x1, y1, r;
    uint32_t rgb;
    int bx0, bx1, by0, by1;
};

// block-wide copy of n bytes: 16-byte pieces when dst and src agree modulo 16, single bytes otherwise
__device__ __forceinline__ void render_copy(uint8_t* dst, const uint8_t* src, int64_t n) {
    const int t = threadIdx.x;
    if ((((uintptr_t)dst ^ (uintptr_t)src) & 15) == 0) {
        int64_t head = (16 - ((uintptr_t)dst & 15)) & 15;
        if (head > n) head = n;
        if (t < head) dst[t] = src[t];
        const int64_t n16 = (n - head) >> 4;
        uint4* d4 = (uint4*)(dst + head);
        const uint4* s4 = (const uint4*)(src + head);
        for (int64_t i = t; i < n16; i += 4 * kRenderThreads) {       // four loads in flight before the stores
            uint4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (i + u * kRenderThreads < n16) v[u] = s4[i + u * kRenderThreads];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (i + u * kRenderThreads < n16) d4[i + u * kRenderThreads] = v[u];
        }
        for (int64_t i = head + (n16 << 4) + t; i < n; i += kRenderThreads) dst[i] = src[i];
    } else {
        for (int64_t i = t; i < n; i += kRenderThreads) dst[i] = src[i];
    }
}

// ordered block-wide compaction: the slot of this thread's entry among the kept ones; *total = kept count
__device__ __forceinline__ int render_rank(bool keep, int* s_warp, int* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned b = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s_warp[warp] = __popc(b);
    __syncthreads();
    int base = 0, sum = 0;
#pragma unroll
    for (int w = 0; w < kRenderThreads / 32; ++w) {
        const int c = s_warp[w];
        base += w < warp ? c : 0;
        sum += c;
    }
    *total = sum;
    __syncthreads();
    return base + __popc(b & ((1u << lane) - 1u));
}

// exact: squared distance of pixel (x, y) to the closed segment <= r^2, in int64 (|coordinates| <= 2^14, r <= 256)
__device__ __forceinline__ bool render_seg_hit(const RenderSeg& s, int x, int y) {
    const int64_t dx = s.x1 - s.x0, dy = s.y1 - s.y0, qx = x - s.x0, qy = y - s.y0;
    const int64_t r2 = (int64_t)s.r * s.r;
    const int64_t t = qx * dx + qy * dy, L = dx * dx + dy * dy;
    if (t <= 0) return qx * qx + qy * qy <= r2;
    if (t >= L) {
        const int64_t ex = x - s.x1, ey = y - s.y1;
        return ex * ex + ey * ey <= r2;
    }
    const int64_t c = qx * dy - qy * dx;
    return c * c <= r2 * L;
}

// float64 reciprocal of a nonzero integer and square root of v >= 0 from the single-precision MUFU estimates and
// two Newton steps: no IEEE slow-path subroutine (whose calling convention spills the kernel's live registers)
__device__ __forceinline__ double render_rcp(double x) {
    double r = (double)__fdividef(1.0f, (float)x);
    r = r * (2.0 - x * r);
    return r * (2.0 - x * r);
}

__device__ __forceinline__ double render_sqrt(double v) {
    if (v <= 0.0) return 0.0;
    double y = (double)rsqrtf((float)v);
    y = y * (1.5 - 0.5 * v * y * y);
    y = y * (1.5 - 0.5 * v * y * y);
    return v * y;
}

// The pixels of row y within distance r of the segment form one interval (the capsule is convex).  Its ends,
// estimated in float64 as the hull of the two end discs and the strip beside the segment; the caller decides
// every pixel within one pixel of the estimate exactly, so only the estimate's error (far below a pixel) has
// to be covered.  false: the row misses the capsule.
__device__ __forceinline__ bool render_seg_row(const RenderSeg& s, int y, double* lo, double* hi) {
    const double r = s.r, x0 = s.x0, x1 = s.x1;
    double a = 1e30, b = -1e30;
    const double h0 = r * r - (double)(y - s.y0) * (y - s.y0), h1 = r * r - (double)(y - s.y1) * (y - s.y1);
    if (h0 >= 0) { const double w = render_sqrt(h0); a = fmin(a, x0 - w); b = fmax(b, x0 + w); }
    if (h1 >= 0) { const double w = render_sqrt(h1); a = fmin(a, x1 - w); b = fmax(b, x1 + w); }
    const int64_t idx = s.x1 - s.x0, idy = s.y1 - s.y0, iry = y - s.y0;
    const int64_t iL = idx * idx + idy * idy;
    if (iL > 0) {
        const double dx = (double)idx, dy = (double)idy, ry = (double)iry, L = (double)iL;
        double sa = -1e30, sb = 1e30;
        bool ok = true;
        if (idy != 0) {                          // |(x - x0) dy - ry dx| <= r sqrt(L)
            const double idy_r = render_rcp(dy);
            const double c = x0 + ry * dx * idy_r, w = r * render_sqrt(L) * fabs(idy_r);
            sa = c - w;
            sb = c + w;
        } else {
            ok = (iry * idx) * (iry * idx) <= (int64_t)s.r * s.r * iL;
        }
        if (idx != 0) {                          // 0 <= (x - x0) dx + ry dy <= L
            const double idx_r = render_rcp(dx);
            const double t0 = x0 - ry * dy * idx_r, t1 = x0 + (L - ry * dy) * idx_r;
            sa = fmax(sa, fmin(t0, t1));
            sb = fmin(sb, fmax(t0, t1));
        } else {
            ok = ok && iry * idy >= 0 && iry * idy <= iL;
        }
        if (ok && sa <= sb + 1e-6) { a = fmin(a, sa); b = fmax(b, sb); }
    }
    *lo = a;
    *hi = b;
    return a <= b;
}

__device__ __forceinline__ uint8_t render_blend(uint32_t c, uint32_t o, uint32_t a) {
    return (uint8_t)((c * a + o * (255u - a) + 127u) / 255u);
}

__global__ void __launch_bounds__(kRenderThreads, 4)
k_render(const uint8_t* __restrict__ bg, int64_t bg_stride, int f0, int H, int W, int pitch, int band_rows,
         const uint32_t* __restrict__ bits, const int32_t* __restrict__ bbox, int64_t n_masks,
         const a3d_layer_t* __restrict__ layers, const int64_t* __restrict__ layer_begin,
         const a3d_segment_t* __restrict__ segs, const int64_t* __restrict__ seg_begin, uint8_t* __restrict__ out) {
    extern __shared__ uint4 s_dyn[];
    __shared__ int4 s_lay[kRenderCap];            // {mask | outline << 31, rgba, rows lo | hi << 16, words lo | hi << 16}
    __shared__ RenderSeg s_seg[kRenderCap];
    __shared__ int s_warp[kRenderThreads / 32];
    const int f = f0 + blockIdx.y;
    const int r0 = blockIdx.x * band_rows, r1 = min(H, r0 + band_rows);
    const int64_t row_bytes = (int64_t)W * 3;
    const int64_t nbytes = (r1 - r0) * row_bytes;
    uint8_t* o = out + ((int64_t)f * H + r0) * row_bytes;
    uint8_t* stage = (uint8_t*)s_dyn + ((uintptr_t)o & 15);        // same phase as `out`: aligned write-out
    render_copy(stage, bg + (int64_t)f * bg_stride + r0 * row_bytes, nbytes);
    const int nw = (W + 31) >> 5;
    const int items = (r1 - r0) * nw;
    int64_t li = layer_begin[f], si = seg_begin[f];
    const int64_t le = layer_begin[f + 1], se = seg_begin[f + 1];
    while (li < le || si < se) {
        int nl = 0, ns = 0;
        if (li < le) {
            const int64_t k = li + threadIdx.x;
            bool keep = false;
            int4 e = make_int4(0, 0, 0, 0);
            if (k < le) {
                const a3d_layer_t L = layers[k];
                if (L.mask >= 0 && L.mask < n_masks) {
                    int rmin = 0, rmax = H - 1, wmin = 0, wmax = nw - 1;
                    if (bbox) {
                        const int4 b = ((const int4*)bbox)[L.mask];
                        rmin = max(b.x, 0); rmax = min(b.y, H - 1); wmin = max(b.z, 0); wmax = min(b.w, nw - 1);
                    }
                    rmin = max(rmin, r0);
                    rmax = min(rmax, r1 - 1);
                    keep = rmin <= rmax && wmin <= wmax;
                    const uint32_t rgba = L.rgba[0] | (uint32_t)L.rgba[1] << 8 | (uint32_t)L.rgba[2] << 16 |
                                          (uint32_t)L.rgba[3] << 24;
                    e = make_int4(L.mask | (L.kind == A3D_LAYER_OUTLINE ? (int)0x80000000u : 0), (int)rgba,
                                  rmin | rmax << 16, wmin | wmax << 16);
                }
            }
            const int slot = render_rank(keep, s_warp, &nl);
            if (keep) s_lay[slot] = e;
            li += kRenderCap;
        }
        if (li >= le && si < se) {
            const int64_t k = si + threadIdx.x;
            bool keep = false;
            a3d_segment_t S{};
            int bx0 = 0, bx1 = -1, by0 = 0, by1 = -1;
            if (k < se) {
                S = segs[k];
                bx0 = max(0, min(S.x0, S.x1) - S.radius);
                bx1 = min(W - 1, max(S.x0, S.x1) + S.radius);
                by0 = max(r0, min(S.y0, S.y1) - S.radius);
                by1 = min(r1 - 1, max(S.y0, S.y1) + S.radius);
                keep = bx0 <= bx1 && by0 <= by1;
            }
            const int slot = render_rank(keep, s_warp, &ns);
            if (keep) {
                RenderSeg& e = s_seg[slot];
                e.x0 = S.x0; e.y0 = S.y0; e.x1 = S.x1; e.y1 = S.y1; e.r = S.radius;
                e.rgb = S.rgb[0] | (uint32_t)S.rgb[1] << 8 | (uint32_t)S.rgb[2] << 16;
                e.bx0 = bx0; e.bx1 = bx1; e.by0 = by0; e.by1 = by1;
            }
            si += kRenderCap;
        }
        __syncthreads();
        for (int it = threadIdx.x; it < items; it += kRenderThreads) {
            const int rr = it / nw, j = it - rr * nw, y = r0 + rr;
            uint8_t* px = stage + rr * row_bytes + j * 96;
            const uint32_t valid = rle_valid(j, W);
            for (int k = 0; k < nl; ++k) {
                const int4 e = s_lay[k];
                if (y < (e.z & 0xffff) || y > (e.z >> 16) || j < (e.w & 0xffff) || j > (e.w >> 16)) continue;
                const uint32_t* mb = bits + ((int64_t)(e.x & 0x7fffffff) * H + y) * pitch;
                uint32_t cov = mb[j] & valid;
                if (!cov) continue;
                if (e.x < 0) {                     // outline: set pixels with an unset 4-neighbour
                    const uint32_t up = y > 0 ? mb[j - pitch] : 0u;
                    const uint32_t dn = y + 1 < H ? mb[j + pitch] : 0u;
                    const uint32_t lw = j > 0 ? mb[j - 1] : 0u;
                    const uint32_t rw = j + 1 < nw ? mb[j + 1] : 0u;
                    const uint32_t left = (cov << 1) | (lw >> 31), right = (cov >> 1) | (rw << 31);
                    cov &= ~(up & dn & left & right);
                }
                const uint32_t c0 = e.y & 255, c1 = (e.y >> 8) & 255, c2 = (e.y >> 16) & 255, a = (uint32_t)e.y >> 24;
                while (cov) {
                    const int i = __ffs(cov) - 1;
                    cov &= cov - 1;
                    uint8_t* p = px + 3 * i;
                    p[0] = render_blend(c0, p[0], a);
                    p[1] = render_blend(c1, p[1], a);
                    p[2] = render_blend(c2, p[2], a);
                }
            }
            const int xa = 32 * j, xb = min(W, xa + 32) - 1;
            for (int k = 0; k < ns; ++k) {
                const RenderSeg s = s_seg[k];
                if (y < s.by0 || y > s.by1 || xb < s.bx0 || xa > s.bx1) continue;
                double lo, hi;
                if (!render_seg_row(s, y, &lo, &hi)) continue;
                const int xs = max(max(xa, s.bx0), (int)floor(fmax(lo, -1e9)) - 1);
                const int xe = min(min(xb, s.bx1), (int)ceil(fmin(hi, 1e9)) + 1);
                for (int x = xs; x <= xe; ++x) {
                    if (!render_seg_hit(s, x, y)) continue;
                    uint8_t* p = px + 3 * (x - xa);
                    p[0] = s.rgb & 255;
                    p[1] = (s.rgb >> 8) & 255;
                    p[2] = (s.rgb >> 16) & 255;
                }
            }
        }
        __syncthreads();
    }
    __syncthreads();
    render_copy(o, stage, nbytes);
}

extern "C" {

int a3d_render(const uint8_t* background, int64_t bg_frame_stride, int n_frames, int H, int W,
               const uint32_t* bits, const int32_t* bbox, int64_t n_masks,
               const a3d_layer_t* layers, const int64_t* layer_begin,
               const a3d_segment_t* segs, const int64_t* seg_begin, uint8_t* out, void* stream) {
    if (n_frames < 0 || H <= 0 || W <= 0 || n_masks < 0 || bg_frame_stride < 0)
        return fail(A3D_EINVAL, "a3d_render: bad shape n_frames=%d %dx%d n_masks=%lld stride=%lld", n_frames, H, W,
                    (long long)n_masks, (long long)bg_frame_stride);
    if (H > A3D_RENDER_MAX_SIDE || W > A3D_RENDER_MAX_SIDE)
        return fail(A3D_ELIMIT, "a3d_render: %dx%d frame exceeds %d pixels a side", H, W, A3D_RENDER_MAX_SIDE);
    if (n_frames == 0) return A3D_OK;
    if (!background || !layer_begin || !seg_begin || !out || (n_masks > 0 && !bits))
        return fail(A3D_EINVAL, "a3d_render: null pointer");
    int band_rows = kRenderStageBytes / (3 * W);
    band_rows = band_rows < 1 ? 1 : (band_rows > H ? H : band_rows);
    const int smem = band_rows * 3 * W + 16;
    A3D_CUDA_TRY(cudaFuncSetAttribute(k_render, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const unsigned bands = (unsigned)((H + band_rows - 1) / band_rows);
    for (int f0 = 0; f0 < n_frames; f0 += 65535) {
        const unsigned nf = (unsigned)(n_frames - f0 < 65535 ? n_frames - f0 : 65535);
        k_render<<<dim3(bands, nf), kRenderThreads, smem, (cudaStream_t)stream>>>(
            background, bg_frame_stride, f0, H, W, pitch_words(W), band_rows, bits, bbox, n_masks, layers, layer_begin,
            segs, seg_begin, out);
        A3D_CUDA_TRY(cudaGetLastError());
    }
    return A3D_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------
// plane maps (a3d_plane_maps): per-pixel depth of the nearest planar mask and that mask's colour.
// One CTA per (frame, band of rows).  The frame's layers whose box touches the band are culled into shared
// memory kPlaneCap at a time, in list order; one warp takes one packed word of the band (32 pixels of a row),
// one lane one pixel, and runs k_unproject's float64 ray/plane chain for every culled layer that has the pixel
// set.  The band's running best (z, colour) lives in shared memory across the batches; the band's depth and
// RGB bytes are written once at the end, contiguous and coalesced.  HBM traffic: the outputs and the mask
// words inside the culled layers' boxes.
// ---------------------------------------------------------------------------
constexpr int kPlaneThreads = kRenderThreads;       // render_rank's block size
constexpr int kPlaneCap = kPlaneThreads;            // layers culled per batch: one per thread
constexpr int kPlaneBandPx = 4096;                  // target pixel slots (32 per packed word) of a band

__global__ void __launch_bounds__(kPlaneThreads)
k_plane_maps(const Cam cam, int f0, int band_rows, const uint32_t* __restrict__ bits, const int32_t* __restrict__ bbox,
             int64_t n_masks, const a3d_plane_layer_t* __restrict__ layers, const int64_t* __restrict__ layer_begin,
             uint32_t bg, float* __restrict__ depth_out, uint8_t* __restrict__ rgb_out) {
    extern __shared__ float s_best[];               // [slots] running best z (+inf: none), then [slots] its rgb
    __shared__ int4 s_lay[kPlaneCap];               // {mask, rgb, rows lo | hi << 16, words lo | hi << 16}
    __shared__ float4 s_pl[kPlaneCap];              // {n0, n1, n2, offset}
    __shared__ int s_warp[kPlaneThreads / 32];
    const float INFf = __int_as_float(0x7f800000);
    const int H = cam.H, W = cam.W, pitch = cam.pitch, nw = (W + 31) >> 5;
    const int f = f0 + blockIdx.y;
    const int r0 = blockIdx.x * band_rows, r1 = min(H, r0 + band_rows);
    const int items = (r1 - r0) * nw;
    float* s_z = s_best;
    uint32_t* s_c = reinterpret_cast<uint32_t*>(s_best + band_rows * nw * 32);
    for (int i = threadIdx.x; i < items * 32; i += kPlaneThreads) {
        s_z[i] = INFf;
        s_c[i] = bg;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t le = layer_begin[f + 1];
    for (int64_t li = layer_begin[f]; li < le; li += kPlaneCap) {
        const int64_t k = li + threadIdx.x;
        bool keep = false;
        int4 e = make_int4(0, 0, 0, 0);
        float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k < le) {
            const a3d_plane_layer_t L = layers[k];
            if (L.mask >= 0 && L.mask < n_masks) {
                int rmin = 0, rmax = H - 1, wmin = 0, wmax = nw - 1;
                if (bbox) {
                    const int4 b = ((const int4*)bbox)[L.mask];
                    rmin = max(b.x, 0); rmax = min(b.y, H - 1); wmin = max(b.z, 0); wmax = min(b.w, nw - 1);
                }
                rmin = max(rmin, r0);
                rmax = min(rmax, r1 - 1);
                keep = rmin <= rmax && wmin <= wmax;
                e = make_int4(L.mask, (int)(L.rgb[0] | (uint32_t)L.rgb[1] << 8 | (uint32_t)L.rgb[2] << 16),
                              rmin | rmax << 16, wmin | wmax << 16);
                p = make_float4(L.normal[0], L.normal[1], L.normal[2], L.offset);
            }
        }
        int nl;
        const int slot = render_rank(keep, s_warp, &nl);
        if (keep) {
            s_lay[slot] = e;
            s_pl[slot] = p;
        }
        __syncthreads();
        for (int it = warp; it < items; it += kPlaneThreads / 32) {
            const int rr = it / nw, j = it - rr * nw, y = r0 + rr, x = 32 * j + lane;
            if (x >= W) continue;
            float best = s_z[32 * it + lane];
            uint32_t col = s_c[32 * it + lane];
            for (int q = 0; q < nl; ++q) {
                const int4 L = s_lay[q];
                if (y < (L.z & 0xffff) || y > (L.z >> 16) || j < (L.w & 0xffff) || j > (L.w >> 16)) continue;
                const uint32_t word = bits[((int64_t)L.x * H + y) * pitch + j];
                if (!((word >> lane) & 1u)) continue;
                // the ray is recomputed per layer: nothing float64 stays live across the division's slow path
                const double xd = (double)x, yd = (double)y;
                double rx, ry, rz;
                if (cam.sparse) {
                    rx = __dadd_rn(__dmul_rn(cam.k[0], xd), cam.k[2]);
                    ry = __dadd_rn(__dmul_rn(cam.k[4], yd), cam.k[5]);
                    rz = 1.0;
                } else {
                    rx = __dadd_rn(__dadd_rn(__dmul_rn(cam.k[0], xd), __dmul_rn(cam.k[1], yd)), cam.k[2]);
                    ry = __dadd_rn(__dadd_rn(__dmul_rn(cam.k[3], xd), __dmul_rn(cam.k[4], yd)), cam.k[5]);
                    rz = __dadd_rn(__dadd_rn(__dmul_rn(cam.k[6], xd), __dmul_rn(cam.k[7], yd)), cam.k[8]);
                }
                const float4 P = s_pl[q];
                const double dot = __dadd_rn(__dadd_rn(__dmul_rn((double)P.x, rx), __dmul_rn((double)P.y, ry)),
                                             __dmul_rn((double)P.z, rz));
                const float z = __double2float_rn(__dmul_rn(__ddiv_rn((double)P.w, dot), rz));
                if (z > 0.f && z < best) {         // best <= +inf: a finite z only; NaN fails both; ties keep the first
                    best = z;
                    col = (uint32_t)L.y;
                }
            }
            s_z[32 * it + lane] = best;
            s_c[32 * it + lane] = col;
        }
        __syncthreads();
    }
    __syncthreads();
    for (int rr = 0; rr < r1 - r0; ++rr) {          // row by row: no division by W per output element
        const int64_t row = (int64_t)f * H + r0 + rr;
        if (depth_out) {
            const float* zr = s_z + 32 * rr * nw;
            float* o = depth_out + row * W;
            for (int x = threadIdx.x; x < W; x += kPlaneThreads) {
                const float z = zr[x];
                o[x] = z < INFf ? z : 0.f;
            }
        }
        if (rgb_out) {
            const uint32_t* cr = s_c + 32 * rr * nw;
            uint8_t* o = rgb_out + row * W * 3;
            for (int i = threadIdx.x; i < 3 * W; i += kPlaneThreads) {
                const int px = (int)((unsigned)i / 3u);
                o[i] = (uint8_t)(cr[px] >> (8 * (i - 3 * px)));
            }
        }
    }
}

extern "C" {

int a3d_plane_maps(const a3d_camera_t* cam, int n_frames, const uint32_t* bits, const int32_t* bbox, int64_t n_masks,
                   const a3d_plane_layer_t* layers, const int64_t* layer_begin, const uint8_t bg_rgb[3],
                   float* depth_out, uint8_t* rgb_out, void* stream) {
    if (!cam) return fail(A3D_EINVAL, "a3d_plane_maps: null camera");
    const int H = cam->H, W = cam->W;
    if (n_frames < 0 || H <= 0 || W <= 0 || n_masks < 0)
        return fail(A3D_EINVAL, "a3d_plane_maps: bad shape n_frames=%d %dx%d n_masks=%lld", n_frames, H, W,
                    (long long)n_masks);
    if (H > A3D_RENDER_MAX_SIDE || W > A3D_RENDER_MAX_SIDE)
        return fail(A3D_ELIMIT, "a3d_plane_maps: %dx%d frame exceeds %d pixels a side", H, W, A3D_RENDER_MAX_SIDE);
    if (n_frames == 0 || (!depth_out && !rgb_out)) return A3D_OK;
    if (!layer_begin || (n_masks > 0 && !bits) || (rgb_out && !bg_rgb))
        return fail(A3D_EINVAL, "a3d_plane_maps: null pointer");
    Cam c;
    memcpy(c.k, cam->kinv, sizeof(c.k));
    c.f = cam->f; c.cx = cam->cx; c.cy = cam->cy;
    c.H = H; c.W = W; c.pitch = pitch_words(W);
    c.sparse = (c.k[1] == 0.0 && c.k[3] == 0.0 && c.k[6] == 0.0 && c.k[7] == 0.0 && c.k[8] == 1.0);
    const uint32_t bg = rgb_out ? (bg_rgb[0] | (uint32_t)bg_rgb[1] << 8 | (uint32_t)bg_rgb[2] << 16) : 0u;
    const int row_slots = 32 * ((W + 31) >> 5);
    int band_rows = kPlaneBandPx / row_slots;
    band_rows = band_rows < 1 ? 1 : (band_rows > H ? H : band_rows);
    const int smem = band_rows * row_slots * 8;
    A3D_CUDA_TRY(cudaFuncSetAttribute(k_plane_maps, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const unsigned bands = (unsigned)((H + band_rows - 1) / band_rows);
    for (int f0 = 0; f0 < n_frames; f0 += 65535) {
        const unsigned nf = (unsigned)(n_frames - f0 < 65535 ? n_frames - f0 : 65535);
        k_plane_maps<<<dim3(bands, nf), kPlaneThreads, smem, (cudaStream_t)stream>>>(
            c, f0, band_rows, bits, bbox, n_masks, layers, layer_begin, bg, depth_out, rgb_out);
        A3D_CUDA_TRY(cudaGetLastError());
    }
    return A3D_OK;
}

}  // extern "C"
