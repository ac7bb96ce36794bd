// Stand-alone probe of tcgen05.mma kind::mxf4 (e2m1 x e2m1 -> f32, UE8M0 block scales) as k_score_mma
// uses it: mask words expanded to nibbles (bit -> 0x2 = 1.0, 0 -> 0.0) in the no-swizzle K-major
// layout [word position][row][16 B] with padded position slots, one MMA (K = 64) per two positions,
// every scale byte 0x7F (= 1.0) in TMEM columns 256..511, accumulator in TMEM columns 0..255.
//
// It pins the instruction descriptor and the descriptor fields, and checks that the accumulator
// counts exactly: every product is 0 or 1, so an f32 accumulator with a full 24-bit significand holds
// every count below 2^24 exactly.  The contraction runs over 2^21 + 96 pixels and all 128 x N
// accumulators are read at checkpoints past 2^14, 2^16, 2^20, 786 432 (= 1024 x 768) and 2^21,
// against an integer popcount reference.  Rows: all ones, random at several densities, and a
// candidate with one bit per 64-pixel block (adds 1 per MMA onto a large sum).
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O2 -Xcompiler -mpopcnt -o tools/mma_probe tools/mma_probe.cu
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <cuda_runtime.h>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(2); } } while (0)

constexpr int kM = 128;
constexpr int kNMax = 240;
constexpr int kPos = 8;                 // word positions per round = 4 MMAs
constexpr int kPad = 16;                // as k_score_mma at 8 positions per stage: slots 16-byte aligned only
constexpr int kWords = (1 << 16) + 3;   // words per mask row: 2^21 + 96 pixels (odd: a zero-filled tail chunk)
constexpr int kChecks = 6;
__constant__ int c_check[kChecks];      // word counts after which the accumulators are read

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok, spins = 0;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (!ok && ++spins > (1u << 24)) __trap();
    } while (!ok);
}
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) | ((uint64_t)8 << 32) | (1ull << 46);
}

// A: [128][kWords], B: [N][kWords] mask words; D: [kChecks][128][N] raw f32 accumulator bits
__global__ void __launch_bounds__(128) probe(const uint32_t* A, const uint32_t* B, int N, uint32_t* D) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint32_t tmem_base;
    __shared__ __align__(8) uint64_t bar;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t slotA = kM * 16 + kPad, slotB = (uint32_t)N * 16 + kPad;
    const uint32_t sA = smem_u32(smem), sB = sA + kPos * slotA;
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 0) {
        mbar_init(smem_u32(&bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base;
    {   // scale factors: 0x7F (UE8M0 2^0) in every byte of columns 256..511 of all 128 lanes
        const uint32_t one = 0x7F7F7F7Fu;
        for (int c = 256; c < 512; c += 8)
            asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};"
                         ::"r"(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c), "r"(one) : "memory");
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // e2m1 x e2m1 -> f32, UE8M0 scales, K-major, M = 128
    const uint32_t idesc = (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | (1u << 23) | ((uint32_t)(kM >> 4) << 24);
    int chk = 0;
    uint32_t phase = 0;
    for (int w0 = 0; w0 < kWords; w0 += kPos) {
        const int nw = min(kPos, kWords - w0);
        for (int i = tid; i < (kM + N) * kPos; i += 128) {
            const int m = i / kPos, q = i % kPos;
            const uint32_t w = q < nw ? (m < kM ? A[(size_t)m * kWords + w0 + q] : B[(size_t)(m - kM) * kWords + w0 + q]) : 0u;
            const uint32_t dst = m < kM ? sA + q * slotA + m * 16 : sB + q * slotB + (m - kM) * 16;
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"((w << 1) & 0x22222222u), "r"(w & 0x22222222u),
                         "r"((w >> 1) & 0x22222222u), "r"((w >> 2) & 0x22222222u) : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            for (int j = 0; j < (nw + 1) / 2; ++j) {
                const uint64_t da = make_desc(sA + 2 * j * slotA, slotA);
                const uint64_t db = make_desc(sB + 2 * j * slotB, slotB);
                const uint32_t acc = (w0 > 0 || j > 0) ? 1u : 0u;
                asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %6, 0;\n\t"
                             "tcgen05.mma.cta_group::1.kind::mxf4.block_scale.scale_vec::2X [%0], %1, %2, %3, [%4], [%5], p;\n\t}"
                             ::"r"(tmem), "l"(da), "l"(db), "r"(idesc), "r"(tmem + 256u), "r"(tmem + 384u), "r"(acc) : "memory");
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&bar)) : "memory");
        }
        mbar_wait(smem_u32(&bar), phase);
        phase ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (chk < kChecks && w0 + nw == c_check[chk]) {
            for (int c0 = 0; c0 < N; c0 += 16) {
                uint32_t r[16];
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                             : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                               "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                             : "r"(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                for (int j = 0; j < 16; ++j) D[((size_t)chk * kM + warp * 32 + lane) * N + c0 + j] = r[j];
            }
            ++chk;
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();                                   // smem and accumulator reads done before the next round
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

int main() {
    // checkpoints (words): just past 2^14 and 2^16 pixels, then 786 432, 2^20, 2^20 + 256 and 2^21 + 96 pixels
    const int checks[kChecks] = {(1 << 9) + 8, (1 << 11) + 8, 24576, (1 << 15), (1 << 15) + 8, kWords};
    CK(cudaMemcpyToSymbol(c_check, checks, sizeof(checks)));
    uint64_t s = 0x9E3779B97F4A7C15ull;
    auto rnd = [&]() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return (uint32_t)s; };
    auto word = [&](int kind) -> uint32_t {   // density: 1, 1/2, 1/4, 3/4, 31/32
        switch (kind) {
            case 0: return 0xFFFFFFFFu;
            case 1: return rnd();
            case 2: return rnd() & rnd();
            case 3: return rnd() | rnd();
            default: return ~(rnd() & rnd() & rnd() & rnd() & rnd());
        }
    };
    std::vector<uint32_t> A((size_t)kM * kWords), B((size_t)kNMax * kWords);
    for (int m = 0; m < kM; ++m)
        for (int w = 0; w < kWords; ++w) A[(size_t)m * kWords + w] = word(m % 5);
    for (int n = 0; n < kNMax; ++n)
        for (int w = 0; w < kWords; ++w) {
            uint32_t v = word((n + 1) % 6 == 5 ? 0 : (n % 5));
            if (n % 6 == 5) v = (w & 1) ? 0u : (1u << (w % 31));   // one bit per 64 pixels
            B[(size_t)n * kWords + w] = v;
        }
    // integer reference at every checkpoint
    std::vector<int64_t> ref((size_t)kChecks * kM * kNMax);
    for (int m = 0; m < kM; ++m)
        for (int n = 0; n < kNMax; ++n) {
            const uint32_t* a = &A[(size_t)m * kWords];
            const uint32_t* b = &B[(size_t)n * kWords];
            int64_t acc = 0;
            int c = 0;
            for (int w = 0; w < kWords; ++w) {
                acc += __builtin_popcount(a[w] & b[w]);
                if (w + 1 == checks[c]) ref[((size_t)c++ * kM + m) * kNMax + n] = acc;
            }
        }
    uint32_t *dA, *dB, *dD;
    CK(cudaMalloc(&dA, A.size() * 4)); CK(cudaMalloc(&dB, B.size() * 4));
    CK(cudaMalloc(&dD, (size_t)kChecks * kM * kNMax * 4));
    CK(cudaMemcpy(dA, A.data(), A.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dB, B.data(), B.size() * 4, cudaMemcpyHostToDevice));
    int bad_total = 0;
    for (int N : {16, 192, 240}) {
        const size_t smem = (size_t)kPos * (kM * 16 + kPad) + (size_t)kPos * (N * 16 + kPad);
        CK(cudaFuncSetAttribute(probe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK(cudaMemset(dD, 0xff, (size_t)kChecks * kM * N * 4));
        probe<<<1, 128, smem>>>(dA, dB, N, dD);
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { printf("N=%d: kernel error %s\n", N, cudaGetErrorString(e)); return 3; }
        std::vector<uint32_t> out((size_t)kChecks * kM * N);
        CK(cudaMemcpy(out.data(), dD, out.size() * 4, cudaMemcpyDeviceToHost));
        for (int c = 0; c < kChecks; ++c) {
            int bad = 0;
            int64_t vmax = 0, first_bad_ref = -1;
            float first_bad_got = 0.f;
            for (int m = 0; m < kM; ++m)
                for (int n = 0; n < N; ++n) {
                    const int64_t r = ref[((size_t)c * kM + m) * kNMax + n];
                    float f;
                    memcpy(&f, &out[((size_t)c * kM + m) * N + n], 4);
                    vmax = r > vmax ? r : vmax;
                    if ((double)f != (double)r) {
                        if (!bad) { first_bad_ref = r; first_bad_got = f; }
                        ++bad;
                    }
                }
            printf("N=%3d after %8d pixels: %5d / %d accumulators wrong, largest count %lld", N, checks[c] * 32, bad, kM * N,
                   (long long)vmax);
            if (bad) printf("  (first: got %.1f, want %lld)", first_bad_got, (long long)first_bad_ref);
            printf("\n");
            bad_total += bad;
        }
    }
    printf(bad_total == 0 ? "PROBE OK: kind::mxf4 counts exactly up to 2^21 + 96 (idesc e2m1 x e2m1 -> f32, UE8M0 = 0x7F)\n"
                          : "PROBE MISMATCH\n");
    return bad_total != 0;
}
