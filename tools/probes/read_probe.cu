// probe: achieved HBM read bandwidth for "stream the in-range box of every image" under different structures.
// usage: read_probe <variant> [W=256] [box=230] [B=16384]
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cuda.h>
#include <cuda_runtime.h>
#include <cudaTypedefs.h>
#include "mog_common.cuh"
using namespace mog;

// mbarrier / tensor-copy helpers (the library itself issues no tensor copies)
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, unsigned parity) {
    unsigned ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// bounded: a transaction that never completes (a bug) traps instead of hanging the device
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    for (int it = 0; it < (1 << 24); ++it)
        if (mbar_try_wait(bar, parity)) return;
    asm volatile("trap;");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int x, int y, int z) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(reinterpret_cast<unsigned long long>(map)), "r"(smem_u32(bar)), "r"(x), "r"(y), "r"(z)
                 : "memory");
}

// (a) warp per image, strips of SWC columns (NJC chunks), RB rows per batch, register loads
template <int NJC, int RB>
__global__ void __launch_bounds__(64) k_warp_strips(const float* g, float* out, int B, int W, int box, int off) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int b = blockIdx.x * 2 + warp; b < B; b += gridDim.x * 2) {
        const float* gb = g + (size_t)b * W * W + (size_t)off * W + off;
        float acc = 0.f;
        for (int js = 0; js < box; js += 32 * NJC) {
            for (int i0 = 0; i0 < box; i0 += RB) {
                float v[RB][NJC];
#pragma unroll
                for (int r = 0; r < RB; ++r)
#pragma unroll
                    for (int c = 0; c < NJC; ++c) {
                        const int i = min(i0 + r, box - 1), j = min(js + 32 * c + lane, box - 1);
                        v[r][c] = __ldg(gb + (size_t)i * W + j);
                    }
#pragma unroll
                for (int r = 0; r < RB; ++r)
#pragma unroll
                    for (int c = 0; c < NJC; ++c) acc += v[r][c];
            }
        }
        acc = warp_sum(acc);
        if (lane == 0) out[b] = acc;
    }
}

// (f) CTA of NW warps per image: warp w takes strip w, w+NW, ... (64 columns each), RB rows per batch
template <int NW, int RB>
__global__ void __launch_bounds__(NW * 32) k_cta_strips(const float* g, float* out, int B, int W, int box, int off) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ float red[NW];
    for (int b = blockIdx.x; b < B; b += gridDim.x) {
        const float* gb = g + (size_t)b * W * W + (size_t)off * W + off;
        float acc = 0.f;
        for (int js = warp * 64; js < box; js += 64 * NW) {
            for (int i0 = 0; i0 < box; i0 += RB) {
                float v[RB][2];
#pragma unroll
                for (int r = 0; r < RB; ++r)
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        const int i = min(i0 + r, box - 1), j = min(js + 32 * c + lane, box - 1);
                        v[r][c] = __ldg(gb + (size_t)i * W + j);
                    }
#pragma unroll
                for (int r = 0; r < RB; ++r) acc += v[r][0] + v[r][1];
            }
        }
        acc = warp_sum(acc);
        if (lane == 0) red[warp] = acc;
        __syncthreads();
        if (threadIdx.x == 0) { float s = 0; for (int w = 0; w < NW; ++w) s += red[w]; out[b] = s; }
        __syncthreads();
    }
}

// (c,d,e) warp per image, TMA tiles of TRxTW through a ring of NST stages
template <int TR, int TW, int NST>
__global__ void __launch_bounds__(64) k_tma(const __grid_constant__ CUtensorMap tm, float* out, int B, int W, int box, int off) {
    extern __shared__ __align__(128) unsigned char s_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int TB = TR * TW * 4;
    unsigned char* base = s_raw + warp * (NST * TB + 128);
    float* ring = reinterpret_cast<float*>(base);
    uint64_t* bar = reinterpret_cast<uint64_t*>(base + NST * TB);
    if (lane == 0) {
        for (int s = 0; s < NST; ++s) mbar_init(bar + s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncwarp();
    unsigned phase = 0;
    const int x0 = off & ~3;
    const int ntx = (off + box - x0 + TW - 1) / TW, nty = (box + TR - 1) / TR, nt = ntx * nty;
    for (int b = blockIdx.x * 2 + warp; b < B; b += gridDim.x * 2) {
        float acc = 0.f;
        auto issue = [&](int t) {
            if (lane == 0) {
                const int st = t % NST, tx = t / nty, ty = t % nty;
                mbar_expect_tx(bar + st, TB);
                tma_load_3d(reinterpret_cast<unsigned char*>(ring) + st * TB, &tm, bar + st, x0 + tx * TW, off + ty * TR, b);
            }
        };
        for (int t = 0; t < min(NST, nt); ++t) issue(t);
        for (int t = 0; t < nt; ++t) {
            const int st = t % NST;
            mbar_wait(bar + st, (phase >> st) & 1u);
            phase ^= 1u << st;
            const float* tile = ring + st * (TB / 4);
            for (int k = lane; k < TR * TW; k += 32) acc += tile[k];
            __syncwarp();
            if (t + NST < nt) issue(t + NST);
        }
        acc = warp_sum(acc);
        if (lane == 0) out[b] = acc;
    }
}

// (g) reference: plain streaming read of the whole tensor
__global__ void k_stream(const float4* g, float* out, size_t n4) {
    float acc = 0.f;
    for (size_t k = blockIdx.x * (size_t)blockDim.x + threadIdx.x; k < n4; k += (size_t)gridDim.x * blockDim.x) {
        const float4 v = __ldg(g + k);
        acc += v.x + v.y + v.z + v.w;
    }
    if (acc == 123.456f) out[0] = acc;
}

template <typename F>
static float time_it(F f) {
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    f(); f();
    cudaEventRecord(e0);
    for (int k = 0; k < 5; ++k) f();
    cudaEventRecord(e1); cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    return ms / 5;
}

int main(int argc, char** argv) {
    const int W = argc > 2 ? atoi(argv[2]) : 256, box = argc > 3 ? atoi(argv[3]) : 230, B = argc > 4 ? atoi(argv[4]) : 16384;
    const int off = (W - box) / 2 + 1;
    const size_t n = (size_t)B * W * W;
    float *g, *out;
    cudaMalloc(&g, n * 4); cudaMalloc(&out, B * 4 + 16); cudaMemset(g, 0, n * 4);
    void* f = nullptr; cudaDriverEntryPointQueryResult q;
    cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q);
    auto enc = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(f);
    auto mk = [&](int bw, int bh) {
        CUtensorMap tm;
        const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)W, (cuuint64_t)B}; const cuuint64_t strides[2] = {(cuuint64_t)W * 4, (cuuint64_t)W * W * 4};
        const cuuint32_t bx[3] = {(cuuint32_t)bw, (cuuint32_t)bh, 1}; const cuuint32_t es[3] = {1, 1, 1};
        CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, g, dims, strides, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) printf("encode failed %d\n", (int)r);
        return tm;
    };
    const double box_gb = (double)B * box * box * 4 / 1e9;
    auto report = [&](const char* name, float ms) {
        cudaError_t e = cudaDeviceSynchronize();
        printf("%-34s %8.1f us  %7.0f GB/s of box bytes (%s)\n", name, ms * 1e3, box_gb / (ms * 1e-3), cudaGetErrorString(e));
    };
    const int grid = 148 * 16;
    report("stream whole tensor (float4)", time_it([&] { k_stream<<<148 * 8, 512>>>((const float4*)g, out, n / 4); }) * (float)(box_gb / (n * 4 / 1e9)));
    report("warp/img strips64 RB2", time_it([&] { k_warp_strips<2, 2><<<grid, 64>>>(g, out, B, W, box, off); }));
    report("warp/img strips64 RB4", time_it([&] { k_warp_strips<2, 4><<<grid, 64>>>(g, out, B, W, box, off); }));
    report("warp/img strips64 RB8", time_it([&] { k_warp_strips<2, 8><<<grid, 64>>>(g, out, B, W, box, off); }));
    report("warp/img strips128 RB4", time_it([&] { k_warp_strips<4, 4><<<grid, 64>>>(g, out, B, W, box, off); }));
    report("warp/img fullrow(256) RB2", time_it([&] { k_warp_strips<8, 2><<<grid, 64>>>(g, out, B, W, box, off); }));
    report("warp/img fullrow(256) RB4", time_it([&] { k_warp_strips<8, 4><<<grid, 64>>>(g, out, B, W, box, off); }));
    report("cta4/img strips64 RB4", time_it([&] { k_cta_strips<4, 4><<<148 * 8, 128>>>(g, out, B, W, box, off); }));
    report("cta4/img strips64 RB8", time_it([&] { k_cta_strips<4, 8><<<148 * 8, 128>>>(g, out, B, W, box, off); }));
    report("cta8/img strips64 RB4 (2 img rows)", time_it([&] { k_cta_strips<8, 4><<<148 * 4, 256>>>(g, out, B, W, box, off); }));
#define TMA_CASE(TR, TW, NST, CTAS)                                                                                     \
    {                                                                                                                   \
        CUtensorMap tm = mk(TW, TR);                                                                                    \
        const int smem = 2 * (NST * TR * TW * 4 + 128);                                                                 \
        cudaFuncSetAttribute(k_tma<TR, TW, NST>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);                    \
        report("tma " #TR "x" #TW " st" #NST " ctas/sm " #CTAS, time_it([&] { k_tma<TR, TW, NST><<<148 * CTAS, 64, smem>>>(tm, out, B, W, box, off); })); \
    }
    TMA_CASE(8, 64, 4, 8)
    TMA_CASE(8, 64, 4, 4)
    TMA_CASE(32, 64, 3, 4)
    TMA_CASE(8, 256, 3, 4)
    TMA_CASE(16, 256, 3, 2)
    TMA_CASE(32, 256, 2, 1)
    TMA_CASE(16, 128, 3, 4)
    return 0;
}
