// Warp-per-image sampler kernels (sm_100a).
//
// The images of this workload are small (28x28 ... 256x256, one channel) and there are thousands of
// them, so one WARP owns one image: no block barriers, 32-64 independent images in flight per SM to hide
// the theta -> coordinates -> gather -> store latency chain, lanes run along the contiguous (x) axis so
// every global access is a coalesced row segment.
//
// Separable thetas (t01 == t10 == 0: every AIR call site, air_number_bbox_location.py:513-531,565-584)
// use per-row / per-column axis tables (bit-identical to the per-pixel evaluation, see Theta::separable).
//   forward : per row one broadcast LDS.128 (row entry) + 4 gathers + 11 flops per pixel.
//   backward: *gather form*, no atomics, deterministic.  With W_x[j][x] / W_y[i][y] the 1-D tap weights,
//             dU = W_y^T (G W_x).  Rows are streamed in the order that makes y0 non-decreasing; for each
//             output row the warp forms T[x] = sum_j W_x[j][x] g[i][j] from a per-warp shared-memory row
//             buffer and folds it into two running source rows (y0, y0+1) held in registers; a source
//             row is stored exactly once (coalesced) when the stream moves past it, untouched rows are
//             zero-filled on the way.  dU is therefore written once and never read.
// General affine thetas fall back, inside the same kernels, to per-pixel evaluation and (backward) to a
// warp-local zero-fill followed by L2 atomics (red.global.add.f32) on the image's own dU lines.
#pragma once
#include "mog_common.cuh"

namespace mog {

constexpr int kBwdRB = 4;         // rows per batch of the streaming backward
constexpr int kFwdRB = 8;         // rows per batch of the forward hot loop
constexpr int kBwdMinBlocks = 10; // __launch_bounds__ minimum CTAs per SM of the streaming backward
constexpr int kFwdMinBlocks = 16; // ... and of the forward
constexpr int kWarpsPerCta = 2;
constexpr int kWarpThreads = kWarpsPerCta * 32;

struct FwdArgs {
    const float* U;
    const float* theta;
    float* out;
    // composite only
    const float* z_pres;
    const float* stop_sum;
    const float* canvas_in;
    float threshold;
    long long B;
    int u_div;
    int bulk_zero;  // 1: out-of-range output rows are zero-filled by the bulk-copy engine (large outputs)
    Geo g;
};

// Theta built in the kernel from the model's (s, x, y) (template parameter SXY of the kernels: 1 = read, 2 = write; theta in
// FwdArgs / BwdArgs is then unused): shift [B][2], scale [B]; the backward returns d_shift [B][2], d_scale [B] plus the
// optional add-ins g_shift_in / g_scale_in (gradients that reached the same shift / scale through the step's other sampler
// call).  A kernel parameter of its own, so that FwdArgs / BwdArgs -- and with them the code generated for the theta-taking
// kernels -- are what they were before this path existed.
struct SxyArgs {
    const float* shift;
    const float* scale;
    const float* g_shift_in;
    const float* g_scale_in;
    float* d_shift;
    float* d_scale;
};

struct BwdArgs {
    const float* U;
    const float* theta;
    const float* gout;
    float* dU;
    float* dtheta;
    // composite only
    const float* z_pres;
    const float* stop_sum;
    float* dz;
    float threshold;
    long long Bsrc;
    int u_div;
    int coop_zero;  // dU zero-fill: 0 each warp its own image (small sources); 1 the CTA sweeps its group's region
                    // linearly (large sources); 2 bulk-copy engine outside the footprint rows (large, u_div == 1, C == 1)
    Geo g;
};

// SXY (template parameter of the kernels): 0 = theta given, 1 / 2 = theta built from (s, x, y) for the read / write call;
// compile time, so that the theta-taking kernels are exactly what they were before this path existed
template <int SXY>
__device__ __forceinline__ void load_theta(Theta& th, const float* theta, const SxyArgs& sx, long long b) {
    if constexpr (SXY != 0) th.load_sxy(sx.shift, sx.scale, b, SXY);
    else th.load(theta + 6 * b);
}

// one lane writes the image's transform gradient: dtheta [6], or -- theta built from (s, x, y) -- d_shift, d_scale by the
// chain rule of Theta::load_sxy (the arithmetic of mog_air_thetas_backward)
__device__ __forceinline__ void store_dtheta(float* __restrict__ dtheta, const float* __restrict__ shift,
                                             const float* __restrict__ scale, const float* __restrict__ g_shift_in,
                                             const float* __restrict__ g_scale_in, float* __restrict__ d_shift,
                                             float* __restrict__ d_scale, int sxy_mode, long long b, const float (&p)[7]) {
    if (sxy_mode == 0) {
        if (dtheta) {
#pragma unroll
            for (int k = 0; k < 6; ++k) dtheta[6 * b + k] = p[k];
        }
        return;
    }
    if (!d_shift || !d_scale) return;
    float ds, dx, dy;
    if (sxy_mode == 1) {
        ds = p[0] + p[4]; dx = p[2]; dy = p[5];
    } else {
        const float s = __ldg(scale + b), x = __ldg(shift + 2 * b), y = __ldg(shift + 2 * b + 1);
        const float inv = 1.0f / s, inv2 = inv * inv;
        ds = (x * p[2] + y * p[5]) * inv2 - (p[0] + p[4]) * inv2;
        dx = -p[2] * inv; dy = -p[5] * inv;
    }
    if (g_scale_in) ds += __ldg(g_scale_in + b);
    if (g_shift_in) { dx += __ldg(g_shift_in + 2 * b); dy += __ldg(g_shift_in + 2 * b + 1); }
    d_scale[b] = ds;
    d_shift[2 * b] = dx; d_shift[2 * b + 1] = dy;
}

// end of one image of the backward: warp-sum the lanes' partials p = (dtheta [6], dz); lane 0 stores the transform
// gradient and, composite, dz
template <bool COMPOSITE, int SXY>
__device__ __forceinline__ void store_image_grads(const BwdArgs& a, const SxyArgs& sx, long long b, float (&p)[7], int lane) {
#pragma unroll
    for (int k = 0; k < 7; ++k) p[k] = warp_sum(p[k]);
    if (lane == 0) {
        store_dtheta(a.dtheta, sx.shift, sx.scale, sx.g_shift_in, sx.g_scale_in, sx.d_shift, sx.d_scale, SXY, b, p);
        if (COMPOSITE && a.dz) a.dz[b] = p[6];
    }
}

// forward tables of a separable theta: the taps of output column j, and the row entry {y0*Ws*4, y1*Ws*4, ay, by} of output
// row i with the source rows as byte offsets (hot forward path: pointer + 32-bit byte offset = one IMAD.WIDE.U32)
__device__ __forceinline__ Axis col_axis(const Theta& th, const Geo& g, int j) {
    return axis_tap(affine_row(th.t[0], th.t[1], th.t[2], lin_at(j, g.step_w), 0.0f), g.wsc, g.Ws);
}
__device__ __forceinline__ int4 row_entry_bytes(const Theta& th, const Geo& g, int i) {
    return pack_axis(axis_tap(affine_row(th.t[3], th.t[4], th.t[5], 0.0f, lin_at(i, g.step_h)), g.hsc, g.Hs),
                     g.Ws * (int)sizeof(float));
}

// Hide a pointer's provenance from the optimiser so it stays a 64-bit base register instead of being
// re-derived (4-6 integer instructions per tap) from the kernel argument inside the inner loop.
template <typename T>
__device__ __forceinline__ T* opaque(T* p) {
    asm volatile("" : "+l"(p));
    return p;
}
__device__ __forceinline__ float ldg_f32(const char* p) { return __ldg(reinterpret_cast<const float*>(p)); }

// zero p[0, n) with the whole CTA: one linear, fully coalesced sweep (16-byte stores between the first and last
// 16-byte boundaries).  Used for the contiguous dU / output region of the CTA's group of images: a few hundred
// long linear streams chip-wide keep DRAM pages open, thousands of per-warp streams do not.
__device__ __forceinline__ void fill_zero_cta(float* __restrict__ p, long long n) {
    if (n <= 0) return;
    const int mis = (int)((reinterpret_cast<uintptr_t>(p) >> 2) & 3);
    const long long head = min(n, (long long)((4 - mis) & 3));
    const long long nv = (n - head) >> 2;
    const long long tail = head + 4 * nv;
    if ((long long)threadIdx.x < head) p[threadIdx.x] = 0.0f;
    float4* v = reinterpret_cast<float4*>(p + head);
    for (long long k = threadIdx.x; k < nv; k += blockDim.x) v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tail + threadIdx.x < n) p[tail + threadIdx.x] = 0.0f;
}

// zero p[begin, end) with 16-byte stores between the first and last 16-byte boundaries
__device__ __forceinline__ void fill_zero(float* __restrict__ p, int begin, int end, int lane) {
    if (end <= begin) return;
    const int mis = (int)((reinterpret_cast<uintptr_t>(p + begin) >> 2) & 3);  // floats past a 16-byte boundary
    const int head = min(end, begin + ((4 - mis) & 3));
    const int nv = (end - head) >> 2;
    const int tail = head + 4 * nv;
    if (begin + lane < head) p[begin + lane] = 0.0f;
    float4* v = reinterpret_cast<float4*>(p + head);
    for (int k = lane; k < nv; k += 32) v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tail + lane < end) p[tail + lane] = 0.0f;
}

// ---- zero fill by the bulk-copy engine -----------------------------------------------------------------
// A large, mostly-zero result (the canvas-sized output of a write, the canvas-sized dU of a read) is HBM write
// traffic that needs no arithmetic.  One lane hands the contiguous zero regions to the bulk asynchronous copy
// engine (cp.async.bulk shared -> global from a small zeroed shared-memory block) and the warp goes on to its
// gathers instead of issuing ~500 16-byte store instructions per image.  The regions handed over are disjoint
// from everything the warp writes itself, so no completion wait is needed before the end of the kernel (only
// that the shared block outlives the engine's reads).  Measured on the 256x256 <-> 64x64 cell: read backward
// 1102 -> 1072 us.  (Fill alone runs in 662 us and the arithmetic alone in 489 us, yet together they take
// 1072 us: the gathers' latency grows with the write stream; L2 prefetch of the inputs, evict-first hints on
// the fills and a concurrent memset on a second stream were all measured and did not help.)
constexpr int kZeroBytes = 4096;      // zeroed shared-memory block per CTA (the largest single copy)
constexpr int kBulkMinFloats = 512;   // shorter regions: plain stores

__device__ __forceinline__ void bulk_zero_init(void* zero_block) {
    float4* z = reinterpret_cast<float4*>(zero_block);
    for (int k = threadIdx.x; k < kZeroBytes / 16; k += blockDim.x) z[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the async proxy
    __syncthreads();
}
__device__ __forceinline__ void bulk_zero_drain(int lane) {  // before exit: the engine has finished READING shared memory
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
// zero p[begin, end): 16-byte-aligned middle by the copy engine (lane 0 issues), ragged ends by the lanes
__device__ __forceinline__ void fill_zero_bulk(float* __restrict__ p, int begin, int end, int lane, unsigned zero_smem) {
    if (end - begin < kBulkMinFloats) { fill_zero(p, begin, end, lane); return; }
    const int mis = (int)((reinterpret_cast<uintptr_t>(p + begin) >> 2) & 3);
    const int head = begin + ((4 - mis) & 3);
    const int nv = (end - head) >> 2;
    const int tail = head + 4 * nv;
    if (begin + lane < head) p[begin + lane] = 0.0f;
    if (tail + lane < end) p[tail + lane] = 0.0f;
    if (lane == 0) {
        unsigned long long dst = __cvta_generic_to_global(p + head);
        for (unsigned left = (unsigned)nv * 16u; left > 0;) {
            const unsigned sz = left < (unsigned)kZeroBytes ? left : (unsigned)kZeroBytes;
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(zero_smem), "r"(sz) : "memory");
            dst += sz;
            left -= sz;
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    __syncwarp();
}

// General affine theta and/or several channels: per-pixel evaluation of transformer.py:75-116.  Kept out of
// line so that its register needs do not constrain the hot (separable, one channel) path.
// (scalar arguments only: taking the address of the kernel-parameter struct would force a local copy)
template <bool COMPOSITE>
__device__ __noinline__ void fwd_general_image(const float* __restrict__ Ub, float* __restrict__ ob,
                                               const float* __restrict__ cb, float t0, float t1, float t2, float t3,
                                               float t4, float t5, float z, bool inplace, int lane, int Hs, int Ws,
                                               int C, int Ho, int Wo, float step_w, float step_h, float wsc, float hsc) {
    Theta th;
    th.t[0] = t0; th.t[1] = t1; th.t[2] = t2; th.t[3] = t3; th.t[4] = t4; th.t[5] = t5;
    Geo g;
    g.Hs = Hs; g.Ws = Ws; g.C = C; g.Ho = Ho; g.Wo = Wo; g.N = Ho * Wo; g.S = Hs * Ws;
    g.step_w = step_w; g.step_h = step_h; g.wsc = wsc; g.hsc = hsc; g.magic_wo = 0;
    for (int j0 = 0; j0 < g.Wo; j0 += 32) {
        const int j = j0 + lane;
        if (j >= g.Wo) continue;
        for (int i = 0; i < g.Ho; ++i) {
            Axis X, Y;
            taps_general(th, g, i, j, X, Y);
            const int r0 = Y.c0 * g.Ws, r1 = Y.c1 * g.Ws;
            const long long n = (long long)i * g.Wo + j;
            if (r0 == r1) {
                // y out of range: exactly +0 in the reference (DESIGN.md "borders")
                if (COMPOSITE) {
                    if (!inplace) ob[n] = __fadd_rn(cb[n], 0.0f);
                } else {
                    for (int c = 0; c < C; ++c) ob[n * C + c] = 0.0f;
                }
                continue;
            }
            // transformer.py:112-115
            const float wa = __fmul_rn(X.a, Y.a), wb = __fmul_rn(X.a, Y.b), wc = __fmul_rn(X.b, Y.a), wd = __fmul_rn(X.b, Y.b);
            const float* pa = Ub + (long long)(r0 + X.c0) * C;
            const float* pb = Ub + (long long)(r1 + X.c0) * C;
            const float* pc = Ub + (long long)(r0 + X.c1) * C;
            const float* pd = Ub + (long long)(r1 + X.c1) * C;
            for (int c = 0; c < C; ++c) {
                // transformer.py:116  add_n in list order
                float v = __fadd_rn(__fmul_rn(wa, __ldg(pa + c)), __fmul_rn(wb, __ldg(pb + c)));
                v = __fadd_rn(v, __fmul_rn(wc, __ldg(pc + c)));
                v = __fadd_rn(v, __fmul_rn(wd, __ldg(pd + c)));
                if (COMPOSITE)
                    ob[n] = __fadd_rn(cb[n], __fmul_rn(z, v));  // :724-726
                else
                    ob[n * C + c] = v;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// forward (also the fused write+composite forward)
// ---------------------------------------------------------------------------------------------------
template <bool COMPOSITE, int SXY>
__global__ void __launch_bounds__(kWarpThreads, kFwdMinBlocks) stn_fwd_warp_kernel(const FwdArgs a, const SxyArgs sx) {
    extern __shared__ int4 s_dyn[];
    const Geo& g = a.g;
    const int C = g.C;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int4* s_row = s_dyn + warp * (g.Ho + g.Wo);  // per-warp row table, then column table
    int4* s_col = s_row + g.Ho;
    const long long nwarps = (long long)gridDim.x * kWarpsPerCta;
    const bool bulk = !COMPOSITE && a.bulk_zero;
    unsigned zero_smem = 0;
    if (bulk) {  // zeroed block behind the tables: source of the bulk zero fills
        bulk_zero_init(s_dyn + kWarpsPerCta * (g.Ho + g.Wo));
        zero_smem = (unsigned)__cvta_generic_to_shared(s_dyn + kWarpsPerCta * (g.Ho + g.Wo));
    }

    for (long long b = (long long)blockIdx.x * kWarpsPerCta + warp; b < a.B; b += nwarps) {
        Theta th;
        load_theta<SXY>(th, a.theta, sx, b);
        const bool sep = th.separable();
        float z = 1.0f;
        bool active = true;
        if (COMPOSITE) {
            z = __ldg(a.z_pres + b);
            active = a.stop_sum ? (__ldg(a.stop_sum + b) < a.threshold) : true;
        }
        const float* __restrict__ Ub = a.U + (b / a.u_div) * (long long)g.S * C;
        float* __restrict__ ob = a.out + b * (long long)g.N * C;
        // kept as a base register: re-derived from b in the chunk loop below, it costs a local-memory reload per chunk
        if (!COMPOSITE) ob = opaque(ob);
        const float* __restrict__ cb = COMPOSITE ? a.canvas_in + b * (long long)g.N : nullptr;
        const bool inplace = COMPOSITE && (a.canvas_in == a.out);

        if (COMPOSITE && !active) {
            // where(mask, ., 0): canvas + 0  (air_number_bbox_location.py:722-727)
            if (!inplace)
                for (int n = lane; n < g.N; n += 32) ob[n] = __fadd_rn(cb[n], 0.0f);
            continue;
        }
        if (sep && C == 1) {
            // ---- hot path: axis-aligned theta, one channel ------------------------------------------
            __syncwarp();  // previous image's readers are done with the row table
            int ilo = g.Ho, ihi = -1;  // in-range rows form one interval (the coordinate map is monotone)
            for (int i = lane; i < g.Ho; i += 32) {
                const int4 e = row_entry_bytes(th, g, i);
                s_row[i] = e;
                if (e.x != e.y) { ilo = min(ilo, i); ihi = max(ihi, i); }
            }
            for (int j = lane; j < g.Wo; j += 32) {
                const Axis X = col_axis(th, g, j);
                s_col[j] = make_int4(X.c0 * 4, X.c1 * 4, __float_as_int(X.a), __float_as_int(X.b));
            }
            ilo = __reduce_min_sync(0xffffffffu, ilo);
            ihi = __reduce_max_sync(0xffffffffu, ihi) + 1;
            if (ihi <= ilo) { ilo = 0; ihi = 0; }
            __syncwarp();
            // y out of range: both row taps alias one row and the weights pair up as +w/-w in add_n order,
            // so the reference's result is exactly +0 for finite inputs (DESIGN.md "borders"): those rows
            // are zero-filled with wide stores; the in-place composite has nothing to add there.
            if (!COMPOSITE) {
                if (bulk) {
                    fill_zero_bulk(ob, 0, ilo * g.Wo, lane, zero_smem);
                    fill_zero_bulk(ob, ihi * g.Wo, g.N, lane, zero_smem);
                } else {
                    fill_zero(ob, 0, ilo * g.Wo, lane);
                    fill_zero(ob, ihi * g.Wo, g.N, lane);
                }
            } else if (!inplace) {
                for (int n = lane; n < ilo * g.Wo; n += 32) ob[n] = __fadd_rn(cb[n], 0.0f);
                for (int n = ihi * g.Wo + lane; n < g.N; n += 32) ob[n] = __fadd_rn(cb[n], 0.0f);
            }
            const int4* rows = s_row + ilo;
            const int nrows = ihi - ilo;
            // Loop order: a batch of kFwdRB output rows, then the 32-column chunks across it.  The batch's source
            // rows are gathered again by every chunk within a few hundred cycles, i.e. out of L1, instead of
            // once per full sweep over the image (L2 latency on every gather when the warps' sweeps exceed L1).
            for (int i0 = 0; i0 < nrows; i0 += kFwdRB) {
                const int nb = nrows - i0;
                float* obat = ob + (long long)(ilo + i0) * g.Wo;
                const float* cbat = COMPOSITE ? cb + (long long)(ilo + i0) * g.Wo : nullptr;
                for (int j0 = 0; j0 < g.Wo; j0 += 32) {
                    const int j = j0 + lane;
                    if (j >= g.Wo) continue;
                    const int4 cx = s_col[j];  // {x0*4, x1*4, ax, bx}
                    const float xa = __int_as_float(cx.z), xb = __int_as_float(cx.w);
                    const char* Ux0 = opaque(reinterpret_cast<const char*>(Ub) + cx.x);
                    const char* Ux1 = opaque(reinterpret_cast<const char*>(Ub) + cx.y);
                    float* orow = opaque(obat + j);
                    const float* crow = COMPOSITE ? opaque(cbat + j) : nullptr;
                    // all 4*kFwdRB gathers are issued before the first dependent multiply / store, so one warp
                    // keeps 32 loads in flight; the tail batch is predicated rather than serialised.
                    float I[kFwdRB][4], cin[kFwdRB];
#pragma unroll
                    for (int r = 0; r < kFwdRB; ++r) {
                        // tail rows re-load the batch's last valid row (always a legal address) instead of
                        // predicating the loads; only their stores are skipped
                        const int rr = min(r, nb - 1);
                        const int4 cy = rows[i0 + rr];  // {y0*Ws*4, y1*Ws*4, ay, by}: byte offsets of the source rows
                        I[r][0] = ldg_f32(Ux0 + (unsigned)cy.x);
                        I[r][1] = ldg_f32(Ux0 + (unsigned)cy.y);
                        I[r][2] = ldg_f32(Ux1 + (unsigned)cy.x);
                        I[r][3] = ldg_f32(Ux1 + (unsigned)cy.y);
                        if (COMPOSITE) cin[r] = crow[rr * g.Wo];
                    }
#pragma unroll
                    for (int r = 0; r < kFwdRB; ++r) {
                        if (r < nb) {
                            const int4 cy = rows[i0 + r];
                            const float ay = __int_as_float(cy.z), by = __int_as_float(cy.w);
                            // transformer.py:112-116
                            float v = __fadd_rn(__fmul_rn(__fmul_rn(xa, ay), I[r][0]), __fmul_rn(__fmul_rn(xa, by), I[r][1]));
                            v = __fadd_rn(v, __fmul_rn(__fmul_rn(xb, ay), I[r][2]));
                            v = __fadd_rn(v, __fmul_rn(__fmul_rn(xb, by), I[r][3]));
                            if (COMPOSITE) v = __fadd_rn(cin[r], __fmul_rn(z, v));  // :724-726
                            orow[r * g.Wo] = v;
                        }
                    }
                }
            }
            continue;
        }
        // ---- general affine theta and/or several channels: per-pixel evaluation (cold, out of line) ------
        fwd_general_image<COMPOSITE>(Ub, ob, cb, th.t[0], th.t[1], th.t[2], th.t[3], th.t[4], th.t[5], z, inplace, lane, g.Hs,
                                     g.Ws, g.C, g.Ho, g.Wo, g.step_w, g.step_h, g.wsc, g.hsc);
    }
    if (bulk) bulk_zero_drain(lane);
}

// ---------------------------------------------------------------------------------------------------
// backward (also the fused write+composite backward)
// ---------------------------------------------------------------------------------------------------
// per-warp shared memory layout (in 4-byte words): row table 4*Ho | col table 4*Wo | run table Ws |
// ga [kBwdRB][Wo+1] | gb [kBwdRB][Wo+1]   (column Wo of every ga/gb row is a zero slot)
// (rounded up to a multiple of 4 words so every warp's int4 tables stay 16-byte aligned)
__host__ __device__ inline int bwd_warp_smem_words(const Geo& g) {
    return (4 * g.Ho + 4 * g.Wo + g.Ws + 2 * kBwdRB * (g.Wo + 1) + 3) & ~3;
}

struct InRange {
    int ilo, ihi, jlo, jhi;   // in-range output rows [ilo, ihi] and columns [jlo, jhi] (hi < lo: none)
};

// Axis tables of both backward kernels for a separable theta, one entry per output row / column: row {y0*ws4, y_t, ay, by}
// with ws4 = Ws*4 (source rows as byte offsets), column {x0, x_t, ax, bx} with x0 in bytes (x0*4) when COL_BYTES.
// STREAM_ORDER stores the rows in the order that makes y0 non-decreasing (reversed when t4 < 0).  Also clears the run table
// s_run[Ws].  Returns the in-range rows and columns, the same on every lane: only those contribute (out-of-range taps
// cancel), and each is one interval because every rounding step of the coordinate map is monotone.  Ends with a __syncwarp.
template <bool COL_BYTES, bool STREAM_ORDER>
__device__ __forceinline__ InRange build_bwd_tables(const Theta& th, const Geo& g, int4* s_row, int4* s_col, int* s_run, int ws4,
                                                    int lane) {
    int ilo = g.Ho, ihi = -1, jlo = g.Wo, jhi = -1;
    const bool ascending = !(th.t[4] < 0.0f);
    for (int i = lane; i < g.Ho; i += 32) {
        const float yt = lin_at(i, g.step_h);
        const Axis Y = axis_tap(affine_row(th.t[3], th.t[4], th.t[5], 0.0f, yt), g.hsc, g.Hs);
        s_row[!STREAM_ORDER || ascending ? i : g.Ho - 1 - i] =
            make_int4(Y.c0 * ws4, __float_as_int(yt), __float_as_int(Y.a), __float_as_int(Y.b));
        if (Y.c0 != Y.c1) { ilo = min(ilo, i); ihi = max(ihi, i); }
    }
    for (int j = lane; j < g.Wo; j += 32) {
        const float xt = lin_at(j, g.step_w);
        const Axis X = axis_tap(affine_row(th.t[0], th.t[1], th.t[2], xt, 0.0f), g.wsc, g.Ws);
        s_col[j] = make_int4(COL_BYTES ? X.c0 * 4 : X.c0, __float_as_int(xt), __float_as_int(X.a), __float_as_int(X.b));
        if (X.c0 != X.c1) { jlo = min(jlo, j); jhi = max(jhi, j); }
    }
    for (int x = lane; x < g.Ws; x += 32) s_run[x] = 0;
    ilo = __reduce_min_sync(0xffffffffu, ilo); ihi = __reduce_max_sync(0xffffffffu, ihi);
    jlo = __reduce_min_sync(0xffffffffu, jlo); jhi = __reduce_max_sync(0xffffffffu, jhi);
    __syncwarp();
    return {ilo, ihi, jlo, jhi};
}

// Column runs over the in-range columns [jlo, jhi] of a table built by build_bwd_tables<COL_BYTES, ...>: source column x
// receives output columns [start, end) = {j : x0[j] == x}, packed s_run[x] = start | end << 16 (empty stays 0).  Returns
// the longest run, the same on every lane.
template <bool COL_BYTES>
__device__ __forceinline__ int build_col_runs(const int4* s_col, int* s_run, int jlo, int jhi, int lane) {
    int rmax = 0;
    for (int j = jlo + lane; j <= jhi; j += 32) {
        const int x0 = s_col[j].x;
        if (j == jlo || s_col[j - 1].x != x0) {
            int e = j + 1;
            while (e <= jhi && s_col[e].x == x0) ++e;
            s_run[COL_BYTES ? x0 >> 2 : x0] = j | (e << 16);
            rmax = max(rmax, e - j);
        }
    }
    return __reduce_max_sync(0xffffffffu, rmax);
}

// store (first transform: the image was zero-filled up front) or accumulate (later transforms of the same
// source image) one dU element
__device__ __forceinline__ void emit_px(char* p, float v, bool ok, bool first) {
    if (ok) {
        float* q = reinterpret_cast<float*>(p);
        *q = first ? v : (*q + v);
    }
}


// General affine theta and/or several channels: L2 atomics (red.global.add.f32) on the image's own dU lines, which the
// caller has zero-filled; dtheta/dz by warp shuffles.  Out of line (cold path).
// Warp-aggregated atomics were built and measured for this path in round 2 (neighbour hand-over of the right taps by one
// shuffle + shuffle sums over runs of equal addresses, one reduction per run) and lost on B200 in both regimes:
// rotated 256 -> 64 read (about one source pixel per output pixel) 439 us plain vs 554 us aggregated; rotated 64 -> 256
// write at full-cover scale (3.6 output pixels per source pixel, the case aggregation is for) 7.2 ms plain vs 17.7 ms
// aggregated (4096 images; bench.py aux_kernels.general_affine, profiles/r02_general_affine.md).  The L2 reduction units
// absorb the duplicates faster than the warp can find them, so the plain per-lane form stays.
template <bool COMPOSITE>
__device__ __noinline__ void bwd_general_image(const float* __restrict__ Ub, float* __restrict__ dUb,
                                               const float* __restrict__ gb, float* __restrict__ dtheta_b,
                                               float* __restrict__ dz_b, float t0, float t1, float t2, float t3, float t4,
                                               float t5, float z, int lane, int Hs, int Ws, int C, int Ho, int Wo,
                                               float step_w, float step_h, float wsc, float hsc) {
    Theta th;
    th.t[0] = t0; th.t[1] = t1; th.t[2] = t2; th.t[3] = t3; th.t[4] = t4; th.t[5] = t5;
    Geo g;
    g.Hs = Hs; g.Ws = Ws; g.C = C; g.Ho = Ho; g.Wo = Wo; g.N = Ho * Wo; g.S = Hs * Ws;
    g.step_w = step_w; g.step_h = step_h; g.wsc = wsc; g.hsc = hsc; g.magic_wo = 0;
    float p[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int j0 = 0; j0 < g.Wo; j0 += 32) {
        const int j = j0 + lane;
        if (j >= g.Wo) continue;
        const float xt = lin_at(j, g.step_w);
        for (int i = 0; i < g.Ho; ++i) {
            Axis X, Y;
            taps_general(th, g, i, j, X, Y);
            // Out of range on an axis: the two taps alias one pixel with weights +w/-w, so every
            // gradient contribution cancels in exact arithmetic (DESIGN.md "borders").
            if (X.c0 == X.c1 || Y.c0 == Y.c1) continue;
            const int r0 = Y.c0 * g.Ws, r1 = Y.c1 * g.Ws;
            const int ia = (r0 + X.c0) * C, ib = (r1 + X.c0) * C, ic = (r0 + X.c1) * C, id = (r1 + X.c1) * C;
            const float wa = X.a * Y.a, wb = X.a * Y.b, wc = X.b * Y.a, wd = X.b * Y.b;
            float sx = 0.f, sy = 0.f;
            const long long n = (long long)i * g.Wo + j;
            for (int c = 0; c < C; ++c) {
                const float gc = __ldg(gb + n * C + c);
                const float gv = COMPOSITE ? gc * z : gc;
                const float Ia = __ldg(Ub + ia + c), Ib = __ldg(Ub + ib + c);
                const float Ic = __ldg(Ub + ic + c), Id = __ldg(Ub + id + c);
                if (dUb) {
                    atomicAdd(dUb + ia + c, wa * gv);
                    atomicAdd(dUb + ib + c, wb * gv);
                    atomicAdd(dUb + ic + c, wc * gv);
                    atomicAdd(dUb + id + c, wd * gv);
                }
                sx += gv * (Y.a * (Ic - Ia) + Y.b * (Id - Ib));
                sy += gv * (X.a * (Ib - Ia) + X.b * (Id - Ic));
                if (COMPOSITE) p[6] += gc * (wa * Ia + wb * Ib + wc * Ic + wd * Id);
            }
            const float yt = lin_at(i, g.step_h);
            p[0] += sx * xt; p[1] += sx * yt; p[2] += sx;
            p[3] += sy * xt; p[4] += sy * yt; p[5] += sy;
        }
    }
    __syncwarp();
    const float half_wsc = g.wsc * 0.5f, half_hsc = g.hsc * 0.5f;
    p[0] *= half_wsc; p[1] *= half_wsc; p[2] *= half_wsc;
    p[3] *= half_hsc; p[4] *= half_hsc; p[5] *= half_hsc;
#pragma unroll
    for (int k = 0; k < 7; ++k) p[k] = warp_sum(p[k]);
    if (lane == 0) {
        if (dtheta_b) {
#pragma unroll
            for (int k = 0; k < 6; ++k) dtheta_b[k] = p[k];
        }
        if (COMPOSITE && dz_b) *dz_b = p[6];
    }
}

template <bool COMPOSITE, int NXC, int SXY>
__global__ void __launch_bounds__(kWarpThreads, kBwdMinBlocks) stn_bwd_warp_kernel(const BwdArgs a, const SxyArgs sx) {
    extern __shared__ int4 s_dyn[];
    const Geo& g = a.g;
    const int C = g.C;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int* s_base = reinterpret_cast<int*>(s_dyn) + warp * bwd_warp_smem_words(g);
    int4* s_row = reinterpret_cast<int4*>(s_base);
    int4* s_col = s_row + g.Ho;
    int* s_run = reinterpret_cast<int*>(s_col + g.Wo);
    float* s_ga = reinterpret_cast<float*>(s_run + g.Ws);
    float* s_gb = s_ga + kBwdRB * (g.Wo + 1);
    if (lane < kBwdRB) {  // zero slots read by empty run positions
        s_ga[lane * (g.Wo + 1) + g.Wo] = 0.0f;
        s_gb[lane * (g.Wo + 1) + g.Wo] = 0.0f;
    }
    __syncwarp();
    const long long nwarps = (long long)gridDim.x * kWarpsPerCta;
    const int SC = g.S * C;
    const float half_wsc = g.wsc * 0.5f, half_hsc = g.hsc * 0.5f;
    const bool bulk = a.dU && a.coop_zero == 2;
    unsigned zero_smem = 0;
    if (bulk) {  // zeroed block behind the per-warp tables
        int* zb = reinterpret_cast<int*>(s_dyn) + kWarpsPerCta * bwd_warp_smem_words(g);
        bulk_zero_init(zb);
        zero_smem = (unsigned)__cvta_generic_to_shared(zb);
    }

    // One group of kWarpsPerCta consecutive source images per CTA iteration: the group's dU region is contiguous
    // and is zero-filled by the whole CTA in one linear sweep; after the barrier every warp works on its own
    // image (footprint rows overwrite the zeros while the lines are still in L2).
    for (long long g0 = (long long)blockIdx.x * kWarpsPerCta; g0 < a.Bsrc; g0 += nwarps) {
        if (a.dU && a.coop_zero == 1) {
            const long long ng = min((long long)kWarpsPerCta, a.Bsrc - g0);
            __syncthreads();  // (uniform trip count: every warp of the CTA runs this loop the same number of times)
            fill_zero_cta(a.dU + g0 * (long long)SC, ng * (long long)SC);
            __syncthreads();
        }
        const long long bs = g0 + warp;
        if (bs >= a.Bsrc) continue;
        const float* __restrict__ Ub = a.U + bs * (long long)SC;
        float* __restrict__ dUb = a.dU ? a.dU + bs * (long long)SC : nullptr;
        if (dUb && a.coop_zero == 0) {   // small sources: the warp zero-fills its own image (no CTA barrier)
            fill_zero(dUb, 0, SC, lane);
            __syncwarp();
        }

        for (int t = 0; t < a.u_div; ++t) {
            const long long b = bs * a.u_div + t;
            Theta th;
            load_theta<SXY>(th, a.theta, sx, b);
            const bool sep = th.separable() && C == 1;
            float z = 1.0f;
            bool active = true;
            if (COMPOSITE) {
                z = __ldg(a.z_pres + b);
                active = a.stop_sum ? (__ldg(a.stop_sum + b) < a.threshold) : true;
            }
            const float* __restrict__ gb = a.gout + b * (long long)g.N * C;
            float p[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // dtheta (6) + dz

            if (!active) {
                // (dU of an inactive image stays zero)
                if (bulk) fill_zero_bulk(dUb, 0, SC, lane, zero_smem);
            } else if (!sep) {
                // ---------- general affine / multi-channel: cold, out of line (writes dtheta/dz itself) ----
                if (bulk) {
                    fill_zero(dUb, 0, SC, lane);
                    __syncwarp();
                }
                bwd_general_image<COMPOSITE>(Ub, dUb, gb, a.dtheta ? a.dtheta + 6 * b : nullptr,
                                             (COMPOSITE && a.dz) ? a.dz + b : nullptr, th.t[0], th.t[1], th.t[2], th.t[3],
                                             th.t[4], th.t[5], z, lane, g.Hs, g.Ws, g.C, g.Ho, g.Wo, g.step_w,
                                             g.step_h, g.wsc, g.hsc);
                continue;
            } else {
                // ---------- separable: gather form, streaming over rows ----------------------------------
                // In range, x1 = x0+1 and y1 = y0+1: table entries are {byte offset of c0, lin, a, b} and the four
                // taps sit at base, base+4, base+Ws*4, base+Ws*4+4.
                __syncwarp();
                const bool need_dU = dUb != nullptr;
                const bool first_transform = (t == 0);  // the group zero-fill made dU final outside the footprint
                const int ws4 = g.Ws * 4;
                const auto [ilo, ihi, jlo, jhi] = build_bwd_tables<true, false>(th, g, s_row, s_col, s_run, ws4, lane);
                if (bulk) {
                    // rows of dU outside the footprint band go to the copy engine; the band itself (which the
                    // stream below overwrites) is zeroed with ordinary stores, ordered before them by the warp
                    if (ihi >= ilo && jhi >= jlo) {
                        const int ya = s_row[ilo].x, yb = s_row[ihi].x;
                        const int ylo = min(ya, yb) / ws4, yend = max(ya, yb) / ws4 + 2;  // band rows [ylo, yend)
                        fill_zero_bulk(dUb, 0, ylo * g.Ws, lane, zero_smem);
                        fill_zero_bulk(dUb, yend * g.Ws, SC, lane, zero_smem);
                        // (the band itself is zeroed just ahead of the stream, a few rows at a time: see band_off below)
                    } else {
                        fill_zero_bulk(dUb, 0, SC, lane, zero_smem);
                    }
                    __syncwarp();
                }
                if (ihi >= ilo && jhi >= jlo) {
                    const int rmax = build_col_runs<true>(s_col, s_run, jlo, jhi, lane);
                    const int xa = s_col[jlo].x >> 2, xb = s_col[jhi].x >> 2;
                    const int fw = max(xa, xb) + 2 - min(xa, xb);   // footprint columns [xlo, xhi + 1]
                    const int njc = (jhi - jlo + 32) >> 5;
                    __syncwarp();
                    // Source columns are handled in strips of NXC*32 (register budget): a footprint wider than
                    // one strip streams the rows once per strip; dtheta/dz are accumulated in the first pass only.
                    const int xlo_all = min(xa, xb), nxc_all = (fw + 31) >> 5;
                    for (int cg = 0; cg < nxc_all && (cg == 0 || need_dU); cg += NXC) {
                    const int xlo = xlo_all + cg * 32;
                    const int nxc = min(NXC, nxc_all - cg);
                    const bool first_pass = cg == 0;
                    int runA[NXC], runB[NXC];
#pragma unroll
                    for (int c = 0; c < NXC; ++c) {
                        const int x = xlo + c * 32 + lane;
                        runA[c] = (c < nxc && x < g.Ws) ? s_run[x] : 0;
                        runB[c] = (c < nxc && x - 1 < g.Ws && x > 0) ? s_run[x - 1] : 0;
                    }
                    float acc0[NXC], acc1[NXC];
#pragma unroll
                    for (int c = 0; c < NXC; ++c) { acc0[c] = 0.f; acc1[c] = 0.f; }
                    int offcur = -1;  // byte offset of the source row held in acc0 (acc1: next row); -1 = none
                    const bool ascending = !(th.t[4] < 0.0f);
                    const int nrows = ihi - ilo + 1;
                    // Large sources (bulk mode): the band rows are zeroed by ordinary stores just before the stream overwrites
                    // them, the rows of one batch at a time (first strip pass; whole rows, one contiguous fill), so that the
                    // zero and the value of a line meet in L2.  Zeroing the whole band up front cost a second DRAM write of
                    // part of it (ncu, 256 <- 64: 5.37 GB of traffic for 4.79 GB of algorithmic bytes).  Zeroing only a strip's
                    // own columns per pass was measured too: the per-row fills cost more instructions than the traffic saves.
                    int band_off = ascending ? s_row[ilo].x : s_row[ihi].x;   // byte offset of the first band row not yet zeroed
                    const char* Ubc = opaque(reinterpret_cast<const char*>(Ub));
                    char* dUbc = reinterpret_cast<char*>(dUb) + (xlo + lane) * 4;
                    const int P = g.Wo + 1;  // pitch of the per-row ga/gb buffers; column Wo is a zero slot

                    for (int ii0 = 0; ii0 < nrows; ii0 += kBwdRB) {
                        const int nb = min(kBwdRB, nrows - ii0);
                        if (bulk && first_pass) {   // zero the source rows this batch reaches (ordered before phase 2 by the __syncwarp below)
                            const int ilast = ascending ? ilo + ii0 + nb - 1 : ihi - ii0 - nb + 1;
                            const int upto = s_row[ilast].x + 2 * ws4;
                            fill_zero(dUb, band_off >> 2, upto >> 2, lane);
                            band_off = max(band_off, upto);
                        }
                        // ---- phase 1 (output-column side): loads of kBwdRB rows in flight together ----
                        for (int jc = 0; jc < njc; ++jc) {
                            const int j = jlo + jc * 32 + lane;
                            if (j > jhi) continue;
                            const int4 cj = s_col[j];
                            const float xt = __int_as_float(cj.y), ax = __int_as_float(cj.z), bx = __int_as_float(cj.w);
                            int4 cy[kBwdRB];
                            float gq[kBwdRB], I[kBwdRB][4];
#pragma unroll
                            for (int r = 0; r < kBwdRB; ++r) {
                                {
                                    const int rr = min(r, nb - 1);  // tail rows re-load the last valid row
                                    const int i = ascending ? ilo + ii0 + rr : ihi - ii0 - rr;
                                    cy[r] = s_row[i];
                                    gq[r] = __ldg(gb + i * g.Wo + j);
                                    if (first_pass) {  // the taps only feed dtheta / dz
                                        const char* pa = Ubc + (unsigned)(cy[r].x + cj.x);
                                        const char* pb = pa + ws4;
                                        I[r][0] = ldg_f32(pa); I[r][2] = ldg_f32(pa + 4);
                                        I[r][1] = ldg_f32(pb); I[r][3] = ldg_f32(pb + 4);
                                    } else {
                                        I[r][0] = I[r][1] = I[r][2] = I[r][3] = 0.f;
                                    }
                                }
                            }
#pragma unroll
                            for (int r = 0; r < kBwdRB; ++r) {
                                if (r < nb) {
                                    const float yt = __int_as_float(cy[r].y), ay = __int_as_float(cy[r].z), by = __int_as_float(cy[r].w);
                                    const float gv = COMPOSITE ? gq[r] * z : gq[r];
                                    const float sx = gv * (ay * (I[r][2] - I[r][0]) + by * (I[r][3] - I[r][1]));
                                    const float sy = gv * (ax * (I[r][1] - I[r][0]) + bx * (I[r][3] - I[r][2]));
                                    p[0] += sx * xt; p[1] += sx * yt; p[2] += sx;
                                    p[3] += sy * xt; p[4] += sy * yt; p[5] += sy;
                                    if (COMPOSITE)
                                        p[6] += gq[r] * ((ax * ay) * I[r][0] + (ax * by) * I[r][1] + (bx * ay) * I[r][2] + (bx * by) * I[r][3]);
                                    if (need_dU) { s_ga[r * P + j] = ax * gv; s_gb[r * P + j] = bx * gv; }
                                }
                            }
                        }
                        if (!need_dU) continue;
                        __syncwarp();
                        // ---- phase 2 (source-column side): T[x] = sum_{j in run(x)} ax g + sum_{j in run(x-1)} bx g
                        //      uniform trip count rmax (longest run of this image); empty slots read a zero.
                        //      Each 32-column chunk then walks the batch's rows with its own copy of the
                        //      stream state: a source row is stored once, when the stream moves past it. ----
                        int off_end = offcur;
#pragma unroll
                        for (int c = 0; c < NXC; ++c) {
                            if (c < nxc) {
                                const int a0 = runA[c] & 0xffff, a1 = runA[c] >> 16;
                                const int b0 = runB[c] & 0xffff, b1 = runB[c] >> 16;
                                float T[kBwdRB];
#pragma unroll
                                for (int r = 0; r < kBwdRB; ++r) T[r] = 0.f;
                                for (int q = 0; q < rmax; ++q) {
                                    const int ia = (a0 + q < a1) ? a0 + q : g.Wo;
                                    const int ib = (b0 + q < b1) ? b0 + q : g.Wo;
#pragma unroll
                                    for (int r = 0; r < kBwdRB; ++r) T[r] += s_ga[r * P + ia] + s_gb[r * P + ib];
                                }
                                const bool xok = xlo + c * 32 + lane < g.Ws;
                                char* colp = dUbc + c * 128;
                                int oc = offcur;
                                float v0 = acc0[c], v1 = acc1[c];
#pragma unroll
                                for (int r = 0; r < kBwdRB; ++r) {
                                    if (r < nb) {
                                        const int i = ascending ? ilo + ii0 + r : ihi - ii0 - r;
                                        const int4 cy = s_row[i];
                                        const int off = cy.x;
                                        if (off != oc) {
                                            if (oc >= 0) {
                                                emit_px(colp + oc, v0, xok, first_transform);
                                                if (off == oc + ws4) {
                                                    v0 = v1; v1 = 0.f;
                                                } else {
                                                    emit_px(colp + oc + ws4, v1, xok, first_transform);
                                                    v0 = 0.f; v1 = 0.f;
                                                }
                                            }
                                            oc = off;
                                        }
                                        v0 += __int_as_float(cy.z) * T[r];
                                        v1 += __int_as_float(cy.w) * T[r];
                                    }
                                }
                                acc0[c] = v0; acc1[c] = v1;
                                off_end = oc;
                            }
                        }
                        offcur = off_end;
                        __syncwarp();
                    }
                    if (need_dU && offcur >= 0) {
#pragma unroll
                        for (int c = 0; c < NXC; ++c) {
                            if (c < nxc) {
                                const bool xok = xlo + c * 32 + lane < g.Ws;
                                emit_px(dUbc + c * 128 + offcur, acc0[c], xok, first_transform);
                                emit_px(dUbc + c * 128 + offcur + ws4, acc1[c], xok, first_transform);
                            }
                        }
                    }
                    __syncwarp();
                    }  // strips
                }
                // scale: dx_s = dx*(Ws-1.001)/2, dy_s = dy*(Hs-1.001)/2   (transformer.py:75-76)
                p[0] *= half_wsc; p[1] *= half_wsc; p[2] *= half_wsc;
                p[3] *= half_hsc; p[4] *= half_hsc; p[5] *= half_hsc;
            }
            store_image_grads<COMPOSITE, SXY>(a, sx, b, p, lane);
        }
    }
    if (bulk) bulk_zero_drain(lane);
}

}  // namespace mog
