// Backward of the sampler when the output is at least about as wide as the source (the write direction: a window of
// <= 64 columns onto a canvas), separable theta, C = 1: one warp per image, LANES ALONG SOURCE COLUMNS (sm_100a).
//
// The streaming kernel walks the OUTPUT columns (phase 1), parks ax*g and bx*g in shared memory and then walks the
// SOURCE columns (phase 2) to sum the runs; ncu (profiles/r02_*) charges that form 140 warp instructions per 32 in-range
// pixels and, in a CTA-per-image variant, 38 % of the stall samples at the two barriers per batch.  When every source
// column owns a short run of output columns (upsampling or ~1:1), the second walk is all there is to do:
//   * lane l owns source columns x = NCOL*l .. NCOL*l + NCOL-1 (NCOL = 1 for Ws <= 32, 2 for Ws <= 64) and, for each of them,
//     the run of output columns {j : x0[j] == x} = [a0, a1);
//   * a batch of kColRB in-range output rows: the lane reads g[i][j] over its runs straight from global memory (a warp's
//     runs are one contiguous span of the row), accumulates  A = sum ax*g,  Bs = sum bx*g  and the dtheta / dz partial sums
//     -- the four taps of pixel (i, j) are U[y0][x], U[y0][x+1], U[y0+1][x], U[y0+1][x+1]: per lane and source row, loaded
//     once per row batch, not per pixel;
//   * T[x] = A[x] + Bs[x-1] (own register, or one shuffle from the lane below) is folded into the two running source rows
//     (y0, y0 + 1); a source row is stored once, coalesced, when the stream moves past it.
// No shared-memory gather rows, no barriers, no atomics; shared memory holds only the axis tables (16 B per output row /
// column).  Results: same products as the streaming kernel, summed run-by-run instead of column-by-column (fp32 tolerance of
// the gradient contract, DESIGN.md section 4); deterministic.
#pragma once
#include "mog_stn_warp.cuh"

namespace mog {

constexpr int kColRB = 4;          // output rows per batch
constexpr int kColMinBlocks = 10;  // __launch_bounds__: 96 registers, 20 warps per SM (measured against 6 / 7 / 8 / 12,
                                   // profiles/r02_kernel_experiments.md)
constexpr int kColMaxWs = 64;      // source columns: NCOL <= 2 per lane

__host__ __device__ inline int align128(int v) { return (v + 127) & ~127; }

struct ColLayout {
    int row, col, run, total;   // byte offsets within one warp's slice
};
__host__ __device__ inline ColLayout bwd_col_layout(const Geo& g) {
    ColLayout l;
    int o = 0;
    l.row = o; o += g.Ho * 16;
    l.col = o; o += g.Wo * 16;
    l.run = o; o += align128(g.Ws * 4);
    l.total = align128(o);
    return l;
}

template <bool COMPOSITE, int NCOL, int SXY>
__global__ void __launch_bounds__(kWarpThreads, kColMinBlocks) stn_bwd_col_kernel(const BwdArgs a, const SxyArgs sx) {
    extern __shared__ __align__(128) unsigned char s_raw[];
    const Geo& g = a.g;
    const ColLayout L = bwd_col_layout(g);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char* s_mine = s_raw + (size_t)warp * L.total;
    int4* s_row = reinterpret_cast<int4*>(s_mine + L.row);   // stream order: {y0 * Ws * 4, y_t, ay, by}
    int4* s_col = reinterpret_cast<int4*>(s_mine + L.col);   // {x0, x_t, ax, bx} per output column
    int* s_run = reinterpret_cast<int*>(s_mine + L.run);     // per source column: start | end << 16 of its run (0 = empty)
    const int ws4 = g.Ws * 4;
    const int SC = g.S;
    const float half_wsc = g.wsc * 0.5f, half_hsc = g.hsc * 0.5f;
    const long long nwarps = (long long)gridDim.x * kWarpsPerCta;
    const int x = NCOL * lane;   // first source column of this lane

    for (long long b = (long long)blockIdx.x * kWarpsPerCta + warp; b < a.Bsrc; b += nwarps) {
        const float* __restrict__ Ub = a.U + b * (long long)SC;
        float* __restrict__ dUb = a.dU ? a.dU + b * (long long)SC : nullptr;
        const float* __restrict__ gb = a.gout + b * (long long)g.N;
        Theta th;
        load_theta<SXY>(th, a.theta, sx, b);
        float z = 1.0f;
        bool active = true;
        if (COMPOSITE) {
            z = __ldg(a.z_pres + b);
            active = a.stop_sum ? (__ldg(a.stop_sum + b) < a.threshold) : true;
        }
        if (dUb) fill_zero(dUb, 0, SC, lane);   // the rows the stream reaches overwrite it (ordered by the __syncwarp below)
        float p[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        __syncwarp();   // also: the previous image's table reads are done
        if (active && !th.separable()) {   // general affine theta: cold path
            bwd_general_image<COMPOSITE>(Ub, dUb, gb, a.dtheta ? a.dtheta + 6 * b : nullptr, (COMPOSITE && a.dz) ? a.dz + b : nullptr,
                                         th.t[0], th.t[1], th.t[2], th.t[3], th.t[4], th.t[5], z, lane, g.Hs, g.Ws, 1, g.Ho,
                                         g.Wo, g.step_w, g.step_h, g.wsc, g.hsc);
            continue;
        }
        if (active) {
            const auto [ilo, ihi, jlo, jhi] = build_bwd_tables<false, true>(th, g, s_row, s_col, s_run, ws4, lane);
            const bool ascending = !(th.t[4] < 0.0f);   // the stream order of s_row
            if (ihi >= ilo && jhi >= jlo) {
                const int rmax = build_col_runs<false>(s_col, s_run, jlo, jhi, lane);
                __syncwarp();
                const bool need_dU = dUb != nullptr;
                int a0[NCOL], a1[NCOL];
#pragma unroll
                for (int c = 0; c < NCOL; ++c) {
                    const int r = (x + c < g.Ws) ? s_run[x + c] : 0;
                    a0[c] = r & 0xffff; a1[c] = r >> 16;
                }
                const int nrows = ihi - ilo + 1;
                const int4* rows = s_row + (ascending ? ilo : g.Ho - 1 - ihi);   // rows[ii] = stream row ii
                const int gfirst = (ascending ? ilo : ihi) * g.Wo;   // element offsets within the image's gradient (N < 2^31)
                const int gstep = ascending ? g.Wo : -g.Wo;
                const float* Ubx = Ub + x;
                char* colp = reinterpret_cast<char*>(dUb) + x * 4;
                bool tap_ok[NCOL + 1], col_ok[NCOL];
#pragma unroll
                for (int k = 0; k <= NCOL; ++k) tap_ok[k] = x + k < g.Ws;
#pragma unroll
                for (int c = 0; c < NCOL; ++c) col_ok[c] = x + c < g.Ws;
                const bool pair_store = NCOL == 2 && (g.Ws & 1) == 0 && (reinterpret_cast<uintptr_t>(dUb) & 7) == 0;
                float v0[NCOL], v1[NCOL];
#pragma unroll
                for (int c = 0; c < NCOL; ++c) { v0[c] = 0.f; v1[c] = 0.f; }
                int oc = -1;   // byte offset of the source row held in v0 (v1: the next row); -1 = none

                auto emit_row = [&](int off, const float (&v)[NCOL]) {
                    if (NCOL == 2 && pair_store) {
                        if (col_ok[0]) *reinterpret_cast<float2*>(colp + off) = make_float2(v[0], v[NCOL - 1]);
                    } else {
#pragma unroll
                        for (int c = 0; c < NCOL; ++c)
                            if (col_ok[c]) *reinterpret_cast<float*>(colp + off + 4 * c) = v[c];
                    }
                };

                for (int ii0 = 0; ii0 < nrows; ii0 += kColRB) {
                    const int nb = min(kColRB, nrows - ii0);
                    int4 cy[kColRB];
#pragma unroll
                    for (int r = 0; r < kColRB; ++r) cy[r] = rows[ii0 + (r < nb ? r : nb - 1)];
                    // per (row, column): what the pixel needs of the four taps
                    float DX[kColRB][NCOL], E1[kColRB][NCOL], E2[kColRB][NCOL], VA[kColRB][NCOL], VC[kColRB][NCOL];
                    {
                        float Ia[kColRB][NCOL + 1], Ib[kColRB][NCOL + 1];
#pragma unroll
                        for (int r = 0; r < kColRB; ++r) {
#pragma unroll
                            for (int k = 0; k <= NCOL; ++k) {
                                Ia[r][k] = tap_ok[k] ? __ldg(Ubx + ((cy[r].x >> 2) + k)) : 0.f;
                                Ib[r][k] = tap_ok[k] ? __ldg(Ubx + ((cy[r].x >> 2) + g.Ws + k)) : 0.f;
                            }
                        }
#pragma unroll
                        for (int r = 0; r < kColRB; ++r) {
                            const float ay = __int_as_float(cy[r].z), by = __int_as_float(cy[r].w);
#pragma unroll
                            for (int c = 0; c < NCOL; ++c) {
                                DX[r][c] = ay * (Ia[r][c + 1] - Ia[r][c]) + by * (Ib[r][c + 1] - Ib[r][c]);
                                E1[r][c] = Ib[r][c] - Ia[r][c];
                                E2[r][c] = Ib[r][c + 1] - Ia[r][c + 1];
                                if (COMPOSITE) {
                                    VA[r][c] = ay * Ia[r][c] + by * Ib[r][c];
                                    VC[r][c] = ay * Ia[r][c + 1] + by * Ib[r][c + 1];
                                }
                            }
                        }
                    }
                    float A[kColRB][NCOL], Bs[kColRB][NCOL];
#pragma unroll
                    for (int r = 0; r < kColRB; ++r) {
#pragma unroll
                        for (int c = 0; c < NCOL; ++c) { A[r][c] = 0.f; Bs[r][c] = 0.f; }
                    }
                    int grow[kColRB];   // offset of the batch's rows (rows past the end: the last valid one, masked below)
#pragma unroll
                    for (int r = 0; r < kColRB; ++r) grow[r] = gfirst + (ii0 + (r < nb ? r : nb - 1)) * gstep;
                    for (int q = 0; q < rmax; ++q) {
                        float gq[kColRB][NCOL];
                        int4 cj[NCOL];
                        bool valid[NCOL];
#pragma unroll
                        for (int c = 0; c < NCOL; ++c) {
                            const int j = a0[c] + q;
                            valid[c] = j < a1[c];
                            const int jj = valid[c] ? j : jlo;
                            cj[c] = s_col[jj];
#pragma unroll
                            for (int r = 0; r < kColRB; ++r) {   // (always a valid address: the mask is applied to the value)
                                const float gl = __ldg(gb + (grow[r] + jj));
                                gq[r][c] = (valid[c] && r < nb) ? gl : 0.f;
                            }
                        }
#pragma unroll
                        for (int c = 0; c < NCOL; ++c) {
                            const float xt = __int_as_float(cj[c].y);
                            const float ax = valid[c] ? __int_as_float(cj[c].z) : 0.f;
                            const float bx = valid[c] ? __int_as_float(cj[c].w) : 0.f;
                            float SX = 0.f, SY = 0.f;
#pragma unroll
                            for (int r = 0; r < kColRB; ++r) {
                                const float yt = __int_as_float(cy[r].y);
                                const float gv = COMPOSITE ? gq[r][c] * z : gq[r][c];
                                A[r][c] += ax * gv;
                                Bs[r][c] += bx * gv;
                                const float sx = gv * DX[r][c];
                                const float sy = gv * (ax * E1[r][c] + bx * E2[r][c]);
                                SX += sx; SY += sy;
                                p[1] += sx * yt; p[4] += sy * yt;
                                if (COMPOSITE) p[6] += gq[r][c] * (ax * VA[r][c] + bx * VC[r][c]);
                            }
                            p[0] += SX * xt; p[2] += SX; p[3] += SY * xt; p[5] += SY;
                        }
                    }
                    if (!need_dU) continue;
                    // ---- fold T[x] = A[x] + Bs[x - 1] into the two running source rows ----
#pragma unroll
                    for (int r = 0; r < kColRB; ++r) {
                        const float below = __shfl_up_sync(0xffffffffu, Bs[r][NCOL - 1], 1);   // Bs of column x - 1 (lane 0: none)
                        if (r < nb) {
                            float T[NCOL];
                            T[0] = A[r][0] + (lane > 0 ? below : 0.f);
#pragma unroll
                            for (int c = 1; c < NCOL; ++c) T[c] = A[r][c] + Bs[r][c - 1];
                            const int off = cy[r].x;
                            if (off != oc) {
                                if (oc >= 0) {
                                    emit_row(oc, v0);
                                    if (off == oc + ws4) {
#pragma unroll
                                        for (int c = 0; c < NCOL; ++c) { v0[c] = v1[c]; v1[c] = 0.f; }
                                    } else {
                                        emit_row(oc + ws4, v1);
#pragma unroll
                                        for (int c = 0; c < NCOL; ++c) { v0[c] = 0.f; v1[c] = 0.f; }
                                    }
                                }
                                oc = off;
                            }
                            const float ay = __int_as_float(cy[r].z), by = __int_as_float(cy[r].w);
#pragma unroll
                            for (int c = 0; c < NCOL; ++c) { v0[c] += ay * T[c]; v1[c] += by * T[c]; }
                        }
                    }
                }
                if (need_dU && oc >= 0) {
                    emit_row(oc, v0);
                    emit_row(oc + ws4, v1);
                }
                // scale: dx_s = dx*(Ws-1.001)/2, dy_s = dy*(Hs-1.001)/2   (transformer.py:75-76)
                p[0] *= half_wsc; p[1] *= half_wsc; p[2] *= half_wsc;
                p[3] *= half_hsc; p[4] *= half_hsc; p[5] *= half_hsc;
            }
        }
        store_image_grads<COMPOSITE, SXY>(a, sx, b, p, lane);
    }
}

}  // namespace mog
