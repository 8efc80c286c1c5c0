// libmogstn -- fused ASR regularisers (one thread per image).
//
// Replaces ~60 tiny TF ops of /root/reference/air/air_number_bbox_location.py:645-681 (entropy),
// :970-1015 (marginal / min-element count penalties), :1016-1027 (size window), :1029-1069
// (out-of-canvas, pairwise size, pairwise overlap) with one forward and one backward kernel over
// [B,T] inputs (T <= 16).  Latency-bound work (<= 116 B per image): no roofline claim.
// Sub-gradient tie rules follow TF (oracle/asr_ref.py): max(v,0) passes gradient when v >= 0,
// max(a,b) routes to a when a >= b, abs'(0) = 0, reduce_min splits equally among ties.
#include "mog_common.cuh"

namespace mog {

constexpr int kAsrThreads = 128;
constexpr int MAXT = MOG_ASR_MAX_STEPS;
constexpr int MAXK = MOG_ASR_MAX_COUNTS;

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float softplusf_(float x) { return fmaxf(x, 0.0f) + log1pf(expf(-fabsf(x))); }
// tf.nn.sigmoid_cross_entropy_with_logits(labels=z, logits=x)
__device__ __forceinline__ float bce_logits(float z, float x) { return fmaxf(x, 0.0f) - x * z + log1pf(expf(-fabsf(x))); }
__device__ __forceinline__ float logit_eps(float p) { return logf(p + 1e-8f) - logf(1.0f - p + 1e-8f); }
__device__ __forceinline__ float dlogit_eps(float p) { return 1.0f / (p + 1e-8f) + 1.0f / (1.0f - p + 1e-8f); }
__device__ __forceinline__ float sgn(float v) { return (v > 0.0f) ? 1.0f : ((v < 0.0f) ? -1.0f : 0.0f); }

// STEPS: also count the active images of every step into psum[T + t] (active is [T][B] bytes); the parameter comes last
// so that the plain instantiation keeps its parameter offsets.
template <bool STEPS>
__global__ void __launch_bounds__(256) asr_colsum_kernel(const float* __restrict__ log_odds, float* psum, long long B,
                                                          int T, const unsigned char* __restrict__ active) {
    float acc[MAXT], cnt[STEPS ? MAXT : 1];
#pragma unroll
    for (int t = 0; t < MAXT; ++t) acc[t] = 0.0f;
    if (STEPS)
#pragma unroll
        for (int t = 0; t < MAXT; ++t) cnt[STEPS ? t : 0] = 0.0f;
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x)
#pragma unroll
        for (int t = 0; t < MAXT; ++t)
            if (t < T) {
                acc[t] += sigmoidf_(__ldg(log_odds + b * T + t));
                if (STEPS) cnt[STEPS ? t : 0] += (__ldg(active + t * B + b) != 0) ? 1.0f : 0.0f;
            }
#pragma unroll
    for (int t = 0; t < MAXT; ++t) {
        if (t < T) {
            const float v = warp_sum(acc[t]);
            if ((threadIdx.x & 31) == 0) atomicAdd(psum + t, v);
            if (STEPS) {
                const float n = warp_sum(cnt[STEPS ? t : 0]);
                if ((threadIdx.x & 31) == 0) atomicAdd(psum + T + t, n);
            }
        }
    }
}

struct AsrArgs {
    const float* log_odds;
    const float* shifts;
    const float* scales;
    const float* psum;
    float inv_B;
    long long B;
    int T;
    mog_asr_config cfg;
    // forward
    float* per_image;
    float* components;
    float* margin;
    // backward
    const float* g_per_image;
    const float* g_margin;
    float* d_log_odds;
    float* d_shifts;
    float* d_scales;
    // executed trip count (STEPS forward, nullable)
    int* steps_out;
};

// The reference loop's trip count from the global per-step active counts n[0:T) (psum[T:2T) of the STEPS colsum): the
// loop's `any` test first fails after step t when n[t] == 0, so it ran t + 1 steps; T if every n[t < T-1] is positive.
__device__ __forceinline__ int executed_steps(const float* n, int T) {
    for (int t = 0; t < T - 1; ++t)
        if (!(n[t] > 0.0f)) return t + 1;
    return T;
}

// STEPS: every loop, mean and the margin run over the executed steps T = executed_steps(psum + S, S) only; arrays keep
// row stride S = a.T, and the backward writes exact zeros into the columns t >= T.
template <bool BACKWARD, bool STEPS>
__global__ void __launch_bounds__(kAsrThreads) asr_kernel(const AsrArgs a) {
    const mog_asr_config& cf = a.cfg;
    const int S = a.T;
    const int T = STEPS ? executed_steps(a.psum + S, S) : S, K = cf.num_counts;
    const float cs = cf.canvas_size;
    const bool count_on = cf.gamma_margin > 1e-8f;  // :973 gates BOTH count penalties
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;

    // ---- batch-level marginal term (:979-991): one thread of the grid writes it ----
    if (!BACKWARD && b == 0) {
        float m = 0.0f;
        if (count_on)
            for (int t = 0; t < T; ++t) {
                float mobj = 0.0f;
                for (int k = 0; k < K; ++k) mobj += (t < cf.counts[k]) ? 1.0f : 0.0f;
                mobj /= (float)K;
                const float pbar = a.psum[t] * a.inv_B;
                m += bce_logits(mobj, logit_eps(pbar)) * cf.gamma_margin;
            }
        *a.margin = m;
        if (STEPS && a.steps_out) *a.steps_out = T;
    }
    if (b >= a.B) return;

    float lo[MAXT], P[MAXT], px[MAXT], cx[MAXT], cy[MAXT];
    for (int t = 0; t < T; ++t) {
        lo[t] = __ldg(a.log_odds + b * S + t);
        P[t] = sigmoidf_(lo[t]);
        px[t] = __ldg(a.scales + b * S + t) * cs;
        cx[t] = (__ldg(a.shifts + (b * S + t) * 2 + 0) + 1.0f) * cs / 2.0f;
        cy[t] = (__ldg(a.shifts + (b * S + t) * 2 + 1) + 1.0f) * cs / 2.0f;
    }

    // ---- min-element count penalty (:993-1010) ----
    float bce_k[MAXK];
    float elem_min = 0.0f;
    int nties = 0;
    if (count_on) {
        for (int k = 0; k < K; ++k) {
            float s = 0.0f;
            for (int t = 0; t < T; ++t) s += bce_logits((t < cf.counts[k]) ? 1.0f : 0.0f, logit_eps(P[t]));
            bce_k[k] = s;
            elem_min = (k == 0) ? s : fminf(elem_min, s);
        }
        for (int k = 0; k < K; ++k) nties += (bce_k[k] == elem_min) ? 1 : 0;
    }

    if (!BACKWARD) {
        float pr_num = 0.0f;
        if (cf.gamma_num > 1e-8f)
            for (int t = 0; t < T; ++t)
                pr_num += (P[t] * softplusf_(-lo[t]) + (1.0f - P[t]) * softplusf_(lo[t])) * cf.gamma_num;  // :676-678
        float area = 0.0f, outl = 0.0f, size = 0.0f, over = 0.0f;
        for (int t = 0; t < T; ++t) {
            area += fmaxf(cf.size_max - px[t], 0.0f) + fmaxf(px[t] - cf.size_min, 0.0f);  // :1018-1023
            const float minx = cx[t] - 0.5f * px[t], miny = cy[t] - 0.5f * px[t];
            const float maxx = cx[t] + 0.5f * px[t], maxy = cy[t] + 0.5f * px[t];
            outl += fmaxf(-minx, 0.0f) + fmaxf(-miny, 0.0f) + fmaxf(maxx - cs, 0.0f) + fmaxf(maxy - cs, 0.0f);  // :1041-1044
            for (int u = 0; u < T; ++u) {
                size += fmaxf(fabsf(px[t] - px[u]) - 3.0f, 0.0f);  // :1048-1051
                if (u != t) {
                    const float md = fmaxf(fabsf(cx[t] - cx[u]), fabsf(cy[t] - cy[u]));
                    over += fmaxf((px[t] + px[u]) / 2.0f - md, 0.0f);  // :1054-1062
                }
            }
        }
        area /= (float)T;  // reduce_mean over steps (:1024-1025)
        const float elem = count_on ? elem_min * cf.gamma_elem : 0.0f;
        a.per_image[b] = pr_num + cf.gamma_area * area + cf.gamma_bbox * (over + outl) + cf.gamma_size * size + elem;
        if (a.components) {
            float* c = a.components + b * MOG_ASR_NUM_COMPONENTS;
            c[0] = pr_num; c[1] = elem; c[2] = area; c[3] = outl; c[4] = size; c[5] = over;
        }
        return;
    }

    // ---- backward ----
    const float gp = __ldg(a.g_per_image + b);
    const float gm = a.g_margin ? __ldg(a.g_margin) : 0.0f;
    float dpx[MAXT], dcx[MAXT], dcy[MAXT];
    for (int t = 0; t < T; ++t) { dpx[t] = 0.0f; dcx[t] = 0.0f; dcy[t] = 0.0f; }
    for (int t = 0; t < T; ++t) {
        // log-odds path: entropy + count penalties
        float dlo = 0.0f;
        if (cf.gamma_num > 1e-8f) dlo += gp * cf.gamma_num * (-lo[t] * P[t] * (1.0f - P[t]));
        if (count_on) {
            const float x = logit_eps(P[t]);
            const float sx = sigmoidf_(x);
            float dx = 0.0f;
            for (int k = 0; k < K; ++k)
                if (bce_k[k] == elem_min) dx += sx - ((t < cf.counts[k]) ? 1.0f : 0.0f);
            float dP = gp * cf.gamma_elem * (dx / (float)nties) * dlogit_eps(P[t]);
            float mobj = 0.0f;
            for (int k = 0; k < K; ++k) mobj += (t < cf.counts[k]) ? 1.0f : 0.0f;
            mobj /= (float)K;
            const float pbar = a.psum[t] * a.inv_B;
            dP += gm * cf.gamma_margin * (sigmoidf_(logit_eps(pbar)) - mobj) * dlogit_eps(pbar) * a.inv_B;
            dlo += dP * P[t] * (1.0f - P[t]);
        }
        a.d_log_odds[b * S + t] = dlo;

        // geometry path
        const float ga = gp * cf.gamma_area / (float)T;
        dpx[t] += ga * (((px[t] - cf.size_min) >= 0.0f ? 1.0f : 0.0f) - ((cf.size_max - px[t]) >= 0.0f ? 1.0f : 0.0f));
        const float gb = gp * cf.gamma_bbox;
        const float minx = cx[t] - 0.5f * px[t], miny = cy[t] - 0.5f * px[t];
        const float maxx = cx[t] + 0.5f * px[t], maxy = cy[t] + 0.5f * px[t];
        const float lx = (-minx >= 0.0f) ? 1.0f : 0.0f, ly = (-miny >= 0.0f) ? 1.0f : 0.0f;
        const float hx = (maxx - cs >= 0.0f) ? 1.0f : 0.0f, hy = (maxy - cs >= 0.0f) ? 1.0f : 0.0f;
        dcx[t] += gb * (hx - lx);
        dcy[t] += gb * (hy - ly);
        dpx[t] += gb * 0.5f * (lx + ly + hx + hy);
        const float gs = gp * cf.gamma_size;
        for (int u = 0; u < T; ++u) {
            const float d = px[t] - px[u];
            if (fabsf(d) - 3.0f >= 0.0f) {  // ordered pair (t,u): d/dpx_t = sgn(d), d/dpx_u = -sgn(d)
                dpx[t] += gs * sgn(d);
                dpx[u] -= gs * sgn(d);
            }
            if (u != t) {
                const float xd = fabsf(cx[t] - cx[u]), yd = fabsf(cy[t] - cy[u]);
                const float v = (px[t] + px[u]) / 2.0f - fmaxf(xd, yd);
                if (v >= 0.0f) {
                    dpx[t] += gb * 0.5f;
                    dpx[u] += gb * 0.5f;
                    if (xd >= yd) {
                        const float s = sgn(cx[t] - cx[u]);
                        dcx[t] -= gb * s;
                        dcx[u] += gb * s;
                    } else {
                        const float s = sgn(cy[t] - cy[u]);
                        dcy[t] -= gb * s;
                        dcy[u] += gb * s;
                    }
                }
            }
        }
    }
    for (int t = 0; t < T; ++t) {
        a.d_scales[b * S + t] = dpx[t] * cs;
        a.d_shifts[(b * S + t) * 2 + 0] = dcx[t] * cs / 2.0f;
        a.d_shifts[(b * S + t) * 2 + 1] = dcy[t] * cs / 2.0f;
    }
    if (STEPS)
        for (int t = T; t < S; ++t) {
            a.d_log_odds[b * S + t] = 0.0f;
            a.d_scales[b * S + t] = 0.0f;
            a.d_shifts[(b * S + t) * 2 + 0] = 0.0f;
            a.d_shifts[(b * S + t) * 2 + 1] = 0.0f;
        }
}

static int check_asr(long long B, int T, const mog_asr_config* cfg) {
    MOG_REQUIRE(B >= 0 && T > 0 && T <= MAXT, MOG_ERR_DIM, "asr: need B >= 0 and 1 <= T <= %d (B=%lld T=%d)", MAXT, B, T);
    MOG_REQUIRE(cfg != nullptr, MOG_ERR_NULL, "asr: cfg is NULL");
    MOG_REQUIRE(cfg->num_counts >= 0 && cfg->num_counts <= MAXK, MOG_ERR_DIM, "asr: num_counts=%d out of [0,%d]",
                cfg->num_counts, MAXK);
    MOG_REQUIRE(!(cfg->gamma_margin > 1e-8f) || cfg->num_counts > 0, MOG_ERR_DIM,
                "asr: gamma_margin > 0 needs at least one count");
    return MOG_OK;
}

// The launches of the plain entry points and of their *_steps forms (STEPS: psum has 2T floats, the second half the global
// per-step active counts that give the executed trip count; psum is then required whatever gamma_margin is).
template <bool STEPS>
static int asr_colsum(const float* log_odds, const unsigned char* active, float* psum, long long B, int T,
                      cudaStream_t stream) {
    MOG_REQUIRE(B >= 0 && T > 0 && T <= MAXT, MOG_ERR_DIM, "asr colsum: need 1 <= T <= %d (T=%d)", MAXT, T);
    MOG_REQUIRE(B == 0 || (log_odds && psum && (!STEPS || active)), MOG_ERR_NULL, "asr colsum: NULL pointer");
    if (B == 0) return MOG_OK;
    long long blocks = (B + 255) / 256;
    const long long cap = (long long)sm_count() * 4;
    if (blocks > cap) blocks = cap;
    asr_colsum_kernel<STEPS><<<(int)blocks, 256, 0, stream>>>(log_odds, psum, B, T, active);
    MOG_CUDA_LAUNCH_CHECK(STEPS ? "asr_colsum_kernel<steps>" : "asr_colsum_kernel");
    return MOG_OK;
}

template <bool STEPS>
static int asr_forward(const float* log_odds, const float* shifts, const float* scales, const float* psum,
                       float inv_global_batch, long long B, int T, const mog_asr_config* cfg, float* per_image,
                       float* components, float* margin, int* steps_out, cudaStream_t stream) {
    if (int rc = check_asr(B, T, cfg)) return rc;
    MOG_REQUIRE(margin && (B == 0 || (log_odds && shifts && scales && per_image)), MOG_ERR_NULL, "asr forward: NULL pointer");
    MOG_REQUIRE(STEPS ? psum != nullptr : (!(cfg->gamma_margin > 1e-8f) || psum), MOG_ERR_NULL,
                STEPS ? "asr forward: psum (2T floats) required" : "asr forward: psum required when gamma_margin > 0");
    AsrArgs a{};
    a.log_odds = log_odds; a.shifts = shifts; a.scales = scales; a.psum = psum; a.inv_B = inv_global_batch;
    a.B = B; a.T = T; a.cfg = *cfg; a.per_image = per_image; a.components = components; a.margin = margin;
    a.steps_out = steps_out;
    const long long blocks = B > 0 ? (B + kAsrThreads - 1) / kAsrThreads : 1;
    asr_kernel<false, STEPS><<<(int)blocks, kAsrThreads, 0, stream>>>(a);
    MOG_CUDA_LAUNCH_CHECK(STEPS ? "asr_kernel<fwd, steps>" : "asr_kernel<fwd>");
    return MOG_OK;
}

template <bool STEPS>
static int asr_backward(const float* log_odds, const float* shifts, const float* scales, const float* psum,
                        float inv_global_batch, const float* g_per_image, const float* g_margin, long long B, int T,
                        const mog_asr_config* cfg, float* d_log_odds, float* d_shifts, float* d_scales,
                        cudaStream_t stream) {
    if (int rc = check_asr(B, T, cfg)) return rc;
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(log_odds && shifts && scales && g_per_image && d_log_odds && d_shifts && d_scales, MOG_ERR_NULL,
                "asr backward: NULL pointer");
    MOG_REQUIRE(STEPS ? psum != nullptr : (!(cfg->gamma_margin > 1e-8f) || psum), MOG_ERR_NULL,
                STEPS ? "asr backward: psum (2T floats) required" : "asr backward: psum required when gamma_margin > 0");
    AsrArgs a{};
    a.log_odds = log_odds; a.shifts = shifts; a.scales = scales; a.psum = psum; a.inv_B = inv_global_batch;
    a.B = B; a.T = T; a.cfg = *cfg; a.g_per_image = g_per_image; a.g_margin = g_margin;
    a.d_log_odds = d_log_odds; a.d_shifts = d_shifts; a.d_scales = d_scales;
    const long long blocks = (B + kAsrThreads - 1) / kAsrThreads;
    asr_kernel<true, STEPS><<<(int)blocks, kAsrThreads, 0, stream>>>(a);
    MOG_CUDA_LAUNCH_CHECK(STEPS ? "asr_kernel<bwd, steps>" : "asr_kernel<bwd>");
    return MOG_OK;
}

}  // namespace mog

using namespace mog;

extern "C" int mog_asr_reg_colsum(const float* log_odds, float* psum, int64_t B, int T, void* stream) {
    return asr_colsum<false>(log_odds, nullptr, psum, B, T, (cudaStream_t)stream);
}

extern "C" int mog_asr_reg_colsum_steps(const float* log_odds, const unsigned char* active, float* psum, int64_t B, int T,
                                        void* stream) {
    return asr_colsum<true>(log_odds, active, psum, B, T, (cudaStream_t)stream);
}

extern "C" int mog_asr_reg_forward(const float* log_odds, const float* shifts, const float* scales, const float* psum,
                                   float inv_global_batch, int64_t B, int T, const mog_asr_config* cfg,
                                   float* per_image, float* components, float* margin, void* stream) {
    return asr_forward<false>(log_odds, shifts, scales, psum, inv_global_batch, B, T, cfg, per_image, components, margin,
                              nullptr, (cudaStream_t)stream);
}

extern "C" int mog_asr_reg_forward_steps(const float* log_odds, const float* shifts, const float* scales,
                                         const float* psum, float inv_global_batch, int64_t B, int T,
                                         const mog_asr_config* cfg, float* per_image, float* components, float* margin,
                                         int32_t* steps_out, void* stream) {
    return asr_forward<true>(log_odds, shifts, scales, psum, inv_global_batch, B, T, cfg, per_image, components, margin,
                             steps_out, (cudaStream_t)stream);
}

extern "C" int mog_asr_reg_backward(const float* log_odds, const float* shifts, const float* scales, const float* psum,
                                    float inv_global_batch, const float* g_per_image, const float* g_margin, int64_t B,
                                    int T, const mog_asr_config* cfg, float* d_log_odds, float* d_shifts,
                                    float* d_scales, void* stream) {
    return asr_backward<false>(log_odds, shifts, scales, psum, inv_global_batch, g_per_image, g_margin, B, T, cfg,
                               d_log_odds, d_shifts, d_scales, (cudaStream_t)stream);
}

extern "C" int mog_asr_reg_backward_steps(const float* log_odds, const float* shifts, const float* scales,
                                          const float* psum, float inv_global_batch, const float* g_per_image,
                                          const float* g_margin, int64_t B, int T, const mog_asr_config* cfg,
                                          float* d_log_odds, float* d_shifts, float* d_scales, void* stream) {
    return asr_backward<true>(log_odds, shifts, scales, psum, inv_global_batch, g_per_image, g_margin, B, T, cfg,
                              d_log_odds, d_shifts, d_scales, (cudaStream_t)stream);
}
