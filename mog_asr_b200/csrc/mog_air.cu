// libmogstn -- per-step elementwise math of the AIR loop body, fused (SURVEY 8(f) rank 2).
//
// /root/reference/air/air_number_bbox_location.py builds these from ~10 TF ops each, every loop iteration:
//   gauss_sample : _sample_from_mvn (:180-184) + tanh/sigmoid squashing of the shift / scale latents (:433-436,
//                  :456-459) and the VAE latent draw (air/vae.py:28-31):  latent = mean + eps*sqrt(exp(logvar))
//   thetas       : theta_r = [[s,0,x],[0,s,y]] (:511-531), theta_w = [[1/s,0,-x/s],[0,1/s,-y/s]] (:563-584)
//   zpres        : Concrete sample y = (log_odds + log(u+eps) - log(1-u+eps))/temperature (air/concrete.py:20-27),
//                  z_pres = sigmoid(y) (:631), stopping_sum += 1 - z_pres (:712), the two activity masks
//                  (stopping_sum < threshold before / after the update, :698-702 / :722-787)
// One launch forward and one backward each; [B]-wide, latency-bound (no roofline claim).
#include "mog_common.cuh"

namespace mog {

constexpr int kAirThreads = 256;
static inline int air_blocks(long long n) {
    long long b = (n + kAirThreads - 1) / kAirThreads;
    const long long cap = (long long)sm_count() * 8;
    return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

// act: 0 = none, 1 = tanh, 2 = sigmoid
__global__ void air_gauss_fwd(const float* __restrict__ mean, const float* __restrict__ logvar, const float* __restrict__ eps,
                              float* __restrict__ latent, float* __restrict__ squashed, long long n, int act) {
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const float l = mean[k] + eps[k] * sqrtf(expf(logvar[k]));
        latent[k] = l;
        if (act == 1) squashed[k] = tanhf(l);
        else if (act == 2) squashed[k] = 1.0f / (1.0f + expf(-l));
    }
}

// g_latent / g_squashed nullable; squashed = saved forward output (act != 0)
__global__ void air_gauss_bwd(const float* __restrict__ logvar, const float* __restrict__ eps, const float* __restrict__ squashed,
                              const float* __restrict__ g_latent, const float* __restrict__ g_squashed,
                              float* __restrict__ d_mean, float* __restrict__ d_logvar, long long n, int act) {
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        float dl = g_latent ? g_latent[k] : 0.0f;
        if (act != 0 && g_squashed) {
            const float a = squashed[k];
            dl += g_squashed[k] * (act == 1 ? (1.0f - a * a) : a * (1.0f - a));
        }
        d_mean[k] = dl;
        d_logvar[k] = dl * eps[k] * 0.5f * sqrtf(expf(logvar[k]));
    }
}

__global__ void air_thetas_fwd(const float* __restrict__ shift, const float* __restrict__ scale, float* __restrict__ theta_r,
                               float* __restrict__ theta_w, long long B) {
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        const float s = scale[b], x = shift[2 * b], y = shift[2 * b + 1];
        float* r = theta_r + 6 * b;
        r[0] = s; r[1] = 0.0f; r[2] = x; r[3] = 0.0f; r[4] = s; r[5] = y;
        float* w = theta_w + 6 * b;
        const float inv = 1.0f / s;          // fp32 divides like the reference graph (:570-578)
        w[0] = inv; w[1] = 0.0f; w[2] = -x / s; w[3] = 0.0f; w[4] = inv; w[5] = -y / s;
    }
}

__global__ void air_thetas_bwd(const float* __restrict__ shift, const float* __restrict__ scale, const float* __restrict__ g_r,
                               const float* __restrict__ g_w, float* __restrict__ d_shift, float* __restrict__ d_scale, long long B) {
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        const float s = scale[b], x = shift[2 * b], y = shift[2 * b + 1];
        const float* r = g_r + 6 * b;
        const float* w = g_w + 6 * b;
        const float inv = 1.0f / s, inv2 = inv * inv;
        d_scale[b] = (r[0] + r[4]) - (w[0] + w[4]) * inv2 + (x * w[2] + y * w[5]) * inv2;
        d_shift[2 * b] = r[2] - w[2] * inv;
        d_shift[2 * b + 1] = r[5] - w[5] * inv;
    }
}

__global__ void air_zpres_fwd(const float* __restrict__ log_odds, const float* __restrict__ u, const float* __restrict__ stop_in,
                              float temperature, float threshold, float* __restrict__ y_pre, float* __restrict__ z_pres,
                              float* __restrict__ stop_out, unsigned char* __restrict__ active_prev,
                              unsigned char* __restrict__ active, long long B) {
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        const float uu = u[b];
        const float y = (log_odds[b] + logf(uu + 10e-10f) - logf(1.0f - uu + 10e-10f)) / temperature;
        const float z = 1.0f / (1.0f + expf(-y));
        const float s0 = stop_in[b], s1 = s0 + (1.0f - z);
        y_pre[b] = y; z_pres[b] = z; stop_out[b] = s1;
        active_prev[b] = s0 < threshold; active[b] = s1 < threshold;
    }
}

__global__ void air_zpres_bwd(const float* __restrict__ z_pres, const float* __restrict__ g_y, const float* __restrict__ g_z,
                              float temperature, float* __restrict__ d_log_odds, long long B) {
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        const float z = z_pres[b];
        const float dy = (g_y ? g_y[b] : 0.0f) + (g_z ? g_z[b] * z * (1.0f - z) : 0.0f);
        d_log_odds[b] = dy / temperature;
    }
}

// LSTM cell pointwise part (tf.nn.rnn_cell.LSTMCell, :865-872): gates [B][4H] in the order i, j, f, o,
// c' = sigmoid(f + 1)*c + sigmoid(i)*tanh(j),  h' = sigmoid(o)*tanh(c')   (forget_bias = 1)
// gates2 (nullable): a second addend of the gate pre-activations (the part of the LSTM input that is the same at every
// step, computed once), so that the per-step GEMM does not need an accumulate-into-a-copy
__global__ void air_lstm_fwd(const float* __restrict__ gates, const float* __restrict__ gates2, const float* __restrict__ c_prev,
                             float* __restrict__ c_new, float* __restrict__ h_new, long long B, int H) {
    const long long n = B * (long long)H;
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const long long b = k / H;
        const int u = (int)(k - b * H);
        const float* gr = gates + b * 4 * H;
        float gi = gr[u], gj = gr[H + u], gf = gr[2 * H + u], go = gr[3 * H + u];
        if (gates2) {
            const float* g2 = gates2 + b * 4 * H;
            gi += g2[u]; gj += g2[H + u]; gf += g2[2 * H + u]; go += g2[3 * H + u];
        }
        const float i = 1.0f / (1.0f + expf(-gi)), j = tanhf(gj);
        const float f = 1.0f / (1.0f + expf(-(gf + 1.0f))), o = 1.0f / (1.0f + expf(-go));
        const float c = f * c_prev[k] + i * j;
        c_new[k] = c;
        h_new[k] = o * tanhf(c);
    }
}

// g_h / g_c nullable (gradients w.r.t. h' and c'); d_gates [B][4H], d_c_prev [B][H] fully overwritten
__global__ void air_lstm_bwd(const float* __restrict__ gates, const float* __restrict__ gates2, const float* __restrict__ c_prev,
                             const float* __restrict__ c_new, const float* __restrict__ g_h, const float* __restrict__ g_c,
                             float* __restrict__ d_gates, float* __restrict__ d_c_prev, long long B, int H) {
    const long long n = B * (long long)H;
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const long long b = k / H;
        const int u = (int)(k - b * H);
        const float* gr = gates + b * 4 * H;
        float* dg = d_gates + b * 4 * H;
        float gi = gr[u], gj = gr[H + u], gf = gr[2 * H + u], go = gr[3 * H + u];
        if (gates2) {
            const float* g2 = gates2 + b * 4 * H;
            gi += g2[u]; gj += g2[H + u]; gf += g2[2 * H + u]; go += g2[3 * H + u];
        }
        const float i = 1.0f / (1.0f + expf(-gi)), j = tanhf(gj);
        const float f = 1.0f / (1.0f + expf(-(gf + 1.0f))), o = 1.0f / (1.0f + expf(-go));
        const float tc = tanhf(c_new[k]);
        const float dh = g_h ? g_h[k] : 0.0f;
        const float dc = (g_c ? g_c[k] : 0.0f) + dh * o * (1.0f - tc * tc);
        dg[u] = dc * j * i * (1.0f - i);
        dg[H + u] = dc * i * (1.0f - j * j);
        dg[2 * H + u] = dc * c_prev[k] * f * (1.0f - f);
        dg[3 * H + u] = dh * tc * o * (1.0f - o);
        d_c_prev[k] = dc * f;
    }
}

// ---- the four KL terms of the ELBO, all steps at once ----------------------------------------------------------
// Inputs are [T][B][...] stacks of the per-step tensors; output kl[b] = sum_t ( mask_prev*z_pres_kl + mask*(scale_kl +
// shift_kl + vae_kl) ) (air_number_bbox_location.py:690-787 masked and summed as at :930-935), plus the four separate
// per-image sums the reference logs (components [B][4]: z_pres, scale, shift, vae).
struct KlArgs {
    const float *y_pre, *prior_lo, *post_lo;              // [T][B]
    const unsigned char *active_prev, *active;            // [T][B]
    const float *sc_mean, *sc_lv;                         // [T][B]      (scale latent is 1-d)
    const float *sh_mean, *sh_lv, *g_sh_mean, *g_sh_lv;   // [T][B][2]
    const float *v_mean, *v_lv;                           // [T][B][L]
    long long B;
    int T, L;
    float temp, sc_prior_mean, sc_prior_var, v_prior_mean, v_prior_var;
    // forward
    float *kl, *components;
    // backward
    const float* g_kl;                                    // [B]
    float *d_y_pre, *d_prior_lo, *d_post_lo, *d_sc_mean, *d_sc_lv, *d_sh_mean, *d_sh_lv, *d_g_sh_mean, *d_g_sh_lv, *d_v_mean,
        *d_v_lv;
};

__device__ __forceinline__ float lse0(float a) { return fmaxf(a, 0.0f) + log1pf(expf(-fabsf(a))); }   // log(1 + e^a)
__device__ __forceinline__ float sigm(float a) { return 1.0f / (1.0f + expf(-a)); }

template <bool BACKWARD>
__global__ void __launch_bounds__(128) air_kl_kernel(const KlArgs a) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    const float log_temp = logf(a.temp + 10e-10f);
    const float g = BACKWARD ? a.g_kl[b] : 0.0f;
    float kz = 0.f, ksc = 0.f, ksh = 0.f, kv = 0.f;
    for (int t = 0; t < a.T; ++t) {
        const long long k = (long long)t * a.B + b;
        const bool mp = a.active_prev[k] != 0, m = a.active[k] != 0;
        // Concrete KL (air/concrete.py:30-64 with equal temperatures)
        const float y = a.y_pre[k], lp = a.prior_lo[k], lq = a.post_lo[k];
        const float ap = -y * a.temp + lp, aq = -y * a.temp + lq;
        if (!BACKWARD) {
            const float log_prior = log_temp - y * (a.temp + 1.0f) + lp - 2.0f * lse0(ap);
            const float log_post = log_temp - y * (a.temp + 1.0f) + lq - 2.0f * lse0(aq);
            if (mp) kz += log_post - log_prior;
        } else {
            const float gz = mp ? g : 0.0f;
            const float sp = sigm(ap), sq = sigm(aq);
            a.d_y_pre[k] = gz * 2.0f * a.temp * (sq - sp);
            a.d_post_lo[k] = gz * (1.0f - 2.0f * sq);
            a.d_prior_lo[k] = -gz * (1.0f - 2.0f * sp);
        }
        const float gm = m ? g : 0.0f;
        {   // scale KL against the fixed prior (:731-736)
            const float mu = a.sc_mean[k], lv = a.sc_lv[k], ev = expf(lv), dm = mu - a.sc_prior_mean;
            if (!BACKWARD) {
                if (m) ksc += 0.5f * (logf(a.sc_prior_var) - lv - 1.0f + ev / a.sc_prior_var + dm * dm / a.sc_prior_var);
            } else {
                a.d_sc_mean[k] = gm * dm / a.sc_prior_var;
                a.d_sc_lv[k] = gm * 0.5f * (ev / a.sc_prior_var - 1.0f);
            }
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) {   // shift KL against the learned prior (:750-755)
            const long long q = 2 * k + c;
            const float mu = a.sh_mean[q], lv = a.sh_lv[q], gmu = a.g_sh_mean[q], glv = a.g_sh_lv[q];
            const float gvar = expf(glv), ev = expf(lv), dm = mu - gmu;
            if (!BACKWARD) {
                if (m) ksh += 0.5f * (glv - lv - 1.0f + ev / gvar + dm * dm / gvar);
            } else {
                a.d_sh_mean[q] = gm * dm / gvar;
                a.d_sh_lv[q] = gm * 0.5f * (ev / gvar - 1.0f);
                a.d_g_sh_mean[q] = -gm * dm / gvar;
                a.d_g_sh_lv[q] = gm * 0.5f * (1.0f - ev / gvar - dm * dm / gvar);
            }
        }
        for (int c = 0; c < a.L; ++c) {   // VAE latent KL (:769-774)
            const long long q = k * a.L + c;
            const float mu = a.v_mean[q], lv = a.v_lv[q], ev = expf(lv), dm = mu - a.v_prior_mean;
            if (!BACKWARD) {
                if (m) kv += 0.5f * (logf(a.v_prior_var) - lv - 1.0f + ev / a.v_prior_var + dm * dm / a.v_prior_var);
            } else {
                a.d_v_mean[q] = gm * dm / a.v_prior_var;
                a.d_v_lv[q] = gm * 0.5f * (ev / a.v_prior_var - 1.0f);
            }
        }
    }
    if (!BACKWARD) {
        a.kl[b] = ((kz + ksc) + ksh) + kv;
        if (a.components) {
            float* c = a.components + 4 * b;
            c[0] = kz; c[1] = ksc; c[2] = ksh; c[3] = kv;
        }
    }
}


// ---- bias + activation epilogue of a dense layer (the GEMM itself is the library's) -------------------------------------
// act: 0 none, 1 relu, 2 softplus (beta 1, linear above 20 like the framework op), 3 sigmoid.  out may alias pre.
__global__ void air_bias_act_fwd(const float* __restrict__ pre, const float* __restrict__ bias, float* __restrict__ out, long long n,
                                 int N, int act) {
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const float v = pre[k] + bias[(int)(k % N)];
        float y = v;
        if (act == 1) y = fmaxf(v, 0.0f);
        else if (act == 2) y = v > 20.0f ? v : log1pf(expf(v));
        else if (act == 3) y = 1.0f / (1.0f + expf(-v));
        out[k] = y;
    }
}
// dpre = g * act'(.) expressed through the saved OUTPUT y; dpre may alias g
__global__ void air_bias_act_bwd(const float* __restrict__ y, const float* __restrict__ g, float* __restrict__ dpre, long long n, int act) {
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const float o = y[k];
        float d = g[k];
        if (act == 1) d = o > 0.0f ? d : 0.0f;
        // softplus' = sigmoid(v) = 1 - exp(-softplus(v)); written as -expm1(-o) because for v << 0, o ~ e^v is tiny and
        // 1 - expf(-o) cancels (relative error 1e-5 at v = -5, the gradient exactly 0 below v ~ -17)
        else if (act == 2) d = o > 20.0f ? d : d * -expm1f(-o);
        else if (act == 3) d = d * o * (1.0f - o);
        dpre[k] = d;
    }
}
// pre [B][2L] = x [Wmean | Wlogvar]: add the biases, split, draw the sample (vae.py:21-31)
__global__ void air_bias_gauss_fwd(const float* __restrict__ pre, const float* __restrict__ bm, const float* __restrict__ bv,
                                   const float* __restrict__ eps, float* __restrict__ mean, float* __restrict__ logvar,
                                   float* __restrict__ latent, long long B, int Ld) {
    const long long n = B * Ld;
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const long long b = k / Ld;
        const int l = (int)(k - b * Ld);
        const float m = pre[b * 2 * Ld + l] + bm[l], lv = pre[b * 2 * Ld + Ld + l] + bv[l];
        mean[k] = m; logvar[k] = lv;
        latent[k] = m + eps[k] * sqrtf(expf(lv));
    }
}
__global__ void air_bias_gauss_bwd(const float* __restrict__ logvar, const float* __restrict__ eps, const float* __restrict__ g_mean,
                                   const float* __restrict__ g_logvar, const float* __restrict__ g_latent, float* __restrict__ dpre,
                                   long long B, int Ld) {
    const long long n = B * Ld;
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
        const long long b = k / Ld;
        const int l = (int)(k - b * Ld);
        const float dl = g_latent ? g_latent[k] : 0.0f;
        dpre[b * 2 * Ld + l] = (g_mean ? g_mean[k] : 0.0f) + dl;
        dpre[b * 2 * Ld + Ld + l] = (g_logvar ? g_logvar[k] : 0.0f) + dl * eps[k] * 0.5f * sqrtf(expf(logvar[k]));
    }
}

}  // namespace mog

using namespace mog;

static int check_kl(const KlArgs& a) {
    MOG_REQUIRE(a.B >= 0 && a.T > 0 && a.L > 0 && a.temp > 0.0f && a.sc_prior_var > 0.0f && a.v_prior_var > 0.0f, MOG_ERR_DIM,
                "air kl: B=%lld T=%d L=%d temp=%g", a.B, a.T, a.L, (double)a.temp);
    MOG_REQUIRE(a.B == 0 || (a.y_pre && a.prior_lo && a.post_lo && a.active_prev && a.active && a.sc_mean && a.sc_lv && a.sh_mean &&
                             a.sh_lv && a.g_sh_mean && a.g_sh_lv && a.v_mean && a.v_lv), MOG_ERR_NULL, "air kl: NULL input pointer");
    return MOG_OK;
}

extern "C" int mog_air_kl_forward(const float* y_pre, const float* prior_lo, const float* post_lo, const unsigned char* active_prev,
                                  const unsigned char* active, const float* sc_mean, const float* sc_lv, const float* sh_mean,
                                  const float* sh_lv, const float* g_sh_mean, const float* g_sh_lv, const float* v_mean,
                                  const float* v_lv, int64_t B, int T, int L, float temperature, float scale_prior_mean,
                                  float scale_prior_var, float vae_prior_mean, float vae_prior_var, float* kl, float* components,
                                  void* stream) {
    KlArgs a{};
    a.y_pre = y_pre; a.prior_lo = prior_lo; a.post_lo = post_lo; a.active_prev = active_prev; a.active = active;
    a.sc_mean = sc_mean; a.sc_lv = sc_lv; a.sh_mean = sh_mean; a.sh_lv = sh_lv; a.g_sh_mean = g_sh_mean; a.g_sh_lv = g_sh_lv;
    a.v_mean = v_mean; a.v_lv = v_lv; a.B = B; a.T = T; a.L = L; a.temp = temperature; a.sc_prior_mean = scale_prior_mean;
    a.sc_prior_var = scale_prior_var; a.v_prior_mean = vae_prior_mean; a.v_prior_var = vae_prior_var; a.kl = kl; a.components = components;
    if (int rc = check_kl(a)) return rc;
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(kl, MOG_ERR_NULL, "air kl forward: NULL output");
    air_kl_kernel<false><<<(int)((B + 127) / 128), 128, 0, (cudaStream_t)stream>>>(a);
    MOG_CUDA_LAUNCH_CHECK("air_kl_kernel<fwd>");
    return MOG_OK;
}

extern "C" int mog_air_kl_backward(const float* y_pre, const float* prior_lo, const float* post_lo, const unsigned char* active_prev,
                                   const unsigned char* active, const float* sc_mean, const float* sc_lv, const float* sh_mean,
                                   const float* sh_lv, const float* g_sh_mean, const float* g_sh_lv, const float* v_mean,
                                   const float* v_lv, int64_t B, int T, int L, float temperature, float scale_prior_mean,
                                   float scale_prior_var, float vae_prior_mean, float vae_prior_var, const float* g_kl,
                                   float* d_y_pre, float* d_prior_lo, float* d_post_lo, float* d_sc_mean, float* d_sc_lv,
                                   float* d_sh_mean, float* d_sh_lv, float* d_g_sh_mean, float* d_g_sh_lv, float* d_v_mean,
                                   float* d_v_lv, void* stream) {
    KlArgs a{};
    a.y_pre = y_pre; a.prior_lo = prior_lo; a.post_lo = post_lo; a.active_prev = active_prev; a.active = active;
    a.sc_mean = sc_mean; a.sc_lv = sc_lv; a.sh_mean = sh_mean; a.sh_lv = sh_lv; a.g_sh_mean = g_sh_mean; a.g_sh_lv = g_sh_lv;
    a.v_mean = v_mean; a.v_lv = v_lv; a.B = B; a.T = T; a.L = L; a.temp = temperature; a.sc_prior_mean = scale_prior_mean;
    a.sc_prior_var = scale_prior_var; a.v_prior_mean = vae_prior_mean; a.v_prior_var = vae_prior_var; a.g_kl = g_kl;
    a.d_y_pre = d_y_pre; a.d_prior_lo = d_prior_lo; a.d_post_lo = d_post_lo; a.d_sc_mean = d_sc_mean; a.d_sc_lv = d_sc_lv;
    a.d_sh_mean = d_sh_mean; a.d_sh_lv = d_sh_lv; a.d_g_sh_mean = d_g_sh_mean; a.d_g_sh_lv = d_g_sh_lv; a.d_v_mean = d_v_mean;
    a.d_v_lv = d_v_lv;
    if (int rc = check_kl(a)) return rc;
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(g_kl && d_y_pre && d_prior_lo && d_post_lo && d_sc_mean && d_sc_lv && d_sh_mean && d_sh_lv && d_g_sh_mean && d_g_sh_lv &&
                d_v_mean && d_v_lv, MOG_ERR_NULL, "air kl backward: NULL pointer");
    air_kl_kernel<true><<<(int)((B + 127) / 128), 128, 0, (cudaStream_t)stream>>>(a);
    MOG_CUDA_LAUNCH_CHECK("air_kl_kernel<bwd>");
    return MOG_OK;
}


extern "C" int mog_air_lstm_pointwise_forward(const float* gates, const float* gates2, const float* c_prev, float* c_new, float* h_new, int64_t B,
                                              int H, void* stream) {
    MOG_REQUIRE(B >= 0 && H > 0, MOG_ERR_DIM, "lstm pointwise: B=%lld H=%d", (long long)B, H);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(gates && c_prev && c_new && h_new, MOG_ERR_NULL, "lstm pointwise forward: NULL pointer");
    air_lstm_fwd<<<air_blocks(B * (long long)H), kAirThreads, 0, (cudaStream_t)stream>>>(gates, gates2, c_prev, c_new, h_new, B, H);
    MOG_CUDA_LAUNCH_CHECK("air_lstm_fwd");
    return MOG_OK;
}

extern "C" int mog_air_lstm_pointwise_backward(const float* gates, const float* gates2, const float* c_prev, const float* c_new, const float* g_h,
                                               const float* g_c, float* d_gates, float* d_c_prev, int64_t B, int H,
                                               void* stream) {
    MOG_REQUIRE(B >= 0 && H > 0, MOG_ERR_DIM, "lstm pointwise: B=%lld H=%d", (long long)B, H);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(gates && c_prev && c_new && d_gates && d_c_prev, MOG_ERR_NULL, "lstm pointwise backward: NULL pointer");
    air_lstm_bwd<<<air_blocks(B * (long long)H), kAirThreads, 0, (cudaStream_t)stream>>>(gates, gates2, c_prev, c_new, g_h, g_c, d_gates,
                                                                                       d_c_prev, B, H);
    MOG_CUDA_LAUNCH_CHECK("air_lstm_bwd");
    return MOG_OK;
}


extern "C" int mog_air_gauss_sample_forward(const float* mean, const float* logvar, const float* eps, float* latent,
                                            float* squashed, int64_t n, int act, void* stream) {
    MOG_REQUIRE(n >= 0 && act >= 0 && act <= 2, MOG_ERR_DIM, "gauss_sample: n=%lld act=%d", (long long)n, act);
    if (n == 0) return MOG_OK;
    MOG_REQUIRE(mean && logvar && eps && latent && (act == 0 || squashed), MOG_ERR_NULL, "gauss_sample forward: NULL pointer");
    air_gauss_fwd<<<air_blocks(n), kAirThreads, 0, (cudaStream_t)stream>>>(mean, logvar, eps, latent, squashed, n, act);
    MOG_CUDA_LAUNCH_CHECK("air_gauss_fwd");
    return MOG_OK;
}

extern "C" int mog_air_gauss_sample_backward(const float* logvar, const float* eps, const float* squashed, const float* g_latent,
                                             const float* g_squashed, float* d_mean, float* d_logvar, int64_t n, int act,
                                             void* stream) {
    MOG_REQUIRE(n >= 0 && act >= 0 && act <= 2, MOG_ERR_DIM, "gauss_sample: n=%lld act=%d", (long long)n, act);
    if (n == 0) return MOG_OK;
    MOG_REQUIRE(logvar && eps && d_mean && d_logvar && (act == 0 || !g_squashed || squashed), MOG_ERR_NULL,
                "gauss_sample backward: NULL pointer");
    air_gauss_bwd<<<air_blocks(n), kAirThreads, 0, (cudaStream_t)stream>>>(logvar, eps, squashed, g_latent, g_squashed, d_mean,
                                                                         d_logvar, n, act);
    MOG_CUDA_LAUNCH_CHECK("air_gauss_bwd");
    return MOG_OK;
}

extern "C" int mog_air_thetas_forward(const float* shift, const float* scale, float* theta_r, float* theta_w, int64_t B,
                                      void* stream) {
    MOG_REQUIRE(B >= 0, MOG_ERR_DIM, "thetas: B=%lld", (long long)B);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(shift && scale && theta_r && theta_w, MOG_ERR_NULL, "thetas forward: NULL pointer");
    air_thetas_fwd<<<air_blocks(B), kAirThreads, 0, (cudaStream_t)stream>>>(shift, scale, theta_r, theta_w, B);
    MOG_CUDA_LAUNCH_CHECK("air_thetas_fwd");
    return MOG_OK;
}

extern "C" int mog_air_thetas_backward(const float* shift, const float* scale, const float* g_theta_r, const float* g_theta_w,
                                       float* d_shift, float* d_scale, int64_t B, void* stream) {
    MOG_REQUIRE(B >= 0, MOG_ERR_DIM, "thetas: B=%lld", (long long)B);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(shift && scale && g_theta_r && g_theta_w && d_shift && d_scale, MOG_ERR_NULL, "thetas backward: NULL pointer");
    air_thetas_bwd<<<air_blocks(B), kAirThreads, 0, (cudaStream_t)stream>>>(shift, scale, g_theta_r, g_theta_w, d_shift, d_scale, B);
    MOG_CUDA_LAUNCH_CHECK("air_thetas_bwd");
    return MOG_OK;
}

extern "C" int mog_air_zpres_forward(const float* log_odds, const float* u, const float* stop_in, float temperature,
                                     float threshold, float* y_pre, float* z_pres, float* stop_out, unsigned char* active_prev,
                                     unsigned char* active, int64_t B, void* stream) {
    MOG_REQUIRE(B >= 0 && temperature > 0.0f, MOG_ERR_DIM, "zpres: B=%lld temperature=%g", (long long)B, (double)temperature);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(log_odds && u && stop_in && y_pre && z_pres && stop_out && active_prev && active, MOG_ERR_NULL,
                "zpres forward: NULL pointer");
    air_zpres_fwd<<<air_blocks(B), kAirThreads, 0, (cudaStream_t)stream>>>(log_odds, u, stop_in, temperature, threshold, y_pre,
                                                                         z_pres, stop_out, active_prev, active, B);
    MOG_CUDA_LAUNCH_CHECK("air_zpres_fwd");
    return MOG_OK;
}

extern "C" int mog_air_zpres_backward(const float* z_pres, const float* g_y, const float* g_z, float temperature,
                                      float* d_log_odds, int64_t B, void* stream) {
    MOG_REQUIRE(B >= 0 && temperature > 0.0f, MOG_ERR_DIM, "zpres: B=%lld temperature=%g", (long long)B, (double)temperature);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(z_pres && d_log_odds, MOG_ERR_NULL, "zpres backward: NULL pointer");
    air_zpres_bwd<<<air_blocks(B), kAirThreads, 0, (cudaStream_t)stream>>>(z_pres, g_y, g_z, temperature, d_log_odds, B);
    MOG_CUDA_LAUNCH_CHECK("air_zpres_bwd");
    return MOG_OK;
}

extern "C" int mog_air_bias_act_forward(const float* pre, const float* bias, float* out, int64_t B, int N, int act, void* stream) {
    MOG_REQUIRE(B >= 0 && N > 0 && act >= 0 && act <= 3, MOG_ERR_DIM, "bias_act: B=%lld N=%d act=%d", (long long)B, N, act);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(pre && bias && out, MOG_ERR_NULL, "bias_act forward: NULL pointer");
    air_bias_act_fwd<<<air_blocks(B * (long long)N), kAirThreads, 0, (cudaStream_t)stream>>>(pre, bias, out, B * (long long)N, N, act);
    MOG_CUDA_LAUNCH_CHECK("air_bias_act_fwd");
    return MOG_OK;
}

extern "C" int mog_air_bias_act_backward(const float* y, const float* g, float* dpre, int64_t n, int act, void* stream) {
    MOG_REQUIRE(n >= 0 && act >= 0 && act <= 3, MOG_ERR_DIM, "bias_act: n=%lld act=%d", (long long)n, act);
    if (n == 0) return MOG_OK;
    MOG_REQUIRE(y && g && dpre, MOG_ERR_NULL, "bias_act backward: NULL pointer");
    air_bias_act_bwd<<<air_blocks(n), kAirThreads, 0, (cudaStream_t)stream>>>(y, g, dpre, n, act);
    MOG_CUDA_LAUNCH_CHECK("air_bias_act_bwd");
    return MOG_OK;
}

extern "C" int mog_air_bias_gauss_forward(const float* pre, const float* bias_mean, const float* bias_logvar, const float* eps,
                                          float* mean, float* logvar, float* latent, int64_t B, int L, void* stream) {
    MOG_REQUIRE(B >= 0 && L > 0, MOG_ERR_DIM, "bias_gauss: B=%lld L=%d", (long long)B, L);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(pre && bias_mean && bias_logvar && eps && mean && logvar && latent, MOG_ERR_NULL, "bias_gauss forward: NULL pointer");
    air_bias_gauss_fwd<<<air_blocks(B * (long long)L), kAirThreads, 0, (cudaStream_t)stream>>>(pre, bias_mean, bias_logvar, eps, mean,
                                                                                           logvar, latent, B, L);
    MOG_CUDA_LAUNCH_CHECK("air_bias_gauss_fwd");
    return MOG_OK;
}

extern "C" int mog_air_bias_gauss_backward(const float* logvar, const float* eps, const float* g_mean, const float* g_logvar,
                                           const float* g_latent, float* dpre, int64_t B, int L, void* stream) {
    MOG_REQUIRE(B >= 0 && L > 0, MOG_ERR_DIM, "bias_gauss: B=%lld L=%d", (long long)B, L);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(logvar && eps && dpre, MOG_ERR_NULL, "bias_gauss backward: NULL pointer");
    air_bias_gauss_bwd<<<air_blocks(B * (long long)L), kAirThreads, 0, (cudaStream_t)stream>>>(logvar, eps, g_mean, g_logvar, g_latent,
                                                                                           dpre, B, L);
    MOG_CUDA_LAUNCH_CHECK("air_bias_gauss_bwd");
    return MOG_OK;
}
