// libmogstn -- spatial-transformer sampler of MOG-ASR for B200 (sm_100a).
//
// Replaces the ~70-op TensorFlow graph of /root/reference/air/transformer.py:18-175 (forward) and its
// autodiff (backward) with one kernel each, plus the fused write+composite of
// air/air_number_bbox_location.py:592-600,:718-727.  HBM-bound gather/scatter work: no tensor cores.
//
// Numerical contract (oracle/stn_ref_numpy.py): corner indices bit-exact; forward values computed with
// the reference's operation order, one fp32 rounding per op (explicit _rn intrinsics, no FMA), so they
// are bit-exact for finite inputs too.  Gradients are fp32 with a different (tree) summation order.
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "mog_common.cuh"
#include "mog_stn_warp.cuh"
#include "mog_stn_bwd_col.cuh"

namespace mog {

// ---------------------------------------------------------------------------------------------------
// host-side plumbing
// ---------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

// images of >= 32 KB: the backward's dU is zero-filled by the whole CTA, large zero regions go to the bulk-copy engine
constexpr int kCoopZeroMinFloats = 8192;
constexpr int kStreamCtasPerSm = 64 / kWarpsPerCta;   // grid cap of the forward and the streaming backward: 64 warps per SM
constexpr int kMaxSmemBytes = 200 * 1024;  // leave room under the 227 KB per-CTA limit

// corner probe: same evaluation paths as the forward kernel (tables for separable thetas)
__global__ void __launch_bounds__(256) stn_corners_kernel(const float* theta, int32_t* corners, long long B,
                                                                const Geo g) {
    extern __shared__ int4 s_tab[];
    const long long BN = B * (long long)g.N;
    for (long long b = blockIdx.x; b < B; b += gridDim.x) {
        Theta th;
        th.load(theta + 6 * b);
        const bool sep = th.separable();
        if (sep) {
            __syncthreads();
            build_tables(s_tab, th, g);
            __syncthreads();
        }
        for (int n = threadIdx.x; n < g.N; n += 256) {
            int i, j;
            split_n(g, n, i, j);
            int x0, x1, y0, y1;
            if (sep) {
                const int4 cx = s_tab[j], cy = s_tab[g.Wo + i];
                x0 = cx.x; x1 = cx.y; y0 = cy.x / g.Ws; y1 = cy.y / g.Ws;
            } else {
                Axis X, Y;
                taps_general(th, g, i, j, X, Y);
                x0 = X.c0; x1 = X.c1; y0 = Y.c0; y1 = Y.c1;
            }
            const long long o = b * g.N + n;
            corners[o] = x0;
            corners[BN + o] = x1;
            corners[2 * BN + o] = y0;
            corners[3 * BN + o] = y1;
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------------
static int check_dims(long long B, int Hs, int Ws, int C, int Ho, int Wo, int u_div) {
    MOG_REQUIRE(B >= 0 && Hs > 0 && Ws > 0 && C > 0 && Ho > 0 && Wo > 0, MOG_ERR_DIM,
                "non-positive dimension: B=%lld Hs=%d Ws=%d C=%d Ho=%d Wo=%d", B, Hs, Ws, C, Ho, Wo);
    MOG_REQUIRE(u_div >= 1 && B % u_div == 0, MOG_ERR_DIM, "u_batch_div=%d must be >= 1 and divide B=%lld", u_div, B);
    MOG_REQUIRE((long long)Hs * Ws * C < (1ll << 30) && (long long)Ho * Wo * C < (1ll << 30), MOG_ERR_OVERFLOW,
                "per-image element count exceeds 2^30 (Hs*Ws*C=%lld, Ho*Wo*C=%lld)", (long long)Hs * Ws * C,
                (long long)Ho * Wo * C);
    MOG_REQUIRE((unsigned long long)Ho * Wo * (unsigned long long)Wo < (1ull << 32), MOG_ERR_UNSUPPORTED,
                "Ho*Wo*Wo must be < 2^32 for the index split (Ho=%d Wo=%d)", Ho, Wo);
    MOG_REQUIRE((size_t)(Ho + Wo) * sizeof(int4) <= 64 * 1024, MOG_ERR_UNSUPPORTED, "Ho+Wo=%d too large for the axis tables",
                Ho + Wo);
    return MOG_OK;
}

static int grid_for(long long units, int ctas_per_sm) {
    const long long cap = (long long)sm_count() * ctas_per_sm;
    return (int)(units < cap ? (units > 0 ? units : 1) : cap);
}

template <typename K>
static int set_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) {
            set_error("cudaFuncSetAttribute(%zu B dynamic smem): %s", bytes, cudaGetErrorString(e));
            return (int)e;
        }
    }
    return 0;
}

// Every launcher takes the (s, x, y) arguments: sx.shift == NULL (SxyArgs{}) runs the theta-taking kernel (SXY = 0), otherwise
// theta is built from (s, x, y) in the kernel, SXY = 1 for the read (the plain call), 2 for the write (the composite).  The
// (s, x, y) entry points require a non-NULL shift whenever there is work.
template <bool COMPOSITE>
constexpr int kSxyMode = COMPOSITE ? 2 : 1;

constexpr int kOccupancyCtasPerSm = 0;

// Launch a sampler kernel over `images` images, kWarpsPerCta to a CTA, with at most ctas_per_sm CTAs per SM
// (kOccupancyCtasPerSm: as many as fit at this block and shared-memory size).
template <typename Args>
static int launch_sampler(void (*kernel)(Args, SxyArgs), const char* name, const Args& a, const SxyArgs& sx,
                          long long images, size_t smem, int ctas_per_sm, cudaStream_t st) {
    if (int rc = set_smem(kernel, smem)) return rc;
    if (ctas_per_sm == kOccupancyCtasPerSm &&
        (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kernel, kWarpThreads, smem) != cudaSuccess || ctas_per_sm < 1))
        ctas_per_sm = 1;
    kernel<<<grid_for((images + kWarpsPerCta - 1) / kWarpsPerCta, ctas_per_sm), kWarpThreads, smem, st>>>(a, sx);
    MOG_CUDA_LAUNCH_CHECK(name);
    return MOG_OK;
}

template <bool COMPOSITE>
static int launch_fwd(FwdArgs a, const SxyArgs& sx, cudaStream_t st) {
    if (a.B == 0) return MOG_OK;
    a.bulk_zero = (!COMPOSITE && (long long)a.g.N * a.g.C >= kCoopZeroMinFloats) ? 1 : 0;
    const size_t smem = (size_t)kWarpsPerCta * (a.g.Ho + a.g.Wo) * sizeof(int4) + (a.bulk_zero ? kZeroBytes : 0);
    MOG_REQUIRE(smem <= (size_t)kMaxSmemBytes, MOG_ERR_UNSUPPORTED, "Ho=%d Wo=%d too large for the per-warp tables", a.g.Ho, a.g.Wo);
    return launch_sampler(sx.shift ? stn_fwd_warp_kernel<COMPOSITE, kSxyMode<COMPOSITE>> : stn_fwd_warp_kernel<COMPOSITE, 0>,
                          "stn_fwd_warp_kernel", a, sx, a.B, smem, kStreamCtasPerSm, st);
}

template <bool COMPOSITE, int NXC>
static int launch_bwd_nxc(const BwdArgs& a, const SxyArgs& sx, cudaStream_t st) {
    const size_t smem = (size_t)kWarpsPerCta * bwd_warp_smem_words(a.g) * sizeof(int) + (a.coop_zero == 2 ? kZeroBytes : 0);
    MOG_REQUIRE(smem <= (size_t)kMaxSmemBytes, MOG_ERR_UNSUPPORTED, "Ho=%d Wo=%d Ws=%d too large for the per-warp tables",
                a.g.Ho, a.g.Wo, a.g.Ws);
    return launch_sampler(sx.shift ? stn_bwd_warp_kernel<COMPOSITE, NXC, kSxyMode<COMPOSITE>> : stn_bwd_warp_kernel<COMPOSITE, NXC, 0>,
                          "stn_bwd_warp_kernel", a, sx, a.Bsrc, smem, kStreamCtasPerSm, st);
}

template <bool COMPOSITE>
static int launch_bwd_stream(const BwdArgs& a, const SxyArgs& sx, cudaStream_t st) {
    // NXC = source-column chunks (of 32) kept in registers per streaming pass; wider footprints are strip-mined
    const int nxc = (a.g.Ws + 31) / 32;
    if (nxc <= 1) return launch_bwd_nxc<COMPOSITE, 1>(a, sx, st);
    if (nxc <= 2) return launch_bwd_nxc<COMPOSITE, 2>(a, sx, st);
    return launch_bwd_nxc<COMPOSITE, 4>(a, sx, st);
}

// Source-column form (mog_stn_bwd_col.cuh: one warp per image, lanes along the source columns) for the write direction,
// output at least as large as the source: faster than every other measured form in all 12 sweep cells
// (profiles/r02_kernel_experiments.md).  Everything else streams.
static bool use_bwd_col(const BwdArgs& a) {
    const Geo& g = a.g;
    return g.Wo >= g.Ws && g.Ho >= g.Hs && g.C == 1 && a.u_div == 1 && g.Ws <= kColMaxWs && g.Wo < 65536 &&
           (size_t)bwd_col_layout(g).total * kWarpsPerCta <= (size_t)kMaxSmemBytes;
}

template <bool COMPOSITE, int NCOL>
static int launch_bwd_col_n(const BwdArgs& a, const SxyArgs& sx, cudaStream_t st) {
    return launch_sampler(sx.shift ? stn_bwd_col_kernel<COMPOSITE, NCOL, kSxyMode<COMPOSITE>> : stn_bwd_col_kernel<COMPOSITE, NCOL, 0>,
                          "stn_bwd_col_kernel", a, sx, a.Bsrc, (size_t)bwd_col_layout(a.g).total * kWarpsPerCta,
                          kOccupancyCtasPerSm, st);
}

template <bool COMPOSITE>
static int launch_bwd(BwdArgs a, const SxyArgs& sx, cudaStream_t st) {
    if (a.Bsrc == 0) return MOG_OK;
    a.coop_zero = (long long)a.g.S * a.g.C >= kCoopZeroMinFloats ? 1 : 0;
    if (a.coop_zero && a.dU && a.u_div == 1 && a.g.C == 1) a.coop_zero = 2;
    if (use_bwd_col(a))
        return a.g.Ws <= 32 ? launch_bwd_col_n<COMPOSITE, 1>(a, sx, st) : launch_bwd_col_n<COMPOSITE, 2>(a, sx, st);
    return launch_bwd_stream<COMPOSITE>(a, sx, st);
}

}  // namespace mog

// ---------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------
using namespace mog;

extern "C" int mog_version(void) { return MOG_ABI_VERSION; }

extern "C" int mog_last_error_string(char* buf, size_t n) {
    const size_t len = strlen(g_err);
    if (buf && n) {
        const size_t k = len < n - 1 ? len : n - 1;
        memcpy(buf, g_err, k);
        buf[k] = 0;
    }
    return (int)len;
}

extern "C" int mog_stn_forward(const float* U, const float* theta, float* out, int64_t B, int Hs, int Ws, int C,
                               int Ho, int Wo, int u_batch_div, void* stream) {
    if (int rc = check_dims(B, Hs, Ws, C, Ho, Wo, u_batch_div)) return rc;
    MOG_REQUIRE(B == 0 || (U && theta && out), MOG_ERR_NULL, "mog_stn_forward: NULL pointer (U=%p theta=%p out=%p)", (const void*)U,
                (const void*)theta, (void*)out);
    FwdArgs a{};
    a.U = U; a.theta = theta; a.out = out; a.B = B; a.u_div = u_batch_div;
    a.g = make_geo(Hs, Ws, C, Ho, Wo);
    return launch_fwd<false>(a, SxyArgs{}, (cudaStream_t)stream);
}

extern "C" int mog_stn_corners(const float* theta, int32_t* corners, int64_t B, int Hs, int Ws, int Ho, int Wo,
                               void* stream) {
    if (int rc = check_dims(B, Hs, Ws, 1, Ho, Wo, 1)) return rc;
    MOG_REQUIRE(B == 0 || (theta && corners), MOG_ERR_NULL, "mog_stn_corners: NULL pointer");
    if (B == 0) return MOG_OK;
    const Geo g = make_geo(Hs, Ws, 1, Ho, Wo);
    const size_t smem = (size_t)(Wo + Ho) * sizeof(int4);
    if (int rc = set_smem(stn_corners_kernel, smem)) return rc;
    stn_corners_kernel<<<grid_for(B, 8), 256, smem, (cudaStream_t)stream>>>(theta, corners, B, g);
    MOG_CUDA_LAUNCH_CHECK("stn_corners_kernel");
    return MOG_OK;
}

extern "C" int mog_stn_backward(const float* U, const float* theta, const float* gout, float* dU, float* dtheta,
                                int64_t B, int Hs, int Ws, int C, int Ho, int Wo, int u_batch_div, void* stream) {
    if (int rc = check_dims(B, Hs, Ws, C, Ho, Wo, u_batch_div)) return rc;
    MOG_REQUIRE(B == 0 || (U && theta && gout), MOG_ERR_NULL, "mog_stn_backward: NULL pointer (U=%p theta=%p gout=%p)",
                (const void*)U, (const void*)theta, (const void*)gout);
    if (!dU && !dtheta) return MOG_OK;
    BwdArgs a{};
    a.U = U; a.theta = theta; a.gout = gout; a.dU = dU; a.dtheta = dtheta;
    a.Bsrc = B / u_batch_div; a.u_div = u_batch_div;
    a.g = make_geo(Hs, Ws, C, Ho, Wo);
    return launch_bwd<false>(a, SxyArgs{}, (cudaStream_t)stream);
}

extern "C" int mog_stn_write_composite_forward(const float* U, const float* theta, const float* z_pres,
                                               const float* stop_sum, float threshold, const float* canvas_in,
                                               float* canvas_out, int64_t B, int Hw, int Ww, int Hc, int Wc,
                                               void* stream) {
    if (int rc = check_dims(B, Hw, Ww, 1, Hc, Wc, 1)) return rc;
    MOG_REQUIRE(B == 0 || (U && theta && z_pres && canvas_in && canvas_out), MOG_ERR_NULL,
                "mog_stn_write_composite_forward: NULL pointer");
    FwdArgs a{};
    a.U = U; a.theta = theta; a.out = canvas_out; a.z_pres = z_pres; a.stop_sum = stop_sum; a.canvas_in = canvas_in;
    a.threshold = threshold; a.B = B; a.u_div = 1;
    a.g = make_geo(Hw, Ww, 1, Hc, Wc);
    return launch_fwd<true>(a, SxyArgs{}, (cudaStream_t)stream);
}

extern "C" int mog_stn_write_composite_backward(const float* U, const float* theta, const float* z_pres,
                                                const float* stop_sum, float threshold, const float* gcanvas,
                                                float* dU, float* dtheta, float* dz, int64_t B, int Hw, int Ww,
                                                int Hc, int Wc, void* stream) {
    if (int rc = check_dims(B, Hw, Ww, 1, Hc, Wc, 1)) return rc;
    MOG_REQUIRE(B == 0 || (U && theta && z_pres && gcanvas), MOG_ERR_NULL, "mog_stn_write_composite_backward: NULL pointer");
    if (!dU && !dtheta && !dz) return MOG_OK;
    BwdArgs a{};
    a.U = U; a.theta = theta; a.gout = gcanvas; a.dU = dU; a.dtheta = dtheta; a.z_pres = z_pres;
    a.stop_sum = stop_sum; a.dz = dz; a.threshold = threshold; a.Bsrc = B; a.u_div = 1;
    a.g = make_geo(Hw, Ww, 1, Hc, Wc);
    return launch_bwd<true>(a, SxyArgs{}, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------------
// The two sampler calls of an AIR step with theta built in the kernel from the model's (s, x, y)
// (air_number_bbox_location.py:511-542 read, :563-600 + :718-727 write): shift [B][2] = (x, y), scale [B] = s.
// The backward returns d_shift / d_scale directly; g_shift_in / g_scale_in (nullable) are added to them, so the gradient that
// reached the same (s, x, y) through the step's other call needs no accumulation kernel.
// ---------------------------------------------------------------------------------------------------
extern "C" int mog_stn_read_sxy_forward(const float* U, const float* shift, const float* scale, float* out, int64_t B, int Hs,
                                        int Ws, int Ho, int Wo, void* stream) {
    if (int rc = check_dims(B, Hs, Ws, 1, Ho, Wo, 1)) return rc;
    MOG_REQUIRE(B == 0 || (U && shift && scale && out), MOG_ERR_NULL, "mog_stn_read_sxy_forward: NULL pointer");
    FwdArgs a{};
    a.U = U; a.out = out; a.B = B; a.u_div = 1;
    a.g = make_geo(Hs, Ws, 1, Ho, Wo);
    const SxyArgs sx{shift, scale, nullptr, nullptr, nullptr, nullptr};
    return launch_fwd<false>(a, sx, (cudaStream_t)stream);
}

extern "C" int mog_stn_read_sxy_backward(const float* U, const float* shift, const float* scale, const float* gout,
                                         const float* g_shift_in, const float* g_scale_in, float* dU, float* d_shift,
                                         float* d_scale, int64_t B, int Hs, int Ws, int Ho, int Wo, void* stream) {
    if (int rc = check_dims(B, Hs, Ws, 1, Ho, Wo, 1)) return rc;
    MOG_REQUIRE(B == 0 || (U && shift && scale && gout && d_shift && d_scale), MOG_ERR_NULL, "mog_stn_read_sxy_backward: NULL pointer");
    BwdArgs a{};
    a.U = U; a.gout = gout; a.dU = dU; a.Bsrc = B; a.u_div = 1;
    a.g = make_geo(Hs, Ws, 1, Ho, Wo);
    const SxyArgs sx{shift, scale, g_shift_in, g_scale_in, d_shift, d_scale};
    return launch_bwd<false>(a, sx, (cudaStream_t)stream);
}

extern "C" int mog_stn_write_composite_sxy_forward(const float* U, const float* shift, const float* scale, const float* z_pres,
                                                   const float* stop_sum, float threshold, const float* canvas_in,
                                                   float* canvas_out, int64_t B, int Hw, int Ww, int Hc, int Wc, void* stream) {
    if (int rc = check_dims(B, Hw, Ww, 1, Hc, Wc, 1)) return rc;
    MOG_REQUIRE(B == 0 || (U && shift && scale && z_pres && canvas_in && canvas_out), MOG_ERR_NULL,
                "mog_stn_write_composite_sxy_forward: NULL pointer");
    FwdArgs a{};
    a.U = U; a.out = canvas_out; a.z_pres = z_pres; a.stop_sum = stop_sum;
    a.canvas_in = canvas_in; a.threshold = threshold; a.B = B; a.u_div = 1;
    a.g = make_geo(Hw, Ww, 1, Hc, Wc);
    const SxyArgs sx{shift, scale, nullptr, nullptr, nullptr, nullptr};
    return launch_fwd<true>(a, sx, (cudaStream_t)stream);
}

extern "C" int mog_stn_write_composite_sxy_backward(const float* U, const float* shift, const float* scale, const float* z_pres,
                                                    const float* stop_sum, float threshold, const float* gcanvas,
                                                    const float* g_shift_in, const float* g_scale_in, float* dU, float* d_shift,
                                                    float* d_scale, float* dz, int64_t B, int Hw, int Ww, int Hc, int Wc,
                                                    void* stream) {
    if (int rc = check_dims(B, Hw, Ww, 1, Hc, Wc, 1)) return rc;
    MOG_REQUIRE(B == 0 || (U && shift && scale && z_pres && gcanvas && d_shift && d_scale), MOG_ERR_NULL,
                "mog_stn_write_composite_sxy_backward: NULL pointer");
    BwdArgs a{};
    a.U = U; a.gout = gcanvas; a.dU = dU; a.z_pres = z_pres; a.stop_sum = stop_sum; a.dz = dz;
    a.threshold = threshold; a.Bsrc = B; a.u_div = 1;
    a.g = make_geo(Hw, Ww, 1, Hc, Wc);
    const SxyArgs sx{shift, scale, g_shift_in, g_scale_in, d_shift, d_scale};
    return launch_bwd<true>(a, sx, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------------
// host-buffer entry point (the end-to-end path): chunked H2D -> forward -> backward -> D2H on several streams
// ---------------------------------------------------------------------------------------------------
static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

struct HostChunkLayout {
    size_t U, theta, gout, out, dU, dtheta, total;
};

// chunk = source images per chunk; every source image carries T transforms (T outputs, T thetas, T upstream gradients)
static HostChunkLayout host_chunk_layout(int64_t chunk, int T, int Hs, int Ws, int C, int Ho, int Wo) {
    HostChunkLayout l;
    size_t o = 0;
    l.U = o;      o += align256((size_t)chunk * Hs * Ws * C * sizeof(float));
    l.theta = o;  o += align256((size_t)chunk * T * 6 * sizeof(float));
    l.gout = o;   o += align256((size_t)chunk * T * Ho * Wo * C * sizeof(float));
    l.out = o;    o += align256((size_t)chunk * T * Ho * Wo * C * sizeof(float));
    l.dU = o;     o += align256((size_t)chunk * Hs * Ws * C * sizeof(float));
    l.dtheta = o; o += align256((size_t)chunk * T * 6 * sizeof(float));
    l.total = o;
    return l;
}

extern "C" size_t mog_stn_batch_host_workspace_bytes(int64_t chunk, int T, int Hs, int Ws, int C, int Ho, int Wo, int nstreams) {
    if (chunk <= 0 || T <= 0 || Hs <= 0 || Ws <= 0 || C <= 0 || Ho <= 0 || Wo <= 0 || nstreams <= 0) return 0;
    return host_chunk_layout(chunk, T, Hs, Ws, C, Ho, Wo).total * (size_t)nstreams;
}

extern "C" size_t mog_stn_host_workspace_bytes(int64_t chunk, int Hs, int Ws, int C, int Ho, int Wo, int nstreams) {
    return mog_stn_batch_host_workspace_bytes(chunk, 1, Hs, Ws, C, Ho, Wo, nstreams);
}

#define MOG_CUDA_TRY(expr)                                                \
    do {                                                                  \
        cudaError_t e__ = (expr);                                         \
        if (e__ != cudaSuccess) {                                         \
            set_error("%s: %s", #expr, cudaGetErrorString(e__));          \
            return (int)e__;                                              \
        }                                                                 \
    } while (0)

// batch_transformer form (air/transformer.py:178-195) on host buffers: every source image is uploaded ONCE for its T
// transforms, dU is accumulated over them on the device and downloaded once (or not at all: the AIR read site asks for
// dtheta only, air_number_bbox_location.py:534-542).  Outputs are ordered like the reference's: index b*T + t.
extern "C" int mog_stn_batch_fwd_bwd_host(const float* U_h, const float* thetas_h, const float* gout_h, float* out_h, float* dU_h,
                                          float* dtheta_h, int64_t B, int T, int Hs, int Ws, int C, int Ho, int Wo, int64_t chunk,
                                          void* workspace_d, size_t workspace_bytes, void* const* streams, int nstreams) {
    MOG_REQUIRE(T >= 1, MOG_ERR_DIM, "batch_fwd_bwd_host: T=%d", T);
    if (int rc = check_dims(B * T, Hs, Ws, C, Ho, Wo, T)) return rc;
    MOG_REQUIRE(chunk > 0 && nstreams > 0 && nstreams <= 16, MOG_ERR_DIM, "batch_fwd_bwd_host: chunk=%lld nstreams=%d", (long long)chunk, nstreams);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(U_h && thetas_h && out_h && workspace_d && streams, MOG_ERR_NULL, "batch_fwd_bwd_host: NULL pointer");
    MOG_REQUIRE(gout_h || (!dU_h && !dtheta_h), MOG_ERR_NULL, "batch_fwd_bwd_host: gradients requested without gout");
    const HostChunkLayout l = host_chunk_layout(chunk, T, Hs, Ws, C, Ho, Wo);
    MOG_REQUIRE(workspace_bytes >= l.total * (size_t)nstreams, MOG_ERR_DIM, "batch_fwd_bwd_host: workspace %zu B < required %zu B",
                workspace_bytes, l.total * (size_t)nstreams);
    const size_t imU = (size_t)Hs * Ws * C, imO = (size_t)Ho * Wo * C;
    const Geo g = make_geo(Hs, Ws, C, Ho, Wo);
    int k = 0;
    for (int64_t b0 = 0; b0 < B; b0 += chunk, ++k) {
        const int64_t nb = (B - b0 < chunk) ? (B - b0) : chunk;
        cudaStream_t st = (cudaStream_t)streams[k % nstreams];
        char* base = (char*)workspace_d + l.total * (size_t)(k % nstreams);
        float* dUin = (float*)(base + l.U);
        float* dth = (float*)(base + l.theta);
        float* dgo = (float*)(base + l.gout);
        float* dout = (float*)(base + l.out);
        float* ddU = (float*)(base + l.dU);
        float* ddth = (float*)(base + l.dtheta);
        const bool bwd = dU_h || dtheta_h;
        MOG_CUDA_TRY(cudaMemcpyAsync(dUin, U_h + b0 * imU, nb * imU * sizeof(float), cudaMemcpyHostToDevice, st));
        MOG_CUDA_TRY(cudaMemcpyAsync(dth, thetas_h + b0 * T * 6, nb * T * 6 * sizeof(float), cudaMemcpyHostToDevice, st));
        if (bwd) MOG_CUDA_TRY(cudaMemcpyAsync(dgo, gout_h + b0 * T * imO, nb * T * imO * sizeof(float), cudaMemcpyHostToDevice, st));
        FwdArgs fa{};
        fa.U = dUin; fa.theta = dth; fa.out = dout; fa.B = nb * T; fa.u_div = T; fa.g = g;
        if (int rc = launch_fwd<false>(fa, SxyArgs{}, st)) return rc;
        MOG_CUDA_TRY(cudaMemcpyAsync(out_h + b0 * T * imO, dout, nb * T * imO * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (bwd) {
            BwdArgs ba{};
            ba.U = dUin; ba.theta = dth; ba.gout = dgo; ba.dU = dU_h ? ddU : nullptr; ba.dtheta = dtheta_h ? ddth : nullptr;
            ba.Bsrc = nb; ba.u_div = T; ba.g = g;
            if (int rc = launch_bwd<false>(ba, SxyArgs{}, st)) return rc;
            if (dU_h)
                MOG_CUDA_TRY(cudaMemcpyAsync(dU_h + b0 * imU, ddU, nb * imU * sizeof(float), cudaMemcpyDeviceToHost, st));
            if (dtheta_h)
                MOG_CUDA_TRY(cudaMemcpyAsync(dtheta_h + b0 * T * 6, ddth, nb * T * 6 * sizeof(float), cudaMemcpyDeviceToHost, st));
        }
    }
    const int used = k < nstreams ? k : nstreams;
    for (int i = 0; i < used; ++i) MOG_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)streams[i]));
    return MOG_OK;
}

extern "C" int mog_stn_fwd_bwd_host(const float* U_h, const float* theta_h, const float* gout_h, float* out_h, float* dU_h,
                                    float* dtheta_h, int64_t B, int Hs, int Ws, int C, int Ho, int Wo, int64_t chunk,
                                    void* workspace_d, size_t workspace_bytes, void* const* streams, int nstreams) {
    MOG_REQUIRE(B == 0 || gout_h, MOG_ERR_NULL, "fwd_bwd_host: NULL pointer");
    return mog_stn_batch_fwd_bwd_host(U_h, theta_h, gout_h, out_h, dU_h, dtheta_h, B, 1, Hs, Ws, C, Ho, Wo, chunk, workspace_d,
                                      workspace_bytes, streams, nstreams);
}

// ---------------------------------------------------------------------------------------------------
// The write call site of the AIR loop on host buffers (air_number_bbox_location.py:592-600 + :718-727): T windows per image
// are written onto ONE canvas per image,  canvas[b] = sum_t z[t][b] * sample(W[t][b]; theta[t][b]),  and the gradient of
// the canvas reaches every step's window, theta and z_pres.  Step-major layout ([T][B]...: the model's stacks), so a chunk
// of images is T contiguous pieces per array.  The canvas crosses PCIe once per image instead of once per glimpse.
// ---------------------------------------------------------------------------------------------------
struct CompositeChunkLayout {
    size_t W, theta, z, canvas, gcanvas, dW, dtheta, dz, total;
};

static CompositeChunkLayout composite_chunk_layout(int64_t chunk, int T, int Hw, int Ww, int Hc, int Wc) {
    CompositeChunkLayout l;
    size_t o = 0;
    l.W = o;       o += align256((size_t)chunk * T * Hw * Ww * sizeof(float));
    l.theta = o;   o += align256((size_t)chunk * T * 6 * sizeof(float));
    l.z = o;       o += align256((size_t)chunk * T * sizeof(float));
    l.canvas = o;  o += align256((size_t)chunk * Hc * Wc * sizeof(float));
    l.gcanvas = o; o += align256((size_t)chunk * Hc * Wc * sizeof(float));
    l.dW = o;      o += align256((size_t)chunk * T * Hw * Ww * sizeof(float));
    l.dtheta = o;  o += align256((size_t)chunk * T * 6 * sizeof(float));
    l.dz = o;      o += align256((size_t)chunk * T * sizeof(float));
    l.total = o;
    return l;
}

extern "C" size_t mog_stn_write_composite_host_workspace_bytes(int64_t chunk, int T, int Hw, int Ww, int Hc, int Wc, int nstreams) {
    if (chunk <= 0 || T <= 0 || Hw <= 0 || Ww <= 0 || Hc <= 0 || Wc <= 0 || nstreams <= 0) return 0;
    return composite_chunk_layout(chunk, T, Hw, Ww, Hc, Wc).total * (size_t)nstreams;
}

extern "C" int mog_stn_write_composite_host(const float* W_h, const float* thetas_h, const float* z_h, const float* gcanvas_h,
                                            float* canvas_h, float* dW_h, float* dtheta_h, float* dz_h, int64_t B, int T, int Hw,
                                            int Ww, int Hc, int Wc, int64_t chunk, void* workspace_d, size_t workspace_bytes,
                                            void* const* streams, int nstreams) {
    MOG_REQUIRE(T >= 1 && T <= 4096, MOG_ERR_DIM, "write_composite_host: T=%d", T);
    if (int rc = check_dims(B, Hw, Ww, 1, Hc, Wc, 1)) return rc;
    MOG_REQUIRE(chunk > 0 && nstreams > 0 && nstreams <= 16, MOG_ERR_DIM, "write_composite_host: chunk=%lld nstreams=%d", (long long)chunk, nstreams);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(W_h && thetas_h && z_h && canvas_h && workspace_d && streams, MOG_ERR_NULL, "write_composite_host: NULL pointer");
    const bool bwd = dW_h || dtheta_h || dz_h;
    MOG_REQUIRE(gcanvas_h || !bwd, MOG_ERR_NULL, "write_composite_host: gradients requested without gcanvas");
    const CompositeChunkLayout l = composite_chunk_layout(chunk, T, Hw, Ww, Hc, Wc);
    MOG_REQUIRE(workspace_bytes >= l.total * (size_t)nstreams, MOG_ERR_DIM, "write_composite_host: workspace %zu B < required %zu B",
                workspace_bytes, l.total * (size_t)nstreams);
    const size_t imW = (size_t)Hw * Ww, imC = (size_t)Hc * Wc;
    const Geo g = make_geo(Hw, Ww, 1, Hc, Wc);
    int k = 0;
    for (int64_t b0 = 0; b0 < B; b0 += chunk, ++k) {
        const int64_t nb = (B - b0 < chunk) ? (B - b0) : chunk;
        cudaStream_t st = (cudaStream_t)streams[k % nstreams];
        char* base = (char*)workspace_d + l.total * (size_t)(k % nstreams);
        float* dWin = (float*)(base + l.W);
        float* dth = (float*)(base + l.theta);
        float* dzp = (float*)(base + l.z);
        float* dcv = (float*)(base + l.canvas);
        float* dgc = (float*)(base + l.gcanvas);
        float* ddW = (float*)(base + l.dW);
        float* ddth = (float*)(base + l.dtheta);
        float* ddz = (float*)(base + l.dz);
        // device chunk layout is step-major too: step t of the chunk at offset t * nb
        for (int t = 0; t < T; ++t) {
            const size_t h = (size_t)t * B + b0, d = (size_t)t * nb;
            MOG_CUDA_TRY(cudaMemcpyAsync(dWin + d * imW, W_h + h * imW, nb * imW * sizeof(float), cudaMemcpyHostToDevice, st));
            MOG_CUDA_TRY(cudaMemcpyAsync(dth + d * 6, thetas_h + h * 6, nb * 6 * sizeof(float), cudaMemcpyHostToDevice, st));
            MOG_CUDA_TRY(cudaMemcpyAsync(dzp + d, z_h + h, nb * sizeof(float), cudaMemcpyHostToDevice, st));
        }
        if (bwd) MOG_CUDA_TRY(cudaMemcpyAsync(dgc, gcanvas_h + b0 * imC, nb * imC * sizeof(float), cudaMemcpyHostToDevice, st));
        MOG_CUDA_TRY(cudaMemsetAsync(dcv, 0, nb * imC * sizeof(float), st));
        for (int t = 0; t < T; ++t) {   // canvas += z_t * sample(W_t; theta_t), in place (only in-range rows are touched)
            const size_t d = (size_t)t * nb;
            FwdArgs fa{};
            fa.U = dWin + d * imW; fa.theta = dth + d * 6; fa.out = dcv; fa.z_pres = dzp + d; fa.stop_sum = nullptr;
            fa.canvas_in = dcv; fa.threshold = 0.0f; fa.B = nb; fa.u_div = 1; fa.g = g;
            if (int rc = launch_fwd<true>(fa, SxyArgs{}, st)) return rc;
        }
        MOG_CUDA_TRY(cudaMemcpyAsync(canvas_h + b0 * imC, dcv, nb * imC * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (bwd) {
            for (int t = 0; t < T; ++t) {
                const size_t d = (size_t)t * nb;
                BwdArgs ba{};
                ba.U = dWin + d * imW; ba.theta = dth + d * 6; ba.gout = dgc; ba.z_pres = dzp + d; ba.stop_sum = nullptr;
                ba.dU = dW_h ? ddW + d * imW : nullptr; ba.dtheta = dtheta_h ? ddth + d * 6 : nullptr; ba.dz = dz_h ? ddz + d : nullptr;
                ba.threshold = 0.0f; ba.Bsrc = nb; ba.u_div = 1; ba.g = g;
                if (int rc = launch_bwd<true>(ba, SxyArgs{}, st)) return rc;
            }
            for (int t = 0; t < T; ++t) {
                const size_t h = (size_t)t * B + b0, d = (size_t)t * nb;
                if (dW_h) MOG_CUDA_TRY(cudaMemcpyAsync(dW_h + h * imW, ddW + d * imW, nb * imW * sizeof(float), cudaMemcpyDeviceToHost, st));
                if (dtheta_h) MOG_CUDA_TRY(cudaMemcpyAsync(dtheta_h + h * 6, ddth + d * 6, nb * 6 * sizeof(float), cudaMemcpyDeviceToHost, st));
                if (dz_h) MOG_CUDA_TRY(cudaMemcpyAsync(dz_h + h, ddz + d, nb * sizeof(float), cudaMemcpyDeviceToHost, st));
            }
        }
    }
    const int used = k < nstreams ? k : nstreams;
    for (int i = 0; i < used; ++i) MOG_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)streams[i]));
    return MOG_OK;
}
