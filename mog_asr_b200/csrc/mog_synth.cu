// libmogstn -- object placement of the synthetic Multi-MNIST / Multi-dSprites generator.
//
// One placement loop (place_canvas, below) restates the reference's generate_multi_image; three kernels run it, each with
// the rule object of its overlap rule:
//   mode 0  the reference's bounding_boxes_overlap (multi_mnist.py:77-87) LITERALLY: two boxes clash when their
//           x-intervals (the new one widened by `gap`) intersect, whatever their rows; its second test can only fire for
//           degenerate boxes.
//   mode 1  true box intersection (x AND y intervals, widened by `gap`): a conservative stand-in for the pixel-overlap
//           rule (:53-57,:180-182) -- disjoint boxes never share a pixel.
//   pixels  the pixel-overlap rule itself (mog_synth_place_pixels, PixelRule below).
// Modes 0 and 1 run one thread per canvas (synth_place_kernel, BoxRule); the pixel rule runs one warp per canvas
// (synth_place_pixels_kernel).  Rotated objects labelled with their tight boxes, under any of the three rules, run one
// warp per canvas too (mog_synth_place_rotated, synth_place_rotated_kernel, RotatedRule).
// Randomness is a counter-based hash of (seed, canvas, restart, object, attempt, field) (CanvasDraws), so the oracles
// (oracle/synth_*_ref.py) reproduce every draw bit for bit and canvases do not depend on batch size or launch shape.
// The pixels are pasted afterwards with the sampler's own forward kernel (mog_asr_b200/dataset.py).
#include <algorithm>
#include <cmath>

#include "mog_common.cuh"

namespace mog {

__host__ __device__ inline uint32_t mix32(uint32_t x) {  // "lowbias32" finaliser
    x ^= x >> 16; x *= 0x7feb352dU;
    x ^= x >> 15; x *= 0x846ca68bU;
    x ^= x >> 16;
    return x;
}
// draw32(seed, canvas, restart, object, attempt, field) of the oracles and include/mogstn.h is
// draw32(canvas_key(seed, canvas), restart, object, attempt, field): the key is hashed once per canvas.
__host__ __device__ inline uint32_t canvas_key(uint32_t seed_lo, uint32_t seed_hi, uint32_t canvas) {
    uint32_t h = mix32(seed_lo ^ 0x9e3779b9U);
    h = mix32(h ^ seed_hi);
    return mix32(h ^ canvas);
}
__host__ __device__ inline uint32_t draw32(uint32_t key, uint32_t restart, uint32_t object, uint32_t attempt, uint32_t field) {
    const uint32_t h = mix32(key ^ (restart * 0x85ebca6bU + object));
    return mix32(h ^ (attempt * 0xc2b2ae35U + field));
}
// uniform integer in [lo, hi)  (hi > lo)
__host__ __device__ inline int draw_int(uint32_t h, int lo, int hi) { return lo + (int)(((uint64_t)h * (uint64_t)(hi - lo)) >> 32); }

struct SynthArgs {
    uint32_t seed_lo, seed_hi;
    long long B, first_canvas;
    const long long* first_dev;  // non-null: the first canvas index is read from device memory (the _dev entry points)
    int canvas, G, ncounts, size_min, size_max, gap, margin, mode, share_size, nsprites, max_restarts;
    int counts[MOG_SYNTH_MAX_COUNTS];
    int* num;
    int* pos;
    int* size;
    int* sprite;
};

__device__ __forceinline__ long long first_canvas(const SynthArgs& a) { return a.first_dev ? *a.first_dev : a.first_canvas; }

// The draws of one canvas, one method per drawn quantity; the draw fields are numbered here only.
struct CanvasDraws {
    const SynthArgs& a;
    uint32_t key;
    __device__ __forceinline__ CanvasDraws(const SynthArgs& a_, uint32_t cid) : a(a_), key(canvas_key(a_.seed_lo, a_.seed_hi, cid)) {}
    __device__ __forceinline__ uint32_t h(int restart, int i, int att, int field) const { return draw32(key, restart, i, att, field); }
    __device__ __forceinline__ int count() const { return a.counts[draw_int(h(0, 0, 0, 7), 0, a.ncounts)]; }
    // with share_size, every object of a restart takes the size drawn for object 0 (:119,:136-142)
    __device__ __forceinline__ int size(int restart, int i) const {
        return draw_int(h(restart, a.share_size ? 0 : i, 0, a.share_size ? 1 : 2), a.size_min, a.size_max + 1);
    }
    __device__ __forceinline__ int sprite(int restart, int i) const { return draw_int(h(restart, i, 0, 3), 0, a.nsprites); }
    __device__ __forceinline__ int angle(int restart, int i, int A) const { return draw_int(h(restart, i, 0, 6), 0, A); }
    // positions margin .. canvas - extent - margin (:171-172), `span` of them
    __device__ __forceinline__ int x(int restart, int i, int att, int span) const { return a.margin + draw_int(h(restart, i, att, 4), 0, span); }
    __device__ __forceinline__ int y(int restart, int i, int att, int span) const { return a.margin + draw_int(h(restart, i, att, 5), 0, span); }
};

// The reference's placement loop for one canvas (multi_mnist.py:110-221; the same in multi_dsprites.py:92-302): a count
// is drawn from the configured set; on every restart (:112-113) each object gets a size and a sprite, and a position is
// drawn inside the margins up to 100 times (:169) until it passes the overlap rule (:177-178) and is kept (:203-205);
// an object that cannot be placed starts the canvas over (:209-210).  When every restart fails, the objects of the last
// restart that did fit are kept, and the returned count says how many.  The rule supplies what differs:
//   restart()                 at the start of every restart
//   extent(d, r, i, w, sp)    takes the object's size and sprite; returns the side of the square its position is drawn for
//   fits(x, y, placed)        tries the object at (x, y) against the `placed` objects kept so far
//   accept(placed)            keeps the candidate fits() last passed as object `placed`
// The warp kernels run it on every lane: the draws depend only on the canvas, so its control flow is warp-uniform.
// Its exact form is measured (B200, tools/synth_bench.py): an `if (span > 0)` around the attempts compiles to a pixel rule
// 3-5 % slower, and a `break` out of the attempts to box rules 18 % to 5x slower.
template <class Rule>
__device__ __forceinline__ int place_canvas(const CanvasDraws& d, Rule& rule) {
    const SynthArgs& a = d.a;
    const int n = d.count();
    int placed = 0;
    for (int restart = 0; restart < a.max_restarts; ++restart) {
        placed = 0;
        rule.restart();
        bool ok = true;
        for (int i = 0; i < n && ok; ++i) {
            const int span = a.canvas - rule.extent(d, restart, i, d.size(restart, i), d.sprite(restart, i)) - 2 * a.margin + 1;
            bool found = false;
            for (int att = 0; span > 0 && att < 100 && !found; ++att)
                found = rule.fits(d.x(restart, i, att, span), d.y(restart, i, att, span), placed);
            if (found) {
                rule.accept(placed);
                ++placed;
            } else {
                ok = false;
            }
        }
        if (ok) break;
    }
    return placed;
}

// slot k of canvas b's labels: the box (x, y, w, h) and the sprite
__device__ __forceinline__ void store_label(const SynthArgs& a, long long b, int k, int4 box, int sprite) {
    const long long s = b * a.G + k;
    a.pos[2 * s] = box.x;
    a.pos[2 * s + 1] = box.y;
    a.size[2 * s] = box.z;
    a.size[2 * s + 1] = box.w;
    a.sprite[s] = sprite;
}

// the box rules on boxes (x, y, w, h), n the new one: bounding_boxes_overlap (:77-87) for mode 0, intersection for mode 1
__device__ __forceinline__ bool boxes_clash(int mode, int4 n, int4 q, int gap) {
    const int l1x = n.x - gap, l1y = n.y - gap, r1x = n.x + n.z + gap - 1, r1y = n.y + n.w + gap - 1;  // :79
    const int l2x = q.x, l2y = q.y, r2x = q.x + q.z - 1, r2y = q.y + q.w - 1;                          // :80
    const bool xhit = l1x <= r2x && l2x <= r1x;
    if (mode == 0) return xhit || (l1y >= r2y && l2y >= r1y);                                             // :82-85
    return xhit && l1y <= r2y && l2y <= r1y;
}

// (x, y, w, sprite) -> the square box (x, y, w, w)
__device__ __forceinline__ int4 square(int4 o) { return make_int4(o.x, o.y, o.z, o.z); }

// ---- modes 0 / 1 (mog_synth_place): one thread per canvas ------------------------------------------------------------
struct BoxRule {
    const SynthArgs& a;
    int4* obj;  // placed objects (x, y, w, sprite)
    int4 cand;  // the object being placed, at the position fits() last tried
    __device__ __forceinline__ BoxRule(const SynthArgs& a_, int4* obj_) : a(a_), obj(obj_) {}
    __device__ __forceinline__ void restart() {}
    __device__ __forceinline__ int extent(const CanvasDraws&, int, int, int w, int sp) {
        cand.z = w;
        cand.w = sp;
        return w;
    }
    __device__ __forceinline__ bool fits(int x, int y, int placed) {
        cand.x = x;
        cand.y = y;
        for (int k = 0; k < placed; ++k)
            if (boxes_clash(a.mode, square(cand), square(obj[k]), a.gap)) return false;
        return true;
    }
    __device__ __forceinline__ void accept(int placed) { obj[placed] = cand; }
};

__global__ void __launch_bounds__(128) synth_place_kernel(const SynthArgs a) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= a.B) return;
    int4 obj[MOG_SYNTH_MAX_OBJECTS];
    BoxRule rule(a, obj);
    const int placed = place_canvas(CanvasDraws(a, (uint32_t)(first_canvas(a) + b)), rule);
    a.num[b] = placed;
    for (int k = 0; k < a.G; ++k) {
        const int4 o = k < placed ? obj[k] : make_int4(0, 0, 0, 0);
        store_label(a, b, k, square(o), o.w);
    }
}

// ---- the warp kernels' shared pieces ---------------------------------------------------------------------------------
// One warp per canvas.  The occupancy of the objects placed so far, dilated by `gap` (Chebyshev), is a bitmap in shared
// memory: bit j of word j/32 of row i = canvas pixel (i, j).  A candidate's mask is kept in a second bitmap, so that an
// accepted candidate is OR-ed in without a second evaluation.
constexpr int kPixWarps = 4;                                       // canvases per CTA
constexpr int kPixRowWords = MOG_SYNTH_PIXEL_MAX_CANVAS / 32;      // bitmap words per canvas row
constexpr float kPixThreshold = 0.05f;                             // dataset.py drop threshold (:153-154)

// The value the sampler's forward writes at a pixel whose row axis is in range (transformer.py:112-116), in the forward's
// order (stn_fwd_warp_kernel, fwd_general_image): weights first, then add_n.  The pixel rule rests on its bit-equality
// with what the paste writes.
__device__ __forceinline__ float mask_value(const float* __restrict__ R0, const float* __restrict__ R1, const Axis& X, const Axis& Y) {
    const float wa = __fmul_rn(X.a, Y.a), wb = __fmul_rn(X.a, Y.b);
    const float wc = __fmul_rn(X.b, Y.a), wd = __fmul_rn(X.b, Y.b);
    float v = __fadd_rn(__fmul_rn(wa, __ldg(R0 + X.c0)), __fmul_rn(wb, __ldg(R1 + X.c0)));
    v = __fadd_rn(v, __fmul_rn(wc, __ldg(R0 + X.c1)));
    return __fadd_rn(v, __fmul_rn(wd, __ldg(R1 + X.c1)));
}

// OR rows lo..hi of the candidate's mask into the occupancy, dilated by `dil`: columns by shifts, in place (one lane per
// row) ...
__device__ __forceinline__ void occupy(uint32_t (*occ)[kPixRowWords], uint32_t (*cand)[kPixRowWords], int lo, int hi, int dil,
                                       int cs, int lane) {
    __syncwarp();
    for (int r = lo + lane; r <= hi; r += 32) {
        uint32_t m[kPixRowWords];
#pragma unroll
        for (int c = 0; c < kPixRowWords; ++c) m[c] = cand[r][c];
        for (int d = 0; d < dil; ++d) {
            uint32_t e[kPixRowWords];
#pragma unroll
            for (int c = 0; c < kPixRowWords; ++c)
                e[c] = m[c] | (m[c] << 1) | (m[c] >> 1) | (c > 0 ? m[c - 1] >> 31 : 0u) |
                       (c + 1 < kPixRowWords ? m[c + 1] << 31 : 0u);
#pragma unroll
            for (int c = 0; c < kPixRowWords; ++c) m[c] = e[c];
        }
#pragma unroll
        for (int c = 0; c < kPixRowWords; ++c) cand[r][c] = m[c];
    }
    __syncwarp();
    // ... then rows: occupancy row t takes the candidate rows within `dil` of it (one lane per row, no conflicts)
    for (int t = max(0, lo - dil) + lane; t <= min(cs - 1, hi + dil); t += 32) {
        uint32_t m[kPixRowWords] = {};
        for (int r = max(lo, t - dil); r <= min(hi, t + dil); ++r) {
#pragma unroll
            for (int c = 0; c < kPixRowWords; ++c) m[c] |= cand[r][c];
        }
#pragma unroll
        for (int c = 0; c < kPixRowWords; ++c) occ[t][c] |= m[c];
    }
}

// ---- pixel-overlap rule (mog_synth_place_pixels) ------------------------------------------------------------------
// The reference's rule for its non-"bbox" datasets (multi_mnist.py:53-57,:180-182): a position is rejected only when the
// new object's pixels touch pixels already on the canvas.  "Pixels" are those DeviceMultiObjectDataset.paste keeps: the
// sampler's write-direction forward of the sprite onto the canvas, >= the drop threshold 0.05 (:153-154).
//
// A candidate is evaluated row by row, lanes along canvas columns, with the forward kernel's own helpers and operation
// order (stn_fwd_warp_kernel, mog_stn_warp.cuh), so its values equal what the paste writes bit for bit; one ballot per
// 32 columns gives the row's mask, which is tested against the occupancy (exit on the first hit) and kept.
constexpr int kPixCtasPerSm = 8;  // resident CTAs per SM (63 registers, 16.5 KB shared each) and the grid cap: 32 canvases per SM per pass

struct PixelArgs {
    const float* sprites;     // [nsprites][side][side]
    const float* box_scale;   // [size_max + 1]: t00 = t11 of box_theta for size w
    const float* box_offset;  // [canvas][size_max + 1]: t02 (x) / t12 (y) of box_theta for position p, size w
    Geo g;                    // Hs = Ws = side, Ho = Wo = canvas, C = 1
};

struct PixelRule {
    const PixelArgs& p;
    uint32_t (*occ)[kPixRowWords];   // dilated occupancy
    uint32_t (*cand)[kPixRowWords];  // the candidate's mask
    int4* obj;                       // placed objects (x, y, w, sprite)
    int lane, cs, nw, ld, dil;
    const float* U;                  // the object being placed: sprite, size, theta scale
    int sp, w;
    float sc;
    int x, y, ilo, ihi;              // the candidate fits() last tried and its rows
    __device__ __forceinline__ PixelRule(const SynthArgs& a, const PixelArgs& p_, uint32_t (*occ_)[kPixRowWords],
                                         uint32_t (*cand_)[kPixRowWords], int4* obj_, int lane_)
        : p(p_), occ(occ_), cand(cand_), obj(obj_), lane(lane_), cs(p_.g.Wo), nw((p_.g.Wo + 31) >> 5), ld(a.size_max + 1),
          dil(min(a.gap, p_.g.Wo)) {}  // a wider dilation covers nothing more
    __device__ __forceinline__ void restart() {
        __syncwarp();
        for (int k = lane; k < cs * kPixRowWords; k += 32) occ[0][k] = 0u;
        __syncwarp();
    }
    __device__ __forceinline__ int extent(const CanvasDraws&, int, int, int w_, int sp_) {
        w = w_;
        sp = sp_;
        U = p.sprites + (long long)sp * p.g.S;
        sc = __ldg(p.box_scale + w);
        return w;
    }
    __device__ __forceinline__ bool fits(int x_, int y_, int) {
        const Geo& g = p.g;
        x = x_;
        y = y_;
        // theta of the paste: [[sc, 0, ox], [0, sc, oy]]
        const float ox = __ldg(p.box_offset + x * ld + w), oy = __ldg(p.box_offset + y * ld + w);
        // in-range rows (distinct row taps) form one interval [ilo, ihi]: the coordinate map is monotone.
        // The other rows are exactly +0 (DESIGN.md "borders").
        ilo = cs; ihi = -1;
        for (int i0 = 0; i0 < cs; i0 += 32) {
            bool in = false;
            if (i0 + lane < cs) {
                const Axis Y = axis_tap(affine_row(0.0f, sc, oy, 0.0f, lin_at(i0 + lane, g.step_h)), g.hsc, g.Hs);
                in = Y.c0 != Y.c1;
            }
            const unsigned m = __ballot_sync(0xffffffffu, in);
            if (m) {
                ilo = min(ilo, i0 + __ffs(m) - 1);
                ihi = i0 + 31 - __clz(m);
            }
        }
        // this lane's column taps; every column of an in-range row is evaluated, in range or not
        Axis X[kPixRowWords];
#pragma unroll
        for (int c = 0; c < kPixRowWords; ++c)
            X[c] = axis_tap(affine_row(sc, 0.0f, ox, lin_at(c * 32 + lane, g.step_w), 0.0f), g.wsc, g.Ws);
        bool hit = false;
        for (int r = ilo; r <= ihi && !hit; ++r) {
            const Axis Y = axis_tap(affine_row(0.0f, sc, oy, 0.0f, lin_at(r, g.step_h)), g.hsc, g.Hs);
            const float* __restrict__ R0 = U + Y.c0 * g.Ws;
            const float* __restrict__ R1 = U + Y.c1 * g.Ws;
            uint32_t mine = 0u;
#pragma unroll
            for (int c = 0; c < kPixRowWords; ++c) {
                if (c < nw) {
                    const float v = mask_value(R0, R1, X[c], Y);
                    const uint32_t m = __ballot_sync(0xffffffffu, c * 32 + lane < cs && v >= kPixThreshold);
                    if (lane == c) mine = m;
                    hit |= (m & occ[r][c]) != 0u;
                }
            }
            if (lane < kPixRowWords) cand[r][lane] = mine;
        }
        return !hit;
    }
    __device__ __forceinline__ void accept(int placed) {
        occupy(occ, cand, ilo, ihi, dil, cs, lane);
        if (lane == 0) obj[placed] = make_int4(x, y, w, sp);
        __syncwarp();
    }
};

__global__ void __launch_bounds__(kPixWarps * 32, kPixCtasPerSm) synth_place_pixels_kernel(const SynthArgs a, const PixelArgs p) {
    __shared__ uint32_t s_occ[kPixWarps][MOG_SYNTH_PIXEL_MAX_CANVAS][kPixRowWords];
    __shared__ uint32_t s_cand[kPixWarps][MOG_SYNTH_PIXEL_MAX_CANVAS][kPixRowWords];
    __shared__ int4 s_obj[kPixWarps][MOG_SYNTH_MAX_OBJECTS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int4* obj = s_obj[warp];
    PixelRule rule(a, p, s_occ[warp], s_cand[warp], s_obj[warp], lane);
    const long long first = first_canvas(a);

    for (long long b = (long long)blockIdx.x * kPixWarps + warp; b < a.B; b += (long long)gridDim.x * kPixWarps) {
        const int placed = place_canvas(CanvasDraws(a, (uint32_t)(first + b)), rule);
        __syncwarp();
        if (lane == 0) a.num[b] = placed;
        for (int k = lane; k < a.G; k += 32) {
            const int4 o = k < placed ? obj[k] : make_int4(0, 0, 0, 0);
            store_label(a, b, k, square(o), o.w);
        }
    }
}

// ---- rotated objects, tight-box labels (mog_synth_place_rotated) ---------------------------------------------------
// The reference rotates every object and re-crops it to its tight box, which becomes its label (multi_mnist.py:144-163).
// Here an object of size w at angle (cos, sin) from the caller's table owns the square of side
// e = min(canvas, ceil(w (|cos| + |sin|))) that holds the rotated w-square; the position is drawn for that e-square and
// the paste theta (include/mogstn.h, rotated_theta below) rotates the sprite about the e-square's centre.  The angle is
// redrawn on every restart, like the size.
//
// A candidate is evaluated over its e-square widened by one pixel (clipped to the canvas) with taps_general and the
// add_n order of fwd_general_image, so each value is what mog_stn_forward writes for that theta; lanes run along
// 32-column words aligned to the occupancy bitmap.  The row and column extents of the mask (value >= 0.05) give the
// tight box.  Mode 2 tests the mask against the dilated occupancy (exit on the first hit); modes 0 / 1 test the tight
// box, widened by `gap`, with the box rules.  An object whose mask is empty (a blank sprite) clashes with nothing and is
// labelled with its e-square.
//
// Why no pixel outside the evaluated region reaches 0.05.  Let (u, v) be a pixel's offset in canvas pixels from the
// e-square's centre, R = (w - 1) / 2 and Ws = sprite side.  Up to fp32 rounding the paste maps it to the source
// x_s = (cos u + sin v) / R, y_s = (-sin u + cos v) / R.  axis_tap gives distinct corners (an in-range axis) only for
// 0 <= p < Ws - 1 with p = (s + 1)(Ws - 1.001) / 2, i.e. for -1 <= s < 1 + d with d = 0.002 / (Ws - 1.001) (Ws >= 2; for
// Ws = 1 no axis is ever in range).  With the row axis out of range the forward writes exactly +0 (DESIGN.md "borders").
// With the column axis out of range its two weights are exact negatives (a = c - p, b = p - c), so the add_n sum is
// (P + Q) - P - Q with |P| + |Q| <= |c - p| max|U|: at most 2 ulp of that, i.e. below 2^-22 |c - p| max|U|.  Here
// R >= 1/2 and |u|, |v| <= 127 give |x_s| <= 2 sqrt(2) 127 and |c - p| < 200 Ws, so for sprites in [0, 1] of side below
// 1000 this stays under 0.05.  A pixel whose two axes are in range has |cos u + sin v| and |-sin u + cos v| <= R (1 + d),
// hence |u|, |v| <= R (1 + d)(|cos| + |sin|) <= (e - 1) / 2 + (1 - (|cos| + |sin|)) / 2 + sqrt(2) R d < (e - 1) / 2 + 0.2
// (w (|cos| + |sin|) <= e, R <= 63.5, d <= 0.002), so it lies in the e-square itself (the offsets of its pixels are
// those of a grid of step 1 with |u| <= (e - 1) / 2) with 0.8 pixel to spare for the fp32 rounding of theta and of the
// coordinate map (far below 0.01 pixel).  When e is clamped to the canvas the e-square is the canvas.  The widening by
// one pixel is a second margin; tests/test_dataset_rotated.py checks the region against full-canvas forwards.
constexpr int kRotCtasPerSm = 8;  // grid cap, as kPixCtasPerSm

struct RotArgs {
    const float* sprites;  // [nsprites][side][side]
    float* theta;          // [B][G][6] paste theta of every placed object
    Geo g;                 // Hs = Ws = side, Ho = Wo = canvas, C = 1
    int A;
    double rot[MOG_SYNTH_MAX_ANGLES][2];  // (cos, sin)
};

// include/mogstn.h's theta, fp64 with explicit _rn operations (no FMA contraction), each entry rounded to fp32 once.
// (0 - s) and -(c cy - s cx) rather than -s and s cx - c cy: for (c, s) = (1, +0) every entry, signed zeros included,
// is then box_theta's.
__device__ __forceinline__ void rotated_theta(double c, double s, int w, int e, int x, int y, int cs, Theta& th) {
    const double d = (double)(cs - 1);
    const double sc = __ddiv_rn((double)(w - 1), d);
    const double cx = __dadd_rn(-1.0, __ddiv_rn(__dsub_rn(__dadd_rn(2.0 * x, (double)e), 1.0), d));
    const double cy = __dadd_rn(-1.0, __ddiv_rn(__dsub_rn(__dadd_rn(2.0 * y, (double)e), 1.0), d));
    th.t[0] = (float)__ddiv_rn(c, sc);
    th.t[1] = (float)__ddiv_rn(s, sc);
    th.t[2] = (float)__ddiv_rn(-__dadd_rn(__dmul_rn(c, cx), __dmul_rn(s, cy)), sc);
    th.t[3] = (float)__ddiv_rn(__dsub_rn(0.0, s), sc);
    th.t[4] = (float)__ddiv_rn(c, sc);
    th.t[5] = (float)__ddiv_rn(-__dsub_rn(__dmul_rn(c, cy), __dmul_rn(s, cx)), sc);
}

struct RotatedRule {
    const SynthArgs& a;
    const RotArgs& p;
    uint32_t (*occ)[kPixRowWords];   // dilated occupancy (mode 2)
    uint32_t (*cand)[kPixRowWords];  // the candidate's mask (mode 2)
    int4* box;                       // labels (x, y, w, h)
    int2* obj;                       // (sprite, mask empty)
    float* oth;                      // paste thetas
    int lane, cs, dil;
    bool pix;
    const float* U;                  // the object being placed: sprite, size, angle, extent
    int sp, w, e;
    double co, si;
    int4 lab;                        // the candidate fits() last tried: tight box, mask rows, theta
    int rmin, rmax;
    Theta th;
    __device__ __forceinline__ RotatedRule(const SynthArgs& a_, const RotArgs& p_, uint32_t (*occ_)[kPixRowWords],
                                           uint32_t (*cand_)[kPixRowWords], int4* box_, int2* obj_, float* oth_, int lane_)
        : a(a_), p(p_), occ(occ_), cand(cand_), box(box_), obj(obj_), oth(oth_), lane(lane_), cs(p_.g.Wo),
          dil(min(a_.gap, p_.g.Wo)), pix(a_.mode == 2) {}
    __device__ __forceinline__ void restart() {
        if (pix) {
            __syncwarp();
            for (int k = lane; k < cs * kPixRowWords; k += 32) occ[0][k] = 0u;
            __syncwarp();
        }
    }
    __device__ __forceinline__ int extent(const CanvasDraws& d, int restart, int i, int w_, int sp_) {
        w = w_;
        sp = sp_;
        const int k = d.angle(restart, i, p.A);
        co = p.rot[k][0];
        si = p.rot[k][1];
        e = min(cs, (int)ceil(__dmul_rn((double)w, __dadd_rn(fabs(co), fabs(si)))));
        U = p.sprites + (long long)sp * p.g.S;
        return e;
    }
    __device__ __forceinline__ bool fits(int x, int y, int placed) {
        const Geo& g = p.g;
        rotated_theta(co, si, w, e, x, y, cs, th);
        // the evaluated region: the e-square widened by one pixel, clipped to the canvas
        const int r_lo = max(0, y - 1), r_hi = min(cs - 1, y + e), c_lo = max(0, x - 1), c_hi = min(cs - 1, x + e);
        uint32_t cols = 0u;  // lane c < kPixRowWords: OR of the mask's word c over the rows
        rmin = cs; rmax = -1;
        bool hit = false;
        for (int r = r_lo; r <= r_hi && !hit; ++r) {
            uint32_t mine = 0u;
#pragma unroll
            for (int c = 0; c < kPixRowWords; ++c) {
                if (c * 32 <= c_hi && c * 32 + 31 >= c_lo) {
                    const int j = c * 32 + lane;
                    bool on = false;
                    if (j >= c_lo && j <= c_hi) {
                        Axis X, Y;
                        taps_general(th, g, r, j, X, Y);
                        if (Y.c0 != Y.c1)  // else the forward writes exactly +0
                            on = mask_value(U + Y.c0 * g.Ws, U + Y.c1 * g.Ws, X, Y) >= kPixThreshold;
                    }
                    const uint32_t m = __ballot_sync(0xffffffffu, on);
                    if (lane == c) mine = m;
                    if (m) {
                        rmin = min(rmin, r);
                        rmax = r;
                    }
                    if (pix) hit |= (m & occ[r][c]) != 0u;
                }
            }
            if (pix && lane < kPixRowWords) cand[r][lane] = mine;
            cols |= mine;
        }
        if (hit) return false;
        if (rmax < 0) {  // empty mask: no clash, labelled with the e-square
            lab = make_int4(x, y, e, e);
            return true;
        }
        int cmin = cs, cmax = -1;
#pragma unroll
        for (int c = 0; c < kPixRowWords; ++c) {
            const uint32_t m = __shfl_sync(0xffffffffu, cols, c);
            if (m) {
                cmin = min(cmin, c * 32 + __ffs(m) - 1);
                cmax = c * 32 + 31 - __clz(m);
            }
        }
        lab = make_int4(cmin, rmin, cmax - cmin + 1, rmax - rmin + 1);
        if (!pix)
            for (int q = 0; q < placed; ++q)
                if (!obj[q].y && boxes_clash(a.mode, lab, box[q], a.gap)) return false;
        return true;
    }
    __device__ __forceinline__ void accept(int placed) {
        if (pix && rmax >= 0) occupy(occ, cand, rmin, rmax, dil, cs, lane);
        if (lane == 0) {
            box[placed] = lab;
            obj[placed] = make_int2(sp, rmax < 0 ? 1 : 0);
#pragma unroll
            for (int q = 0; q < 6; ++q) oth[placed * 6 + q] = th.t[q];
        }
        __syncwarp();
    }
};

__global__ void __launch_bounds__(kPixWarps * 32, kRotCtasPerSm) synth_place_rotated_kernel(const SynthArgs a, const RotArgs p) {
    __shared__ uint32_t s_occ[kPixWarps][MOG_SYNTH_PIXEL_MAX_CANVAS][kPixRowWords];
    __shared__ uint32_t s_cand[kPixWarps][MOG_SYNTH_PIXEL_MAX_CANVAS][kPixRowWords];
    __shared__ int4 s_box[kPixWarps][MOG_SYNTH_MAX_OBJECTS];
    __shared__ int2 s_obj[kPixWarps][MOG_SYNTH_MAX_OBJECTS];
    __shared__ float s_th[kPixWarps][MOG_SYNTH_MAX_OBJECTS * 6];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int4* box = s_box[warp];
    const int2* obj = s_obj[warp];
    const float* oth = s_th[warp];
    RotatedRule rule(a, p, s_occ[warp], s_cand[warp], s_box[warp], s_obj[warp], s_th[warp], lane);
    const long long first = first_canvas(a);

    for (long long b = (long long)blockIdx.x * kPixWarps + warp; b < a.B; b += (long long)gridDim.x * kPixWarps) {
        const int placed = place_canvas(CanvasDraws(a, (uint32_t)(first + b)), rule);
        __syncwarp();
        if (lane == 0) a.num[b] = placed;
        for (int k = lane; k < a.G; k += 32) {
            const bool v = k < placed;
            store_label(a, b, k, v ? box[k] : make_int4(0, 0, 0, 0), v ? obj[k].x : 0);
        }
        for (int q = lane; q < a.G * 6; q += 32) p.theta[b * a.G * 6 + q] = q < placed * 6 ? oth[q] : 0.0f;
    }
}

}  // namespace mog

// The checks and SynthArgs fields every placement entry point shares; `what` names the entry point in the messages.
// For B == 0 only the ranges are checked (the call is then a no-op whatever the pointers) and `a` is left as it is.
static int synth_args(const char* what, uint64_t seed, int64_t first_canvas, bool dev, const int64_t* first_dev, int64_t B, int canvas,
                      int max_objects, const int* counts, int num_counts, int size_min, int size_max, int gap, int margin,
                      int share_size, int num_sprites, int* num, int* pos, int* size, int* sprite, mog::SynthArgs& a) {
    MOG_REQUIRE(B >= 0 && canvas > 0 && max_objects > 0 && max_objects <= MOG_SYNTH_MAX_OBJECTS && num_counts > 0 &&
                    num_counts <= MOG_SYNTH_MAX_COUNTS && size_min > 0 && size_max >= size_min && gap >= 0 && margin >= 0 &&
                    num_sprites > 0 && (dev || first_canvas >= 0),
                MOG_ERR_DIM, "%s: B=%lld canvas=%d max_objects=%d num_counts=%d size=[%d,%d] gap=%d margin=%d sprites=%d", what,
                (long long)B, canvas, max_objects, num_counts, size_min, size_max, gap, margin, num_sprites);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(counts && num && pos && size && sprite && (!dev || first_dev), MOG_ERR_NULL, "%s: NULL pointer", what);
    for (int k = 0; k < num_counts; ++k) {
        MOG_REQUIRE(counts[k] >= 0 && counts[k] <= max_objects, MOG_ERR_DIM, "%s: counts[%d]=%d exceeds max_objects=%d", what, k,
                    counts[k], max_objects);
        a.counts[k] = counts[k];
    }
    a.seed_lo = (uint32_t)seed; a.seed_hi = (uint32_t)(seed >> 32);
    a.B = B; a.first_canvas = first_canvas; a.first_dev = (const long long*)first_dev; a.canvas = canvas; a.G = max_objects; a.ncounts = num_counts;
    a.size_min = size_min; a.size_max = size_max; a.gap = gap; a.margin = margin; a.share_size = share_size ? 1 : 0;
    a.nsprites = num_sprites; a.max_restarts = MOG_SYNTH_MAX_RESTARTS;
    a.num = num; a.pos = pos; a.size = size; a.sprite = sprite;
    return MOG_OK;
}

static int synth_place(uint64_t seed, int64_t first_canvas, bool dev, const int64_t* first_dev, int64_t B, int canvas, int max_objects, const int* counts,
                               int num_counts, int size_min, int size_max, int gap, int margin, int mode, int share_size,
                               int num_sprites, int* num, int* pos, int* size, int* sprite, void* stream) {
    using namespace mog;
    SynthArgs a{};
    if (const int rc = synth_args("synth_place", seed, first_canvas, dev, first_dev, B, canvas, max_objects, counts, num_counts, size_min,
                                  size_max, gap, margin, share_size, num_sprites, num, pos, size, sprite, a))
        return rc;
    MOG_REQUIRE(mode == 0 || mode == 1, MOG_ERR_DIM, "synth_place: mode=%d", mode);
    if (B == 0) return MOG_OK;
    a.mode = mode;
    synth_place_kernel<<<(unsigned)((B + 127) / 128), 128, 0, (cudaStream_t)stream>>>(a);
    MOG_CUDA_LAUNCH_CHECK("synth_place_kernel");
    return MOG_OK;
}

static int synth_place_pixels(uint64_t seed, int64_t first_canvas, bool dev, const int64_t* first_dev, int64_t B, int canvas, int max_objects, const int* counts,
                                      int num_counts, int size_min, int size_max, int gap, int margin, int share_size,
                                      const float* sprites, int num_sprites, int sprite_side, const float* box_scale,
                                      const float* box_offset, int* num, int* pos, int* size, int* sprite, void* stream) {
    using namespace mog;
    SynthArgs a{};
    if (const int rc = synth_args("synth_place_pixels", seed, first_canvas, dev, first_dev, B, canvas, max_objects, counts, num_counts,
                                  size_min, size_max, gap, margin, share_size, num_sprites, num, pos, size, sprite, a))
        return rc;
    MOG_REQUIRE(sprite_side > 0, MOG_ERR_DIM, "synth_place_pixels: side=%d", sprite_side);
    MOG_REQUIRE(canvas <= MOG_SYNTH_PIXEL_MAX_CANVAS, MOG_ERR_UNSUPPORTED, "synth_place_pixels: canvas=%d > %d", canvas,
                MOG_SYNTH_PIXEL_MAX_CANVAS);
    MOG_REQUIRE((long long)sprite_side * sprite_side * num_sprites < (1LL << 31), MOG_ERR_OVERFLOW,
                "synth_place_pixels: %d sprites of %dx%d exceed int32 indexing", num_sprites, sprite_side, sprite_side);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(sprites && box_scale && box_offset, MOG_ERR_NULL, "synth_place_pixels: NULL pointer");
    PixelArgs p{};
    p.sprites = sprites; p.box_scale = box_scale; p.box_offset = box_offset;
    p.g = make_geo(sprite_side, sprite_side, 1, canvas, canvas);
    const long long blocks = std::min<long long>((B + kPixWarps - 1) / kPixWarps, (long long)sm_count() * kPixCtasPerSm);
    synth_place_pixels_kernel<<<(unsigned)blocks, kPixWarps * 32, 0, (cudaStream_t)stream>>>(a, p);
    MOG_CUDA_LAUNCH_CHECK("synth_place_pixels_kernel");
    return MOG_OK;
}

static int synth_place_rotated(uint64_t seed, int64_t first_canvas, bool dev, const int64_t* first_dev, int64_t B, int canvas, int max_objects, const int* counts,
                                       int num_counts, int size_min, int size_max, int gap, int margin, int mode, int share_size,
                                       const float* sprites, int num_sprites, int sprite_side, const double* rot, int num_angles,
                                       int* num, int* pos, int* size, int* sprite, float* theta, void* stream) {
    using namespace mog;
    SynthArgs a{};
    if (const int rc = synth_args("synth_place_rotated", seed, first_canvas, dev, first_dev, B, canvas, max_objects, counts, num_counts,
                                  size_min, size_max, gap, margin, share_size, num_sprites, num, pos, size, sprite, a))
        return rc;
    // a size-1 object has no finite theta
    MOG_REQUIRE(canvas > 1 && size_min > 1 && (mode == 0 || mode == 1 || mode == 2) && sprite_side > 0 && num_angles > 0 &&
                    num_angles <= MOG_SYNTH_MAX_ANGLES,
                MOG_ERR_DIM, "synth_place_rotated: canvas=%d size_min=%d mode=%d side=%d angles=%d", canvas, size_min, mode,
                sprite_side, num_angles);
    MOG_REQUIRE(canvas <= MOG_SYNTH_PIXEL_MAX_CANVAS, MOG_ERR_UNSUPPORTED, "synth_place_rotated: canvas=%d > %d", canvas,
                MOG_SYNTH_PIXEL_MAX_CANVAS);
    MOG_REQUIRE((long long)sprite_side * sprite_side * num_sprites < (1LL << 31), MOG_ERR_OVERFLOW,
                "synth_place_rotated: %d sprites of %dx%d exceed int32 indexing", num_sprites, sprite_side, sprite_side);
    if (B == 0) return MOG_OK;
    MOG_REQUIRE(sprites && rot && theta, MOG_ERR_NULL, "synth_place_rotated: NULL pointer");
    a.mode = mode;
    RotArgs p{};
    p.sprites = sprites; p.theta = theta; p.A = num_angles;
    p.g = make_geo(sprite_side, sprite_side, 1, canvas, canvas);
    for (int k = 0; k < num_angles; ++k) {
        const double c = rot[2 * k], s = rot[2 * k + 1];
        // a rotation: the extent e and the bound on the evaluated region (synth_place_rotated_kernel) rest on it
        MOG_REQUIRE(std::isfinite(c) && std::isfinite(s) && std::fabs(c * c + s * s - 1.0) <= 1e-9, MOG_ERR_DIM,
                    "synth_place_rotated: rot[%d] = (%g, %g) is not a unit (cos, sin) pair", k, c, s);
        p.rot[k][0] = c; p.rot[k][1] = s;
    }
    const long long blocks = std::min<long long>((B + kPixWarps - 1) / kPixWarps, (long long)sm_count() * kRotCtasPerSm);
    synth_place_rotated_kernel<<<(unsigned)blocks, kPixWarps * 32, 0, (cudaStream_t)stream>>>(a, p);
    MOG_CUDA_LAUNCH_CHECK("synth_place_rotated_kernel");
    return MOG_OK;
}

// The host-index entry points and their _dev twins (first canvas index read from device memory by the kernel, so that a
// captured CUDA graph can advance it between replays) share one launcher each.
extern "C" int mog_synth_place(uint64_t seed, int64_t first_canvas, int64_t B, int canvas, int max_objects, const int* counts,
                               int num_counts, int size_min, int size_max, int gap, int margin, int mode, int share_size,
                               int num_sprites, int* num, int* pos, int* size, int* sprite, void* stream) {
    return synth_place(seed, first_canvas, false, nullptr, B, canvas, max_objects, counts, num_counts, size_min, size_max, gap, margin,
                       mode, share_size, num_sprites, num, pos, size, sprite, stream);
}

extern "C" int mog_synth_place_dev(uint64_t seed, const int64_t* first_canvas, int64_t B, int canvas, int max_objects,
                                   const int* counts, int num_counts, int size_min, int size_max, int gap, int margin, int mode,
                                   int share_size, int num_sprites, int* num, int* pos, int* size, int* sprite, void* stream) {
    return synth_place(seed, 0, true, first_canvas, B, canvas, max_objects, counts, num_counts, size_min, size_max, gap, margin, mode,
                       share_size, num_sprites, num, pos, size, sprite, stream);
}

extern "C" int mog_synth_place_pixels(uint64_t seed, int64_t first_canvas, int64_t B, int canvas, int max_objects, const int* counts,
                                      int num_counts, int size_min, int size_max, int gap, int margin, int share_size,
                                      const float* sprites, int num_sprites, int sprite_side, const float* box_scale,
                                      const float* box_offset, int* num, int* pos, int* size, int* sprite, void* stream) {
    return synth_place_pixels(seed, first_canvas, false, nullptr, B, canvas, max_objects, counts, num_counts, size_min, size_max, gap,
                              margin, share_size, sprites, num_sprites, sprite_side, box_scale, box_offset, num, pos, size, sprite,
                              stream);
}

extern "C" int mog_synth_place_pixels_dev(uint64_t seed, const int64_t* first_canvas, int64_t B, int canvas, int max_objects,
                                          const int* counts, int num_counts, int size_min, int size_max, int gap, int margin,
                                          int share_size, const float* sprites, int num_sprites, int sprite_side,
                                          const float* box_scale, const float* box_offset, int* num, int* pos, int* size,
                                          int* sprite, void* stream) {
    return synth_place_pixels(seed, 0, true, first_canvas, B, canvas, max_objects, counts, num_counts, size_min, size_max, gap, margin,
                              share_size, sprites, num_sprites, sprite_side, box_scale, box_offset, num, pos, size, sprite, stream);
}

extern "C" int mog_synth_place_rotated(uint64_t seed, int64_t first_canvas, int64_t B, int canvas, int max_objects, const int* counts,
                                       int num_counts, int size_min, int size_max, int gap, int margin, int mode, int share_size,
                                       const float* sprites, int num_sprites, int sprite_side, const double* rot, int num_angles,
                                       int* num, int* pos, int* size, int* sprite, float* theta, void* stream) {
    return synth_place_rotated(seed, first_canvas, false, nullptr, B, canvas, max_objects, counts, num_counts, size_min, size_max, gap,
                               margin, mode, share_size, sprites, num_sprites, sprite_side, rot, num_angles, num, pos, size, sprite,
                               theta, stream);
}

extern "C" int mog_synth_place_rotated_dev(uint64_t seed, const int64_t* first_canvas, int64_t B, int canvas, int max_objects,
                                           const int* counts, int num_counts, int size_min, int size_max, int gap, int margin,
                                           int mode, int share_size, const float* sprites, int num_sprites, int sprite_side,
                                           const double* rot, int num_angles, int* num, int* pos, int* size, int* sprite,
                                           float* theta, void* stream) {
    return synth_place_rotated(seed, 0, true, first_canvas, B, canvas, max_objects, counts, num_counts, size_min, size_max, gap, margin,
                               mode, share_size, sprites, num_sprites, sprite_side, rot, num_angles, num, pos, size, sprite, theta,
                               stream);
}
