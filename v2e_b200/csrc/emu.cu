// DVS pixel model for sm_100a -- hand-written CUDA behind the C ABI in include/v2e_b200.h.
//
// Replaces (reference = SensorsINI/v2e, /root/reference):
//   v2ecore/emulator.py:619-1022  EventEmulator.generate_events
//   v2ecore/emulator_utils.py:18-173, 297-351  lin_log, rescale_intensity_frame, low_pass_filter,
//       subtract_leak_current, compute_event_map, generate_shot_noise
//
// Per frame the reference launches ~40 eager ops + one D2H sync per emitted-event iteration. Here a
// frame is at most three streaming kernels, all on the caller's stream, no host sync:
//   update : frame + per-pixel state -> new state, signed event count per pixel (int16 record),
//            global max (atomicMax), per-(iteration,polarity) histogram
//   filter : only when refractory_period_s > 0: replays the refractory filter on active pixels to
//            get the filtered histogram
//   emit   : active pixels only: block-aggregated compaction into the packed [N][4] float32 rows,
//            base / timestamp_mem patch
// The "plan" (segment offsets of the iteration-major output, running row offset, capacity check)
// is computed by the last block to finish the last counting kernel of the frame.
//
// Arithmetic is bit-compatible with the reference's CPU path: float64 where torch promotes to
// float64, float32 products where a Python scalar meets a float32 tensor, ATen's floor-division
// and linspace formulas. This TU must be compiled with -fmad=false; the only fused multiply-adds
// are the explicit fmaf() in linspace_f32().
#include <cuda_runtime.h>
#include <cooperative_groups.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

#include "../../include/v2e_b200.h"
#include "common.cuh"
#include "tc_common.cuh"   // mbarrier helpers (the update kernel stages its state with TMA bulk copies)

namespace {

constexpr int kThreads = 256;
constexpr int kVec = 4;                 // pixels per thread
constexpr int kSegSmem = 64;            // (iteration,polarity) segments aggregated in shared memory
constexpr int kRecShift = 2;            // record = (signed count << 2) | shot_off << 1 | shot_on
constexpr int kRecMaxCount = 8191;
constexpr int kPhiloxRounds = 7;         // Philox4x32-7: the lightest variant that passes BigCrush (Salmon et al. 2011)

struct FrameCtrl {                      // one per frame slot, device memory, zeroed per step
    int32_t max_n;
    int32_t filter_active;
    uint32_t done[3];                   // last-block tickets: update, filter, shot
    uint32_t n_on, n_off, n_shot_on, n_shot_off, n_events;
    int32_t cs_steps;
    int32_t planned;
    uint64_t ev_base;
    uint64_t pad;
};
static_assert(sizeof(FrameCtrl) == 64, "FrameCtrl layout");

struct EmuDev {                         // passed by value to every kernel
    int32_t n, W, H, n_pad;
    int32_t per_pixel_thres, hdr, state_f64, csdvs;
    int32_t leak_on, lowpass_on, shot_on, refr_on;
    int32_t rng_mode, iter_cap, seg_stride, max_slots;
    double pos_nom, neg_nom;
    float leak_rate_f, leak_jit_f, refr_f, pad0;
    double refr_d, shot_inten_m1;       // refractory_period_s ; (SHOT_NOISE_INTEN_FACTOR-1)
    uint64_t seed;
    void *lp, *base;
    void *lp_out, *base_out;            // where the update kernel stores lp / base: the same arrays, except while
                                        // v2e_emu_time_update replays one frame out of place
    float *pos_thres, *neg_thres, *noise_rate, *tmem;
    double *surround;                   // CSDVS h, ping buffer (cs_cur == 0)
    double *surround2;                  // pong buffer
    int32_t *cs_cur;                    // which buffer holds the current surround
    unsigned long long *cs_max;         // [cs_cap] max|change| of every Euler step of the current frame (double bits)
    int32_t cs_cap, cs_seq_order;
    int32_t cs_ring;                    // buffers in the surround ring (2 unless pixel-sharded: steps per chunk + 1)
    int32_t cs_y_lo, cs_y_hi;           // rows of this handle that count for max|change| (the rank's own rows)
    int32_t own_lo, own_hi;             // pixels [own_lo, own_hi) emit events (a sharded centre-surround handle also
                                        // carries halo rows above / below its own rows); 0 / n otherwise
    int32_t *cs_done;                   // sharded: the Euler iteration of this frame ended in an earlier chunk
    double *cs_bufs;                    // sharded: ring of cs_ring buffers of cs_stride doubles (replaces surround / surround2)
    size_t cs_stride;
    int16_t *rec;
    uint32_t *act_list;                 // [n_pad] pixel indices with a non-zero record (built by the update kernel)
    uint32_t *act_count;                // [max_slots][n_blocks]: entries of each update-block's list segment
    int32_t n_blocks;                   // blocks of the update kernel = list segments of seg_px pixels
    int32_t seg_px, upb;                // block b owns the 128-pixel units [b*units/n_blocks, (b+1)*units/n_blocks): upb or
                                        // upb-1 of them; seg_px = upb * 128 = capacity of a list segment
    int32_t units;                      // ceil(n / 128)
    uint32_t px_off;                    // global index of this handle's pixel 0 (row band of a pixel-sharded clip):
                                        // Philox counters use global pixel indices
    // optional pixel models (emulator.py:58-80, 694-703, 719-725)
    int32_t scidvs, pr_noise;
    void *hp, *prev_photo;              // scidvs_highpass / scidvs_previous_photo, state dtype
    void *pr_eff;                       // photoreceptor + photoreceptor_noise_arr as the change amplifier sees it
    float *tau_arr, *noise_arr;         // scidvs_tau_arr, photoreceptor_noise_arr (float32 tensors)
    const float *lut;                   // [256] lin_log
    FrameCtrl *ctrl;                    // [max_slots+1]
    uint32_t *hist_pre, *hist_post, *segoff, *cursor;   // [max_slots][seg_stride]
    int32_t *abort_flag;                // [2]: status, slot
    unsigned long long *chain_base;     // row at which the frames after a multi-frame chunk continue
};

struct FrameParams {
    double t_prev, t_frame, dt;
    double eps_scale;                   // delta_time / tau          (emulator_utils.py:84)
    float dt_f;                         // float32(delta_time)       (emulator_utils.py:129)
    uint32_t frame_index;               // Philox counter word
    double shot_c;                      // (shot_noise_rate_hz/2)*delta_time (emulator_utils.py:323-324)
    double shot_bound;                  // >= every pixel's ON/OFF shot probability of this frame (x >= 0)
    float shot_lo_f, shot_hi_f;         // float32 fast reject: a draw r with shot_lo_f <= r <= shot_hi_f cannot fire
    uint32_t pref_lo;                   // device RNG: a 12-bit prefix p with pref_lo <= p < 4096 - pref_lo cannot fire
    float pr_vrms_f, pr_ome_f, pr_eps_f;// photoreceptor noise: float32(vrms), float32(1-dt/tau), float32(dt/tau)
    int32_t scidvs_first;               // the frame that creates scidvs_highpass (zeros) and scidvs_previous_photo
    uint64_t capacity;
};

// ---------------------------------------------------------------------------------------------
// ATen restatements
// ---------------------------------------------------------------------------------------------
// aten/src/ATen/native/BinaryOps.h div_floor_floating, a >= 0, b > 0
template <typename S> __device__ __forceinline__ int32_t div_floor_count(S a, S b);
// Exact shortcuts (a >= b > 0): for b <= a < 2b, fmod(a,b) = a-b exactly (Sterbenz), a-(a-b) = b,
// b/b = 1 -> 1; for 2b <= a < 3b, fmod = a-2b exactly, a-(a-2b) = 2b, 2b/b = 2 -> 2. The test
// (a-2b) < b decides a < 3b correctly even where a-2b rounds (a > 4b). Beyond that: the full formula.
template <> __device__ __forceinline__ int32_t div_floor_count<double>(double a, double b) {
    if (a < b) return 0;                // fmod(a,b)=a -> (a-a)/b = 0
    const double b2 = b + b;
    if (a < b2) return 1;
    if (a - b2 < b) return 2;
    double mod = fmod(a, b);
    double div = (a - mod) / b;
    double fl = floor(div);
    if (div - fl > 0.5) fl += 1.0;
    return (int32_t)fl;
}
template <> __device__ __forceinline__ int32_t div_floor_count<float>(float a, float b) {
    if (a < b) return 0;
    const float b2 = b + b;
    if (a < b2) return 1;
    if (a - b2 < b) return 2;
    float mod = fmodf(a, b);
    float div = (a - mod) / b;
    float fl = floorf(div);
    if (div - fl > 0.5f) fl += 1.0f;
    return (int32_t)fl;
}

struct TsParams {                       // torch.linspace(t_prev+ts_step, t_frame, steps, float32)
    float start, end, step;
    int32_t steps;
    int32_t filter_active;
};
__device__ __forceinline__ TsParams make_ts(const FrameParams &p, int32_t max_n, double refr_d) {
    TsParams t;
    t.steps = max_n > 0 ? max_n : 1;
    double ts_step = p.dt / (double)t.steps;             // emulator.py:792
    t.start = (float)(p.t_prev + ts_step);
    t.end = (float)p.t_frame;
    t.step = t.steps > 1 ? (t.end - t.start) / (float)(t.steps - 1) : 0.0f;
    t.filter_active = refr_d > ts_step;                  // emulator.py:830
    return t;
}
__device__ __forceinline__ float linspace_f32(const TsParams &t, int32_t i) {
    if (t.steps == 1) return t.start;
    if (i < t.steps / 2) return fmaf(t.step, (float)i, t.start);
    return fmaf(-t.step, (float)(t.steps - 1 - i), t.end);
}

// lin_log for a non-integer value (emulator_utils.py:18-45); integer values use the table
__device__ __forceinline__ float lin_log_eval(double x) {
    const double f = (1.0 / 20.0) * 2.995732273553991;   // math.log(20)
    double y = (x <= 20.0) ? x * f : log(x);
    y = rint(y * 1e8) / 1e8;
    return (float)y;
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-R (rng_mode 1)
// ---------------------------------------------------------------------------------------------
template <int ROUNDS>
__device__ __forceinline__ uint4 philox4x32(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < ROUNDS; r++) {
        uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0;
        key.y += W1;
    }
    return ctr;
}
// (x>>8 + 0.5) * 2^-24 in (0,1) and (x>>8) * 2^-24 in [0,1): both exact in float32, one instruction after the convert
__device__ __forceinline__ float u01_open(uint32_t x) { return fmaf((float)(x >> 8), 1.0f / 16777216.0f, 0.5f / 16777216.0f); }
__device__ __forceinline__ float u01_half(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }
__device__ __forceinline__ float sqrt_approx(float x) {
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Per-frame noise of one aligned quad of pixels (GLOBAL pixel indices 4q .. 4q+3 of the whole frame, so that a
// pixel-sharded run draws what the unsharded run draws) from ONE Philox call:
//   n[j]    : N(0,1) for the leak jitter (emulator_utils.py:122-124). Box-Muller on fast intrinsics: radius from 24
//             bits, angle from 16 bits -- this stream only has to be normal, not torch's bits;
//   pref[j] : 12 uniform bits per pixel from the bits Box-Muller leaves over: the top of the pixel's shot-noise
//             uniform (emulator_utils.py:340-343). Only a pixel whose prefix lies within pref_lo of either end can
//             fire; it then takes its low bits from a second call (shot_uniform) -- a few pixels per thousand.
__device__ __forceinline__ void noise_quad(uint64_t seed, uint32_t quad, uint32_t frame_index, float n[4],
                                           uint32_t pref[4]) {
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    const uint4 r = philox4x32<kPhiloxRounds>(make_uint4(quad, frame_index, 0u, 0x6c65616bu), key);
    const float a = sqrt_approx(-2.0f * __logf(u01_open(r.x))), b = sqrt_approx(-2.0f * __logf(u01_open(r.z)));
    float sa, ca, sb, cb;
    __sincosf(6.283185307179586f * ((float)(r.y >> 16) * (1.0f / 65536.0f)), &sa, &ca);
    __sincosf(6.283185307179586f * ((float)(r.w >> 16) * (1.0f / 65536.0f)), &sb, &cb);
    n[0] = a * ca; n[1] = a * sa; n[2] = b * cb; n[3] = b * sb;
    pref[0] = (r.x & 0xffu) | ((r.y & 0xfu) << 8);
    pref[1] = (r.y >> 4) & 0xfffu;
    pref[2] = (r.z & 0xffu) | ((r.w & 0xfu) << 8);
    pref[3] = (r.w >> 4) & 0xfffu;
}
// The shot-noise uniform of pixel j of the quad, in [0,1): 12-bit prefix, then 20 bits of a second Philox call,
// truncated to float32 (never rounds up to 1).
__device__ __forceinline__ float shot_uniform(uint64_t seed, uint32_t quad, uint32_t frame_index, int j, uint32_t pref) {
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    const uint4 r = philox4x32<kPhiloxRounds>(make_uint4(quad, frame_index, 1u, 0x73686f74u), key);
    const uint32_t w = j == 0 ? r.x : (j == 1 ? r.y : (j == 2 ? r.z : r.w));
    return __uint2float_rz((pref << 20) | (w >> 12)) * (1.0f / 4294967296.0f);
}
__device__ __forceinline__ bool shot_candidate(uint32_t pref, uint32_t pref_lo) {
    return pref < pref_lo || pref >= 4096u - pref_lo;
}
// noise of the 4 consecutive pixels starting at GLOBAL index g0: one call when g0 is quad-aligned (always, unless a
// row band of a sharded clip starts at an odd offset); otherwise two calls, out of line
__device__ __noinline__ void noise_px4_unaligned(uint64_t seed, uint32_t g0, uint32_t frame_index, float *n, uint32_t *pref) {
    const uint32_t q = g0 >> 2, r = g0 & 3u;
    float na[8];
    uint32_t pa[8];
    noise_quad(seed, q, frame_index, na, pa);
    noise_quad(seed, q + 1, frame_index, na + 4, pa + 4);
    for (int k = 0; k < 4; k++) { n[k] = na[r + k]; pref[k] = pa[r + k]; }
}
__device__ __forceinline__ void noise_px4(uint64_t seed, uint32_t g0, uint32_t frame_index, float n[4], uint32_t pref[4]) {
    if ((g0 & 3u) == 0) noise_quad(seed, g0 >> 2, frame_index, n, pref);
    else noise_px4_unaligned(seed, g0, frame_index, n, pref);
}

// ---------------------------------------------------------------------------------------------
// vector load helpers: 4 consecutive elements starting at i (i % 4 == 0)
// ---------------------------------------------------------------------------------------------
template <int FT> __device__ __forceinline__ void load_frame4(const void *frame, int i, int n, double x[4]) {
    if (FT == V2E_U8) {
        const uint8_t *f = (const uint8_t *)frame;
        if (i + 4 <= n && ((((uintptr_t)f) + i) & 3) == 0) {
            uchar4 v = __ldg((const uchar4 *)(f + i));
            x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++) x[k] = (i + k < n) ? (double)f[i + k] : 0.0;
        }
    } else if (FT == V2E_F32) {
        const float *f = (const float *)frame;
        if (i + 4 <= n && (((uintptr_t)(f + i)) & 15) == 0) {
            float4 v = __ldg((const float4 *)(f + i));
            x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++) x[k] = (i + k < n) ? (double)f[i + k] : 0.0;
        }
    } else {
        const double *f = (const double *)frame;
#pragma unroll
        for (int k = 0; k < 4; k++) x[k] = (i + k < n) ? f[i + k] : 0.0;
    }
}
__device__ __forceinline__ void load_f32x4_any(const float *p, int i, int n, float v[4]) {
    if (i + 4 <= n && (((uintptr_t)(p + i)) & 15) == 0) {
        float4 t = __ldg((const float4 *)(p + i));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
#pragma unroll
        for (int k = 0; k < 4; k++) v[k] = (i + k < n) ? p[i + k] : 0.0f;
    }
}
// state arrays are padded to a multiple of 4 and 256-byte aligned: always vector
__device__ __forceinline__ void ld4(const float *p, int i, float v[4]) {
    float4 t = *(const float4 *)(p + i);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void ld4(const double *p, int i, double v[4]) {
    double2 a = *(const double2 *)(p + i), b = *(const double2 *)(p + i + 2);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
__device__ __forceinline__ void st4(float *p, int i, const float v[4]) {
    *(float4 *)(p + i) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void st4(double *p, int i, const double v[4]) {
    *(double2 *)(p + i) = make_double2(v[0], v[1]);
    *(double2 *)(p + i + 2) = make_double2(v[2], v[3]);
}

// shot-noise flags of one pixel (emulator_utils.py:323-349): bit0 ON, bit1 OFF
__device__ __forceinline__ int shot_flags(const EmuDev &d, double shot_c, double x, float rnd,
                                          float thp, float thn) {
    double inten01 = (x + 20.0) / 275.0;
    double factor = shot_c * (d.shot_inten_m1 * inten01 + 1.0);
    double pre_on, pre_off;
    if (d.per_pixel_thres) {
        pre_on = (double)((float)d.pos_nom / thp);       // emulator.py:475-478, float32 tensor
        pre_off = (double)((float)d.neg_nom / thn);
    } else {
        pre_on = (double)(float)(d.pos_nom / d.pos_nom); // torch.div of two Python floats
        pre_off = (double)(float)(d.neg_nom / d.neg_nom);
    }
    double r = (double)rnd;
    int on = r > 1.0 - factor * pre_on;
    int off = r < factor * pre_off;
    return on | (off << 1);
}

// ---------------------------------------------------------------------------------------------
// emission plan: run by the last block of the last counting kernel of a frame
// ---------------------------------------------------------------------------------------------
__device__ void plan_frame(const EmuDev &d, const FrameParams &p, int slot) {
    __shared__ uint32_t s_part[kThreads];
    __shared__ uint32_t s_tot[2];
    FrameCtrl *c = d.ctrl + slot;
    const int tid = threadIdx.x;
    int32_t max_n = *(volatile int32_t *)&c->max_n;
    if (max_n > d.iter_cap) {
        if (tid == 0 && atomicCAS(d.abort_flag, 0, V2E_E_ITER_CAP) == 0) d.abort_flag[1] = slot;
        return;
    }
    TsParams ts = make_ts(p, max_n, d.refr_d);
    const uint32_t *h = (ts.filter_active && d.refr_on) ? d.hist_post + (size_t)slot * d.seg_stride
                                                         : d.hist_pre + (size_t)slot * d.seg_stride;
    const uint32_t *hs = d.hist_pre + (size_t)slot * d.seg_stride;     // shot counters live at the end
    uint32_t *off = d.segoff + (size_t)slot * d.seg_stride;
    const int nseg = 2 * max_n;
    if (nseg <= 64) {
        // the usual case (a handful of iterations): one warp, two segments per lane, shuffle scan
        if (tid >= 32) return;
        const int s0 = 2 * tid, s1 = 2 * tid + 1;           // (iteration tid, ON) and (iteration tid, OFF)
        const uint32_t v0 = s0 < nseg ? h[s0] : 0u, v1 = s1 < nseg ? h[s1] : 0u;
        uint32_t incl = v0 + v1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (tid >= o) incl += t;
        }
        const uint32_t excl = incl - (v0 + v1);
        if (s0 < nseg) off[s0] = excl;
        if (s1 < nseg) off[s1] = excl + v0;
        const uint32_t sig = __shfl_sync(0xffffffffu, incl, 31);
        const uint32_t sig_on = __reduce_add_sync(0xffffffffu, v0);
        if (tid == 0) {
            const uint32_t shot_on = hs[2 * d.iter_cap], shot_off = hs[2 * d.iter_cap + 1];
            off[2 * d.iter_cap] = sig;
            off[2 * d.iter_cap + 1] = sig + shot_on;
            const uint32_t total = sig + shot_on + shot_off;
            c->filter_active = ts.filter_active && d.refr_on;
            c->n_on = sig_on + shot_on;
            c->n_off = (sig - sig_on) + shot_off;
            c->n_shot_on = shot_on;
            c->n_shot_off = shot_off;
            c->n_events = total;
            const uint64_t base = c->ev_base;
            if (base + total > p.capacity) {
                if (atomicCAS(d.abort_flag, 0, V2E_E_CAPACITY) == 0) d.abort_flag[1] = slot;
            } else {
                d.ctrl[slot + 1].ev_base = base + total;
                *d.chain_base = base + total;
                c->planned = 1;
            }
            __threadfence();
        }
        return;
    }
    const int per = (nseg + kThreads - 1) / kThreads;
    uint32_t sum = 0, on = 0;
    for (int k = 0; k < per; k++) {
        int s = tid * per + k;
        if (s < nseg) {
            uint32_t v = h[s];
            sum += v;
            if ((s & 1) == 0) on += v;
        }
    }
    s_part[tid] = sum;
    if (tid < 2) s_tot[tid] = 0;
    __syncthreads();
    atomicAdd(&s_tot[0], on);
    // exclusive scan of the per-thread partial sums (256 entries, serial by warp 0 lane 0 is fine
    // but a Hillis-Steele pass keeps it short)
    for (int o = 1; o < kThreads; o <<= 1) {
        uint32_t v = tid >= o ? s_part[tid - o] : 0;
        __syncthreads();
        s_part[tid] += v;
        __syncthreads();
    }
    uint32_t run = s_part[tid] - sum;
    for (int k = 0; k < per; k++) {
        int s = tid * per + k;
        if (s < nseg) {
            off[s] = run;
            run += h[s];
        }
    }
    __syncthreads();
    if (tid == 0) {
        uint32_t sig = s_part[kThreads - 1];
        uint32_t sig_on = s_tot[0];
        uint32_t shot_on = hs[2 * d.iter_cap], shot_off = hs[2 * d.iter_cap + 1];
        off[2 * d.iter_cap] = sig;
        off[2 * d.iter_cap + 1] = sig + shot_on;
        uint32_t total = sig + shot_on + shot_off;
        c->filter_active = ts.filter_active && d.refr_on;
        c->n_on = sig_on + shot_on;
        c->n_off = (sig - sig_on) + shot_off;
        c->n_shot_on = shot_on;
        c->n_shot_off = shot_off;
        c->n_events = total;
        uint64_t base = c->ev_base;
        if (base + total > p.capacity) {
            if (atomicCAS(d.abort_flag, 0, V2E_E_CAPACITY) == 0) d.abort_flag[1] = slot;
        } else {
            d.ctrl[slot + 1].ev_base = base + total;
            *d.chain_base = base + total;
            c->planned = 1;
        }
        __threadfence();
    }
}

__device__ __forceinline__ bool last_block(uint32_t *ticket) {
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (s_last) __threadfence();
    return s_last;
}

// ---------------------------------------------------------------------------------------------
// first frame (emulator.py:663-717)
// ---------------------------------------------------------------------------------------------
template <typename S, int FT>
__global__ void __launch_bounds__(kThreads) emu_first_frame_kernel(EmuDev d, FrameParams p, const void *frame) {
    __shared__ float s_lut[256];
    s_lut[threadIdx.x] = d.lut[threadIdx.x];
    __syncthreads();
    int i0 = (blockIdx.x * kThreads + threadIdx.x) * kVec;
    if (i0 >= d.n) return;
    double x[4];
    load_frame4<FT>(frame, i0, d.n, x);
    S lp[4], base[4];
    float tm[4];
    double su[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        double xv = x[k];
        float lnf = 0.f;
        if (!d.hdr) lnf = (FT == V2E_U8 || (xv >= 0.0 && xv <= 255.0 && xv == floor(xv))) ? s_lut[(int)xv] : lin_log_eval(xv);
        if (sizeof(S) == 8) {
            double ln = d.hdr ? xv : (double)lnf;
            double v = ln;
            if (d.lowpass_on) {
                double eps = ((xv + 20.0) / 275.0) * p.eps_scale;
                if (eps > 1.0) eps = 1.0;
                v = (1.0 - eps) * ln + eps * ln;      // lp seeded with log_new, still filtered once
            }
            lp[k] = (S)v;
            su[k] = v;
            base[k] = (S)(d.csdvs ? v - v : v);      // emulator.py:714
        } else {
            lp[k] = (S)lnf;
            base[k] = (S)lnf;
            su[k] = 0.0;
        }
        tm[k] = 0.0f - d.refr_f;                     // emulator.py:508-511
    }
    st4((S *)d.lp, i0, lp);
    st4((S *)d.base, i0, base);
    if (d.refr_on) st4(d.tmem, i0, tm);
    if (d.csdvs) st4(d.cs_bufs ? d.cs_bufs : d.surround, i0, su);     // v2e_emu_first_frame resets cs_cur to 0
}

// ---------------------------------------------------------------------------------------------
// centre-surround model (emulator.py:1061-1124), only when cs_lambda_pixels is set
// ---------------------------------------------------------------------------------------------
// photoreceptor low-pass alone: the surround diffusion needs the whole new lp field first
template <int FT>
__global__ void __launch_bounds__(kThreads) emu_lp_kernel(EmuDev d, FrameParams p, const void *frame) {
    __shared__ float s_lut[256];
    if (*(volatile int32_t *)d.abort_flag) return;
    s_lut[threadIdx.x] = d.lut[threadIdx.x];
    __syncthreads();
    const int i0 = (blockIdx.x * kThreads + threadIdx.x) * kVec;
    if (i0 >= d.n) return;
    double x[4], lp[4];
    load_frame4<FT>(frame, i0, d.n, x);
    ld4((const double *)d.lp, i0, lp);
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const double xv = x[k];
        double ln;
        if (d.hdr) ln = xv;
        else ln = (double)((FT == V2E_U8 || (xv >= 0.0 && xv <= 255.0 && xv == floor(xv))) ? s_lut[(int)xv] : lin_log_eval(xv));
        if (d.lowpass_on) {
            double eps = ((xv + 20.0) / 275.0) * p.eps_scale;
            if (eps > 1.0) eps = 1.0;
            lp[k] = (1.0 - eps) * lp[k] + eps * ln;
        } else {
            lp[k] = ln;
        }
    }
    st4((double *)d.lp, i0, lp);
}

// One Euler step h += alpha_p*(p - h) + alpha_h*lap(float32(h)) with replicate padding
// (emulator.py:1105-1121). p, h float64; the 3x3 stencil is a float32 conv2d whose summation order is the
// reference's CPU backend's (see oracle/emu_oracle.c); alpha_h meets a float32 tensor -> float32 product.
// Step k runs only if every earlier step changed some pixel by more than 1e-5 (the reference's while
// condition); the maxima are exchanged through cs_max.
// Ring form: step `step` of the frame is step `i` of its chunk; it reads ring buffer (cs_cur + i) % cs_ring and writes
// the next one. Single GPU: one chunk per frame, ring of 2 (ping-pong), and the cascade above. Pixel-sharded
// (emulator.py:1102-1124 over row bands): the handle carries K halo rows of the neighbours above / below, a chunk is
// K steps between two halo exchanges, step i of a chunk is valid on rows >= i from a halo edge; the maximum is taken
// over the rank's own rows only and reduced over the ranks after the chunk, so the steps of a chunk run without
// knowing whether an earlier step of the same chunk ended the iteration -- the ring (K + 1 buffers) keeps every
// step's result and emu_csdvs_advance_kernel picks the right one.
__global__ void __launch_bounds__(kThreads)
emu_csdvs_step_kernel(EmuDev d, double alpha_p, float alpha_h, int step, int i, int sharded) {
    if (*(volatile int32_t *)d.abort_flag) return;
    if (sharded) { if (*(volatile int32_t *)d.cs_done) return; }
    else if (step > 0 && __longlong_as_double((long long)d.cs_max[step - 1]) <= 1e-5) return;
    const int cur = (*(volatile int32_t *)d.cs_cur + i) % d.cs_ring;
    const int nxt = (cur + 1) % d.cs_ring;
    const double *h = d.cs_bufs ? d.cs_bufs + (size_t)cur * d.cs_stride : (cur ? d.surround2 : d.surround);
    double *hn = d.cs_bufs ? d.cs_bufs + (size_t)nxt * d.cs_stride : (nxt ? d.surround2 : d.surround);
    const double *pp = (const double *)d.lp;
    const int idx = blockIdx.x * kThreads + threadIdx.x;
    double a = 0.0;
    if (idx < d.n) {
        const int y = idx / d.W, x = idx - y * d.W;
        const int ym = y > 0 ? y - 1 : 0, yp = y < d.H - 1 ? y + 1 : d.H - 1;
        const int xm = x > 0 ? x - 1 : 0, xp = x < d.W - 1 ? x + 1 : d.W - 1;
        const double hc = h[idx];
        const float uu = (float)h[ym * d.W + x], ll = (float)h[y * d.W + xm], cc = -4.0f * (float)hc;
        const float rr = (float)h[y * d.W + xp], dd = (float)h[yp * d.W + x];
        const float acc = d.cs_seq_order ? ((((uu + ll) + cc) + rr) + dd) : (uu + ll) + (cc + (rr + dd));
        const float h_term = alpha_h * acc;
        const double chg = alpha_p * (pp[idx] - hc) + (double)h_term;
        hn[idx] = hc + chg;
        if (y >= d.cs_y_lo && y < d.cs_y_hi) a = fabs(chg);
    }
    // block max of |change| -> one atomicMax (non-negative doubles order like their bit patterns)
    unsigned long long bits = (unsigned long long)__double_as_longlong(a);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long t = __shfl_xor_sync(0xffffffffu, bits, o);
        bits = t > bits ? t : bits;
    }
    __shared__ unsigned long long s_m[kThreads / 32];
    if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = bits;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kThreads / 32; w++) bits = s_m[w] > bits ? s_m[w] : bits;
        atomicMax(&d.cs_max[step], bits);
    }
}

// The same Euler steps s0 .. s1-1 in ONE cooperative launch: a grid-wide barrier between steps instead of a kernel
// launch per step (the iteration is a chain of tiny stencil passes over an L2-resident field: launch latency, not
// bandwidth, was what a step cost). Single GPU: the loop ends right after the first step whose max|change| <= 1e-5, as
// the reference's while loop does (emulator.py:1105-1121), and block 0 records cs_steps_taken and the new ring position.
// Sharded: a chunk of K steps between two halo exchanges, no early exit inside (the maxima are reduced over the ranks
// after the chunk; emu_csdvs_advance_kernel picks the step).
constexpr int kCsThreads = 512;
__global__ void __launch_bounds__(kCsThreads)
emu_csdvs_iter_kernel(EmuDev d, double alpha_p, float alpha_h, int s0, int s1, int sharded, int slot) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ unsigned long long s_m[kCsThreads / 32];
    // uniform over the grid: read before anyone can change them (only the tail of this kernel / later kernels do)
    if (*(volatile int32_t *)d.abort_flag) return;
    if (sharded && *(volatile int32_t *)d.cs_done) return;
    const int cur0 = *(volatile int32_t *)d.cs_cur;
    const double *pp = (const double *)d.lp;
    const int stride = gridDim.x * kCsThreads;
    int taken = s1 - s0;
    for (int s = s0; s < s1; s++) {
        const int cur = (cur0 + (s - s0)) % d.cs_ring, nxt = (cur + 1) % d.cs_ring;
        const double *h = d.cs_bufs ? d.cs_bufs + (size_t)cur * d.cs_stride : (cur ? d.surround2 : d.surround);
        double *hn = d.cs_bufs ? d.cs_bufs + (size_t)nxt * d.cs_stride : (nxt ? d.surround2 : d.surround);
        double a = 0.0;
        for (int idx = blockIdx.x * kCsThreads + threadIdx.x; idx < d.n; idx += stride) {
            const int y = idx / d.W, x = idx - y * d.W;
            const int ym = y > 0 ? y - 1 : 0, yp = y < d.H - 1 ? y + 1 : d.H - 1;
            const int xm = x > 0 ? x - 1 : 0, xp = x < d.W - 1 ? x + 1 : d.W - 1;
            const double hc = h[idx];
            const float uu = (float)h[ym * d.W + x], ll = (float)h[y * d.W + xm], cc = -4.0f * (float)hc;
            const float rr = (float)h[y * d.W + xp], dd = (float)h[yp * d.W + x];
            const float acc = d.cs_seq_order ? ((((uu + ll) + cc) + rr) + dd) : (uu + ll) + (cc + (rr + dd));
            const float h_term = alpha_h * acc;
            const double chg = alpha_p * (pp[idx] - hc) + (double)h_term;
            hn[idx] = hc + chg;
            if (y >= d.cs_y_lo && y < d.cs_y_hi) a = fmax(a, fabs(chg));
        }
        unsigned long long bits = (unsigned long long)__double_as_longlong(a);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            unsigned long long t = __shfl_xor_sync(0xffffffffu, bits, o);
            bits = t > bits ? t : bits;
        }
        if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = bits;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < kCsThreads / 32; w++) bits = s_m[w] > bits ? s_m[w] : bits;
            atomicMax(&d.cs_max[s], bits);
        }
        grid.sync();                            // step s complete everywhere, its maximum final
        if (!sharded && __longlong_as_double((long long)*(volatile unsigned long long *)&d.cs_max[s]) <= 1e-5) {
            taken = s - s0 + 1;
            break;
        }
    }
    if (!sharded && blockIdx.x == 0 && threadIdx.x == 0) {
        d.ctrl[slot].cs_steps = s0 + taken;
        *d.cs_cur = (cur0 + taken) % d.cs_ring;     // everyone read cs_cur before the first barrier
    }
}

// sharded: after the chunk's maxima have been reduced over the ranks. Steps [s0, s1) ran from ring position cs_cur;
// the iteration ends with the first step whose global max|change| <= 1e-5 (that step is applied, emulator.py:1105-1121).
__global__ void emu_csdvs_advance_kernel(EmuDev d, int s0, int s1, int slot) {
    if (*(volatile int32_t *)d.abort_flag) return;
    if (*d.cs_done) return;
    int taken = s1 - s0;
    for (int k = s0; k < s1; k++)
        if (__longlong_as_double((long long)d.cs_max[k]) <= 1e-5) { taken = k - s0 + 1; *d.cs_done = 1; break; }
    *d.cs_cur = (*d.cs_cur + taken) % d.cs_ring;
    d.ctrl[slot].cs_steps = s0 + taken;
}
// sharded halo exchange: the K own rows next to each band edge of the current surround buffer -> send[2][K][W];
// recv[2][K][W] (the neighbours' rows) -> the halo rows of the current buffer
__global__ void emu_csdvs_pack_kernel(EmuDev d, double *send, int K) {
    const double *h = d.cs_bufs + (size_t)(*d.cs_cur) * d.cs_stride;
    const int per = K * d.W;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 2 * per; i += gridDim.x * blockDim.x) {
        const int side = i / per, r = (i - side * per) / d.W, x = i % d.W;
        const int y = side == 0 ? d.cs_y_lo + r : d.cs_y_hi - K + r;        // top K / bottom K own rows
        send[i] = h[(size_t)y * d.W + x];
    }
}
// recv_above / recv_below: [K][W] rows of the neighbour above (its bottom edge) / below (its top edge); null at the
// image border
__global__ void emu_csdvs_unpack_kernel(EmuDev d, const double *recv_above, const double *recv_below, int K) {
    double *h = d.cs_bufs + (size_t)(*d.cs_cur) * d.cs_stride;
    const int per = K * d.W;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 2 * per; i += gridDim.x * blockDim.x) {
        const int side = i / per, r = (i - side * per) / d.W, x = i % d.W;
        // side 0: halo above the own rows (present iff cs_y_lo > 0), side 1: halo below
        if (side == 0 && recv_above && d.cs_y_lo >= K) h[(size_t)(d.cs_y_lo - K + r) * d.W + x] = recv_above[i];
        if (side == 1 && recv_below && d.cs_y_hi + K <= d.H) h[(size_t)(d.cs_y_hi + r) * d.W + x] = recv_below[i - per];
    }
}

__global__ void emu_csdvs_finish_kernel(EmuDev d, int num_steps, int slot) {
    if (*(volatile int32_t *)d.abort_flag) return;
    int steps = num_steps;
    for (int k = 0; k < num_steps; k++)
        if (__longlong_as_double((long long)d.cs_max[k]) <= 1e-5) { steps = k + 1; break; }
    d.ctrl[slot].cs_steps = steps;
    *d.cs_cur = (*d.cs_cur + steps) % d.cs_ring;
}

// ---------------------------------------------------------------------------------------------
// optional front end (SCIDVS and/or photoreceptor noise): emulator.py:686-703, 719-725, 748.
// Low-pass of the whole field, the noise IIR, the nonlinear CR high-pass, and the field the change
// amplifier sees: pr_eff = (scidvs ? 2*hp : lp) + photoreceptor_noise_arr. The update kernel then runs
// with lp_done and reads pr_eff in place of lp.
// ---------------------------------------------------------------------------------------------
template <typename S, int FT>
__global__ void __launch_bounds__(kThreads) emu_front_kernel(EmuDev d, FrameParams p, const void *frame,
                                                             const float *pr_randn, int lp_done) {
    __shared__ float s_lut[256];
    if (*(volatile int32_t *)d.abort_flag) return;
    s_lut[threadIdx.x] = d.lut[threadIdx.x];
    __syncthreads();
    const int i0 = (blockIdx.x * kThreads + threadIdx.x) * kVec;
    if (i0 >= d.n) return;
    double x[4];
    S lp[4], hp[4], pv[4], eff[4];
    float na[4], rn[4], tau[4];
    load_frame4<FT>(frame, i0, d.n, x);
    ld4((const S *)d.lp, i0, lp);
    if (d.scidvs) { ld4((const S *)d.hp, i0, hp); ld4((const S *)d.prev_photo, i0, pv); ld4(d.tau_arr, i0, tau); }
    if (d.pr_noise) {
        ld4(d.noise_arr, i0, na);
        if (pr_randn) load_f32x4_any(pr_randn, i0, d.n, rn);
        else {
            const uint2 key = make_uint2((uint32_t)d.seed, (uint32_t)(d.seed >> 32));
            uint4 r = philox4x32<kPhiloxRounds>(make_uint4((uint32_t)(i0 >> 2), p.frame_index, 2u, 0x70726e7au), key);
            float a = sqrt_approx(-2.0f * __logf(u01_open(r.x))), b = sqrt_approx(-2.0f * __logf(u01_open(r.z)));
            float sa, ca, sb, cb;
            __sincosf(6.283185307179586f * u01_half(r.y), &sa, &ca);
            __sincosf(6.283185307179586f * u01_half(r.w), &sb, &cb);
            rn[0] = a * ca; rn[1] = a * sa; rn[2] = b * cb; rn[3] = b * sb;
        }
    }
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const double xv = x[k];
        if (!lp_done) {
            float lnf = 0.f;
            if (!d.hdr) lnf = (FT == V2E_U8 || (xv >= 0.0 && xv <= 255.0 && xv == floor(xv))) ? s_lut[(int)xv] : lin_log_eval(xv);
            if (sizeof(S) == 8) {
                const double ln = d.hdr ? xv : (double)lnf;
                if (d.lowpass_on) {
                    double eps = ((xv + 20.0) / 275.0) * p.eps_scale;
                    if (eps > 1.0) eps = 1.0;
                    lp[k] = (S)((1.0 - eps) * (double)lp[k] + eps * ln);
                } else {
                    lp[k] = (S)ln;
                }
            } else {
                lp[k] = (S)lnf;
            }
        }
        // photoreceptor noise (emulator.py:694-701; emulator_utils.py:96-99 with a scalar eps, no clamp)
        if (d.pr_noise) {
            const float noise = p.pr_vrms_f * rn[k];
            if (d.lowpass_on) {
                const float a = p.pr_ome_f * na[k], b = p.pr_eps_f * noise;
                na[k] = a + b;
            } else {
                na[k] = noise;
            }
        }
        // SCIDVS (emulator.py:58-80, 719-725)
        S photo = lp[k];
        if (d.scidvs) {
            if (p.scidvs_first) { hp[k] = (S)0; pv[k] = lp[k]; }
            const float inv_tau = 1.0f / tau[k];
            if (sizeof(S) == 8) {
                const double dvdt = (double)inv_tau * sinh((double)hp[k] / (1 / 0.7));
                const double d1 = (double)lp[k] - (double)pv[k], d2 = p.dt * dvdt;
                hp[k] = (S)((double)hp[k] + (d1 - d2));
            } else {
                const float dvdt = inv_tau * sinhf((float)hp[k] / (float)(1 / 0.7));
                const float d1 = (float)lp[k] - (float)pv[k], d2 = p.dt_f * dvdt;
                hp[k] = (S)((float)hp[k] + (d1 - d2));
            }
            pv[k] = lp[k];
            photo = (S)2 * hp[k];
        }
        eff[k] = d.pr_noise ? (S)(photo + (S)na[k]) : (S)(photo + (S)0);
    }
    if (!lp_done) st4((S *)d.lp, i0, lp);
    if (d.scidvs) { st4((S *)d.hp, i0, hp); st4((S *)d.prev_photo, i0, pv); }
    if (d.pr_noise) st4(d.noise_arr, i0, na);
    st4((S *)d.pr_eff, i0, eff);
}

// ---------------------------------------------------------------------------------------------
// update kernel: emulator.py:663-775 for 4 pixels per thread
// RNG: 0 = replay (host-drawn fields), 1 = device (Philox). Everything else is a uniform runtime flag.
// FAST: the configuration fixed at compile time to v2e's CLI defaults in device-RNG mode (per-pixel
// thresholds, low-pass, leak and shot noise on, no hdr / csdvs): every uniform flag test disappears.
//
// Memory path: the per-pixel state (lp, base, thresholds, noise rate: 28 of the 47 bytes per pixel, the
// rest being the 1-byte frame and the stores) is staged through shared memory by 1-D TMA bulk copies
// (cp.async.bulk ... mbarrier::complete_tx). Every warp runs its own two-stage pipeline over 128-pixel
// units (4 pixels per lane): a block owns `upb` consecutive units, warp w takes units w, w+8, ...; lane 0
// issues the copies of the unit after next as soon as the warp has read a stage into registers, and the
// frame bytes of the next unit are prefetched into a register, so DRAM/L2 latency overlaps the arithmetic
// of the unit in between and no block-wide barrier sits in the loop. The grid is exactly one resident wave
// (3 blocks per SM) and the units are dealt out evenly (block sizes differ by at most one unit), so that at
// 1280x720 almost every warp has two units and the few third units run at the end on an otherwise idle SM.
//
// Tables in shared memory (per block, 256 entries, the 8-bit code is the index). With uint8 frames and
// the low-pass on, the update lp' = (1-eps)*lp + eps*ln needs only lp from the pixel: (1-eps) and the
// product eps*ln depend on the code alone, so they are evaluated once per block with exactly the
// reference's float64 operations (emulator_utils.py:84-99) and the pixel does one multiply and one add.
// Otherwise the tables hold lin_log(code) and inten01(code) = (code+20)/275.
// ---------------------------------------------------------------------------------------------
constexpr int kUnitPx = 32 * kVec;                 // pixels of one warp pass
constexpr int kWarps = kThreads / 32;
constexpr int kStages = 2;
template <typename S> struct StageLayout {         // one unit of one warp
    static constexpr int lp = 0;
    static constexpr int base = kUnitPx * (int)sizeof(S);
    static constexpr int thp = 2 * kUnitPx * (int)sizeof(S);
    static constexpr int thn = thp + kUnitPx * 4;
    static constexpr int nr = thn + kUnitPx * 4;
    static constexpr int bytes = nr + kUnitPx * 4;
    static constexpr int block_bytes = bytes * kStages * kWarps;
};

// Executed by the whole (converged) warp with warp-uniform operands; only the lane with leader != 0 issues.
// A plain `if (lane == 0)` around the asm makes nvcc emit an election loop per instruction.
__device__ __forceinline__ void bulk_load_pred(uint32_t dst_smem, const void *src, uint32_t bytes, uint32_t bar,
                                               uint32_t leader) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %4, 0;\n\t"
                 "@q cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n\t}"
                 ::"r"(dst_smem), "l"((uint64_t)src), "r"(bytes), "r"(bar), "r"(leader) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_pred(uint32_t bar, uint32_t bytes, uint32_t leader) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t"
                 "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes), "r"(leader) : "memory");
}

// event count |diff| // threshold with ATen's floor division (div_floor_count above), the common results
// 0 / 1 / 2 without a branch: a = |diff| >= 0, b > 0
template <typename S> __device__ __forceinline__ int32_t div_floor_count_fast(S a, S b) {
    const S b2 = b + b;
    int32_t cnt = (int32_t)(a >= b) + (int32_t)(a >= b2);
    if (a >= b2 && !(a - b2 < b)) cnt = div_floor_count<S>(a, b);     // >= 3 events: rare
    return cnt;
}

template <typename S, int FT, int RNG, bool FAST>
__global__ void __launch_bounds__(kThreads, 3)
emu_update_kernel(EmuDev d, FrameParams p, const void *frame, const float *leak_randn,
                  const float *shot_rand, int slot, int do_plan, int lp_done_arg) {
    const bool f_pp = FAST || d.per_pixel_thres, f_leak = FAST || d.leak_on, f_lp = FAST || d.lowpass_on;
    const bool f_shot = FAST || d.shot_on, f_hdr = FAST ? false : (bool)d.hdr, f_cs = FAST ? false : (bool)d.csdvs;
    const bool lp_done = FAST ? false : (bool)lp_done_arg;
    // code tables usable: uint8 frame, float64 low-pass computed here
    const bool tab = FAST || (FT == V2E_U8 && sizeof(S) == 8 && f_lp && !f_hdr && !lp_done);
    const bool need_lp = f_lp || lp_done;                 // otherwise lp' = lin_log(x): the old value is not read
    extern __shared__ __align__(128) unsigned char s_stage[];
    __shared__ double s_ta[256];                          // tab: 1-eps      else: lin_log
    __shared__ double s_tb[256];                          // tab: eps*ln     else: inten01
    __shared__ uint64_t s_full[kWarps][kStages];
    __shared__ uint32_t s_hist[kSegSmem + 2];
    __shared__ int s_max;
    __shared__ uint32_t s_act_total;
    const int tid = threadIdx.x, lane = tid & 31;
    // the shuffle tells the compiler that the warp index is warp-uniform: the TMA issue below then runs on
    // the uniform datapath instead of an election loop per instruction
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    // abort flag (set by an earlier frame's plan): read now, tested after the copies are in flight so that its
    // round trip is off the critical path; nothing is written before the test
    const int32_t abort_v = *(volatile int32_t *)d.abort_flag;
    const float lut_v = d.lut[tid];
    // this block's units; warp w owns units u0+w, u0+w+8, ...
    const int u0 = (int)(((long long)blockIdx.x * d.units) / d.n_blocks);
    const int u1 = (int)(((long long)(blockIdx.x + 1) * d.units) / d.n_blocks);
    const int nj = (u1 - u0 - warp + kWarps - 1) / kWarps;     // units of this warp (<= 0: none)
    unsigned char *my_stage = s_stage + (size_t)warp * (kStages * StageLayout<S>::bytes);
    // SCIDVS / photoreceptor noise: the front kernel has prepared what the change amplifier sees
    const S *lp_src = (lp_done && d.pr_eff) ? (const S *)d.pr_eff : (const S *)d.lp;
    const uint32_t leader = elect_one();
    const uint32_t stage_u32 = smem_u32(my_stage), bar_u32 = smem_u32(&s_full[warp][0]);
    auto issue = [&](int j) {                // whole warp, warp-uniform arguments
        const uint32_t bar = bar_u32 + 8u * (uint32_t)(j % kStages);
        const uint32_t st = stage_u32 + (uint32_t)(j % kStages) * (uint32_t)StageLayout<S>::bytes;
        const size_t px0 = (size_t)(u0 + warp + j * kWarps) * kUnitPx;
        constexpr uint32_t nS = kUnitPx * (uint32_t)sizeof(S), nF = kUnitPx * 4u;
        const uint32_t total = (need_lp ? nS : 0u) + nS + (f_pp ? 2u * nF : 0u) + (f_leak ? nF : 0u);
        mbar_expect_tx_pred(bar, total, leader);
        if (need_lp) bulk_load_pred(st + StageLayout<S>::lp, lp_src + px0, nS, bar, leader);
        bulk_load_pred(st + StageLayout<S>::base, (const S *)d.base + px0, nS, bar, leader);
        if (f_pp) {
            bulk_load_pred(st + StageLayout<S>::thp, d.pos_thres + px0, nF, bar, leader);
            bulk_load_pred(st + StageLayout<S>::thn, d.neg_thres + px0, nF, bar, leader);
        }
        if (f_leak) bulk_load_pred(st + StageLayout<S>::nr, d.noise_rate + px0, nF, bar, leader);
    };
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < kStages; s++) mbar_init(&s_full[warp][s], 1);
        fence_barrier_init();
    }
    __syncwarp();
#pragma unroll
    for (int s = 0; s < kStages; s++) if (s < nj) issue(s);
    if (tid == 0) { s_act_total = 0; s_max = 0; }
    {
        const double ln = (double)lut_v;
        const double inten01 = ((double)tid + 20.0) / 275.0;
        if (tab) {
            double eps = inten01 * p.eps_scale;          // emulator_utils.py:84
            if (eps > 1.0) eps = 1.0;                    // :96
            s_ta[tid] = 1.0 - eps;                       // :99 (1-eps)
            s_tb[tid] = eps * ln;                        //     eps*log_new_frame
        } else {
            s_ta[tid] = ln;
            s_tb[tid] = inten01;
        }
    }
    if (tid < kSegSmem + 2) s_hist[tid] = 0;
    // frame bytes of the warp's first unit (uint8 frames): in flight across the barrier
    const bool f_al = FT == V2E_U8 && (((uintptr_t)frame) & 3) == 0;
    auto load_codes = [&](int i0) -> uint32_t {          // 4 codes packed little-endian
        const uint8_t *f = (const uint8_t *)frame;
        if (f_al && i0 + 4 <= d.n) return __ldg((const uint32_t *)(f + i0));
        uint32_t v = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) if (i0 + k < d.n) v |= (uint32_t)f[i0 + k] << (8 * k);
        return v;
    };
    uint32_t codes_next = 0;
    if (FT == V2E_U8 && nj > 0) codes_next = load_codes((u0 + warp) * kUnitPx + lane * kVec);
    __syncthreads();
    if (abort_v) {                           // block-uniform; let the copies land before the block's smem goes away
#pragma unroll
        for (int s = 0; s < kStages; s++) if (s < nj) mbar_wait(&s_full[warp][s], 0);
        return;
    }
    FrameCtrl *c = d.ctrl + slot;
    uint32_t *hist = d.hist_pre + (size_t)slot * d.seg_stride;
    const double *su_ptr = nullptr;
    if (f_cs) {
        const int cur = *(volatile int32_t *)d.cs_cur;
        su_ptr = d.cs_bufs ? d.cs_bufs + (size_t)cur * d.cs_stride : (cur ? d.surround2 : d.surround);
    }
    const bool shot_here = f_shot && (RNG == 1 || shot_rand != nullptr);
    const uint32_t seg_base = (uint32_t)blockIdx.x * (uint32_t)d.seg_px;
    const int so = lane * kVec;                          // element offset inside the stage arrays
    int local_max = 0;
    uint32_t acc0 = 0, acc1 = 0;                         // ON / OFF counts of iterations 0 (low half) and 1 (high half)
    auto flush_acc = [&]() {
        if (lane == 0) {
            if (acc0 & 0xffffu) atomicAdd(&s_hist[0], acc0 & 0xffffu);
            if (acc1 & 0xffffu) atomicAdd(&s_hist[1], acc1 & 0xffffu);
            if (acc0 >> 16) atomicAdd(&s_hist[2], acc0 >> 16);
            if (acc1 >> 16) atomicAdd(&s_hist[3], acc1 >> 16);
        }
        acc0 = acc1 = 0;
    };

    for (int j = 0; j < nj; j++) {
        const int i0 = (u0 + warp + j * kWarps) * kUnitPx + lane * kVec;
        const bool t_on = i0 < d.n;
        const unsigned char *st = my_stage + (size_t)(j % kStages) * StageLayout<S>::bytes;
        int mags[4] = {0, 0, 0, 0}, pols[4] = {0, 0, 0, 0}, flg[4] = {0, 0, 0, 0};
        bool cand[4] = {false, false, false, false};
        short recs[4] = {0, 0, 0, 0};
        // direct (unstaged) inputs first: their latency overlaps the wait for the stage
        double x[4] = {0.0, 0.0, 0.0, 0.0};
        const uint32_t codes = codes_next;
        if (FT == V2E_U8 && j + 1 < nj) codes_next = load_codes(i0 + kWarps * kUnitPx);
        float lr[4], sr[4];
        double su[4];
        if (t_on) {
            if (FT != V2E_U8) load_frame4<FT>(frame, i0, d.n, x);
            if (f_cs) ld4(su_ptr, i0, su);
            if (RNG == 0 && f_leak) load_f32x4_any(leak_randn, i0, d.n, lr);
            if (RNG == 0 && shot_here) load_f32x4_any(shot_rand, i0, d.n, sr);
        }
        uint32_t pref[4] = {0u, 0u, 0u, 0u};
        const uint32_t g0 = (uint32_t)i0 + d.px_off;       // global pixel index (Philox counter)
        if (RNG == 1 && (f_leak || f_shot)) noise_px4(d.seed, g0, p.frame_index, lr, pref);
        // staged state -> registers
        S lp[4], base[4];
        float thp[4], thn[4], nr[4];
        mbar_wait(&s_full[warp][j % kStages], (uint32_t)((j / kStages) & 1));
        if (need_lp) ld4((const S *)(st + StageLayout<S>::lp), so, lp);
        ld4((const S *)(st + StageLayout<S>::base), so, base);
        if (f_pp) {
            ld4((const float *)(st + StageLayout<S>::thp), so, thp);
            ld4((const float *)(st + StageLayout<S>::thn), so, thn);
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++) { thp[k] = (float)d.pos_nom; thn[k] = (float)d.neg_nom; }
        }
        if (f_leak) ld4((const float *)(st + StageLayout<S>::nr), so, nr);
        __syncwarp();                                      // the stage has been read by the whole warp
        if (j + kStages < nj) issue(j + kStages);
        // packed counters of this thread's 4 pixels: byte 0 ON events of iteration 0, byte 1 OFF of
        // iteration 0, byte 2 ON of iteration 1, byte 3 OFF of iteration 1 (<= 4 each, <= 128 per warp)
        uint32_t pk = 0;
        int nact = 0, deep = 0;
        if (t_on) {
            bool shot_maybe = false;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int code_u8 = (int)((codes >> (8 * k)) & 0xffu);
                const double xv = (FT == V2E_U8) ? 0.0 : x[k];
                const bool is_code = FT == V2E_U8 || (xv >= 0.0 && xv <= 255.0 && xv == floor(xv));
                const int code = (FT == V2E_U8) ? code_u8 : (is_code ? (int)xv : 0);
                // photoreceptor low-pass (emulator_utils.py:57-109)
                if (!lp_done) {
                    if (tab) {
                        lp[k] = (S)(s_ta[code] * (double)lp[k] + s_tb[code]);
                    } else {
                        double ln;                           // float32 lin_log value, widened (or raw if hdr)
                        if (f_hdr) ln = xv;
                        else ln = is_code ? s_ta[code] : (double)lin_log_eval(xv);
                        if (sizeof(S) == 8 && f_lp) {
                            double inten01 = is_code ? s_tb[code] : (xv + 20.0) / 275.0;
                            double eps = inten01 * p.eps_scale;
                            if (eps > 1.0) eps = 1.0;
                            lp[k] = (S)((1.0 - eps) * (double)lp[k] + eps * ln);
                        } else {
                            lp[k] = (S)ln;                   // float32 state: exact, ln is a widened float32
                        }
                    }
                }
                // leak (emulator_utils.py:114-134): float32 products, subtract in S
                if (f_leak) {
                    float rate = (d.leak_rate_f * nr[k]) * (1.0f - d.leak_jit_f * lr[k]);
                    float delta = (p.dt_f * rate) * thp[k];
                    base[k] = base[k] - (S)delta;
                }
                // difference and event counts (emulator.py:748-772, emulator_utils.py:137-173)
                S diff;
                if (sizeof(S) == 8 && f_cs) diff = (S)(((double)lp[k] - su[k]) - (double)base[k]);
                else diff = lp[k] - base[k];
                S tp, tn;
                if (sizeof(S) == 8 && !f_pp) { tp = (S)d.pos_nom; tn = (S)d.neg_nom; }
                else { tp = (S)thp[k]; tn = (S)thn[k]; }
                // ON iff diff >= tp, OFF iff -diff >= tn (thresholds > 0): one magnitude, one threshold.
                // Results 0 / 1 / 2 of ATen's floor division without a branch (see div_floor_count)
                const bool neg = diff < (S)0;
                const S a = neg ? -diff : diff, b = neg ? tn : tp, b2 = b + b;
                const int ge1 = a >= b, ge2 = a >= b2;
                int32_t mag = ge1 + ge2;
                if (ge2 && !(a - b2 < b)) {                  // >= 3 events: rare
                    mag = div_floor_count<S>(a, b);
                    // before the clamps: the plan reports > iter_cap. Own pixels only (not the halo rows of a
                    // sharded centre-surround handle, nor the padding after the frame's last pixel)
                    if (i0 + k >= d.own_lo && i0 + k < d.own_hi) {
                        local_max = max(local_max, mag);
                        deep = 1;
                    }
                    if (mag > kRecMaxCount) mag = kRecMaxCount;
                }
                // shot noise: the exact test (below) only when the draw can possibly cross. Replay: shot_lo_f /
                // shot_hi_f are float32 bounds rounded outwards from shot_bound >= any per-pixel probability;
                // device RNG: the 12-bit prefix of the uniform decides (shot_candidate)
                if (shot_here) {
                    const bool wild = FT != V2E_U8 && !(xv >= 0.0 && xv <= 255.0);
                    if (RNG == 1) cand[k] = wild || shot_candidate(pref[k], p.pref_lo);
                    else cand[k] = wild || sr[k] < p.shot_lo_f || sr[k] > p.shot_hi_f;
                    shot_maybe |= cand[k];
                }
                recs[k] = (short)((neg ? -mag : mag) << kRecShift);
                mags[k] = mag;
                pols[k] = neg;
            }
            if (i0 + 4 > d.own_hi || i0 < d.own_lo) {      // the frame's last, partial quad; halo rows of a sharded handle
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (i0 + k >= d.own_hi || i0 + k < d.own_lo) { recs[k] = 0; mags[k] = 0; cand[k] = false; }
            }
            if (shot_maybe) {                              // rare
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const double xv = (FT == V2E_U8) ? (double)((codes >> (8 * k)) & 0xffu) : x[k];
                    if ((i0 + k) < d.n && cand[k]) {
                        const float r = RNG == 1 ? shot_uniform(d.seed, (g0 + k) >> 2, p.frame_index, (int)((g0 + k) & 3u), pref[k])
                                                 : sr[k];
                        const int flags = shot_flags(d, p.shot_c, xv, r, thp[k], thn[k]);
                        flg[k] = flags;
                        recs[k] = (short)(recs[k] | flags);
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < 4; k++) {
                local_max = max(local_max, mags[k]);
                mags[k] = min(mags[k], d.iter_cap);
                const uint32_t m = (uint32_t)(mags[k] > 0) | ((uint32_t)(mags[k] > 1) << 16);
                pk += m << (pols[k] ? 8 : 0);
                nact += recs[k] != 0;
            }
            if (!lp_done) st4((S *)d.lp_out, i0, lp);
            if (f_leak) st4((S *)d.base_out, i0, base);
            *(short4 *)(d.rec + i0) = make_short4(recs[0], recs[1], recs[2], recs[3]);
        }
        // per-(iteration,polarity) histogram. Iterations 0 and 1 (almost all events) are counted per thread,
        // reduced with one REDUX and accumulated in (warp-uniform) registers until the warp's last unit; a
        // pixel with >= 3 events takes the ballot loop, shot-noise flags their own (rare) path.
        if (__any_sync(0xffffffffu, nact != 0)) {
            const uint32_t wsum = __reduce_add_sync(0xffffffffu, pk);
            acc0 += wsum & 0x00ff00ffu;                     // ON:  iteration 0 | iteration 1 << 16
            acc1 += (wsum >> 8) & 0x00ff00ffu;              // OFF: iteration 0 | iteration 1 << 16
            if ((j & 255) == 255) flush_acc();              // 16-bit fields, <= 128 per unit
            // compaction of the active pixels into this block's list segment: warp scan, one shared
            // atomic per warp, no global round trip (the segment's place is fixed)
            int incl = nact;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            uint32_t wbase = 0;
            if (lane == 31) wbase = atomicAdd(&s_act_total, (uint32_t)incl);
            wbase = __shfl_sync(0xffffffffu, wbase, 31);
            if (nact) {
                uint32_t pos = seg_base + wbase + (uint32_t)(incl - nact);
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (recs[k] != 0) d.act_list[pos++] = (uint32_t)(i0 + k);
            }
            const unsigned shot_any = __ballot_sync(0xffffffffu, (flg[0] | flg[1] | flg[2] | flg[3]) != 0);
            if (shot_any) {
                int son = 0, soff = 0;
#pragma unroll
                for (int k = 0; k < 4; k++) { son += flg[k] & 1; soff += (flg[k] >> 1) & 1; }
                son = __reduce_add_sync(0xffffffffu, son);
                soff = __reduce_add_sync(0xffffffffu, soff);
                if (lane == 0) {
                    if (son) atomicAdd(&s_hist[kSegSmem], (uint32_t)son);
                    if (soff) atomicAdd(&s_hist[kSegSmem + 1], (uint32_t)soff);
                }
            }
            if (__any_sync(0xffffffffu, deep)) {
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int wmax = __reduce_max_sync(0xffffffffu, mags[k]);
                    for (int it = 2; it < wmax; it++) {
                        unsigned on = __ballot_sync(0xffffffffu, mags[k] > it && !pols[k]);
                        unsigned off = __ballot_sync(0xffffffffu, mags[k] > it && pols[k]);
                        if (lane == 0) {
                            if (on) { if (2 * it < kSegSmem) atomicAdd(&s_hist[2 * it], __popc(on)); else atomicAdd(&hist[2 * it], __popc(on)); }
                            if (off) { if (2 * it + 1 < kSegSmem) atomicAdd(&s_hist[2 * it + 1], __popc(off)); else atomicAdd(&hist[2 * it + 1], __popc(off)); }
                        }
                    }
                }
            }
        }
    }
    flush_acc();
    // block max -> one atomicMax per block
    local_max = warp_reduce_max(local_max);
    if (lane == 0 && local_max > 0) atomicMax(&s_max, local_max);
    __syncthreads();
    if (tid == 0 && s_max > 0) atomicMax(&c->max_n, s_max);
    if (tid == 0) d.act_count[(size_t)slot * d.n_blocks + blockIdx.x] = s_act_total;
    if (tid < kSegSmem && s_hist[tid]) atomicAdd(&hist[tid], s_hist[tid]);
    if (tid >= kSegSmem && tid < kSegSmem + 2 && s_hist[tid])
        atomicAdd(&hist[2 * d.iter_cap + (tid - kSegSmem)], s_hist[tid]);
    if (do_plan) {
        if (last_block(&c->done[0])) plan_frame(d, p, slot);
    }
}

// Warp-synchronous walk over the emitted iterations of "pixel k of every lane" (emulator.py:810-850).
// All 32 lanes must call it. For every iteration up to the warp's largest count, F(it, t, on, off,
// pass) receives the ballots of lanes whose event survives the refractory filter (ON / OFF) and this
// lane's own verdict. tm (timestamp_mem) is updated when the filter is active. Returns the number of
// surviving events of this lane's pixel.
template <typename F>
__device__ __forceinline__ int warp_walk(int mag, int pol, const TsParams &ts, bool filter, float refr_f,
                                         float &tm, F &&f) {
    const int wmax = __reduce_max_sync(0xffffffffu, mag);
    int fin = 0;
    for (int it = 0; it < wmax; it++) {
        const float t = linspace_f32(ts, it);
        bool pass = it < mag;
        if (filter && pass) {
            pass = (t - tm) > refr_f;              // pos_cord*ts[i] - timestamp_mem > refractory
            if (pass) tm = t;
        }
        const unsigned on = __ballot_sync(0xffffffffu, pass && !pol);
        const unsigned off = __ballot_sync(0xffffffffu, pass && pol);
        f(it, t, on, off, pass);
        fin += pass;
    }
    return fin;
}

// ---------------------------------------------------------------------------------------------
// filter-count kernel (only when refractory_period_s > 0): filtered histogram over the active-pixel
// list, no state writes
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
emu_filter_kernel(EmuDev d, FrameParams p, int slot, int do_plan) {
    __shared__ uint32_t s_hist[kSegSmem];
    if (*(volatile int32_t *)d.abort_flag) return;
    const int tid = threadIdx.x, lane = tid & 31;
    FrameCtrl *c = d.ctrl + slot;
    const int32_t max_n = *(volatile int32_t *)&c->max_n;
    const TsParams ts = make_ts(p, max_n, d.refr_d);
    if (!(ts.filter_active && max_n <= d.iter_cap)) {
        // nothing to filter: the update kernel's histogram is final (it completed before this kernel
        // started), so one block plans and everybody else leaves
        if (do_plan && blockIdx.x == 0) plan_frame(d, p, slot);
        return;
    }
    {
        if (tid < kSegSmem) s_hist[tid] = 0;
        __syncthreads();
        uint32_t *hist = d.hist_post + (size_t)slot * d.seg_stride;
        const uint32_t *seg_cnt = d.act_count + (size_t)slot * d.n_blocks;
        for (int sg = blockIdx.x; sg < d.n_blocks; sg += gridDim.x)
        for (uint32_t base = 0, n_act = seg_cnt[sg]; base < n_act; base += kThreads) {
            const uint32_t e = base + tid;
            int mag = 0, pol = 0;
            float tm = 0.f;
            if (e < n_act) {
                const uint32_t idx = d.act_list[(size_t)sg * d.seg_px + e];
                const int cnt = d.rec[idx] >> kRecShift;
                mag = cnt < 0 ? -cnt : cnt;
                pol = cnt < 0;
                if (mag) tm = d.tmem[idx];
            }
            warp_walk(mag, pol, ts, true, d.refr_f, tm, [&](int it, float, unsigned on, unsigned off, bool) {
                if (lane == 0) {
                    if (on) { if (2 * it < kSegSmem) atomicAdd(&s_hist[2 * it], __popc(on)); else atomicAdd(&hist[2 * it], __popc(on)); }
                    if (off) { if (2 * it + 1 < kSegSmem) atomicAdd(&s_hist[2 * it + 1], __popc(off)); else atomicAdd(&hist[2 * it + 1], __popc(off)); }
                }
            });
        }
        __syncthreads();
        if (tid < kSegSmem && s_hist[tid]) atomicAdd(&hist[tid], s_hist[tid]);
    }
    if (do_plan) {
        if (last_block(&c->done[1])) plan_frame(d, p, slot);
    }
}

// ---------------------------------------------------------------------------------------------
// shot-noise flag kernel for rng_mode 0 when the uniform field arrives after the counts
// ---------------------------------------------------------------------------------------------
template <int FT>
__global__ void __launch_bounds__(kThreads)
emu_shot_kernel(EmuDev d, FrameParams p, const void *frame, const float *shot_rand, int slot) {
    __shared__ uint32_t s_cnt[2];
    if (*(volatile int32_t *)d.abort_flag) return;
    const int tid = threadIdx.x;
    if (tid < 2) s_cnt[tid] = 0;
    __syncthreads();
    FrameCtrl *c = d.ctrl + slot;
    const int i0 = (blockIdx.x * kThreads + tid) * kVec;
    if (i0 < d.n) {
        double x[4];
        float sr[4], thp[4], thn[4];
        load_frame4<FT>(frame, i0, d.n, x);
        load_f32x4_any(shot_rand, i0, d.n, sr);
        if (d.per_pixel_thres) { ld4(d.pos_thres, i0, thp); ld4(d.neg_thres, i0, thn); }
        else {
#pragma unroll
            for (int k = 0; k < 4; k++) { thp[k] = (float)d.pos_nom; thn[k] = (float)d.neg_nom; }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (i0 + k >= d.own_hi || i0 + k < d.own_lo) continue;
            int flags = shot_flags(d, p.shot_c, x[k], sr[k], thp[k], thn[k]);
            if (flags) {
                const short old = d.rec[i0 + k];
                if (old == 0) {
                    // the update block that owns this pixel's unit: largest b with b*units/n_blocks <= unit
                    const int sg = (int)((((long long)((i0 + k) / kUnitPx) + 1) * d.n_blocks - 1) / d.units);
                    d.act_list[(size_t)sg * d.seg_px + atomicAdd(&d.act_count[(size_t)slot * d.n_blocks + sg], 1u)] =
                        (uint32_t)(i0 + k);
                }
                d.rec[i0 + k] = (short)(old | flags);
                if (flags & 1) atomicAdd(&s_cnt[0], 1u);
                if (flags & 2) atomicAdd(&s_cnt[1], 1u);
            }
        }
    }
    __syncthreads();
    uint32_t *hist = d.hist_pre + (size_t)slot * d.seg_stride;
    if (tid < 2 && s_cnt[tid]) atomicAdd(&hist[2 * d.iter_cap + tid], s_cnt[tid]);
    if (last_block(&c->done[2])) plan_frame(d, p, slot);
}

// ---------------------------------------------------------------------------------------------
// emit kernel: walks the active-pixel list, writes packed rows + state patch
// (emulator.py:810-870, 906-942, 1024-1059). Warp-ballot compaction: one shared-memory atomic per
// warp and (iteration, polarity) segment, one global atomic per block, chunk and segment.
// ---------------------------------------------------------------------------------------------
template <typename S>
__global__ void __launch_bounds__(kThreads)
emu_emit_kernel(EmuDev d, FrameParams p, int slot, float4 *events) {
    __shared__ uint32_t s_cnt[kSegSmem + 2];
    __shared__ uint32_t s_base[kSegSmem + 2];
    if (*(volatile int32_t *)d.abort_flag) return;
    const int tid = threadIdx.x, lane = tid & 31;
    const unsigned lt_mask = (1u << lane) - 1u;
    FrameCtrl *c = d.ctrl + slot;
    if (!c->planned) return;
    if (c->n_events == 0) return;
    const int32_t max_n = c->max_n;
    const TsParams ts = make_ts(p, max_n, d.refr_d);
    const bool filter = ts.filter_active && d.refr_on;
    const float ts_last = linspace_f32(ts, ts.steps - 1);
    const uint32_t *segoff = d.segoff + (size_t)slot * d.seg_stride;
    uint32_t *cursor = d.cursor + (size_t)slot * d.seg_stride;
    const uint64_t ev_base = c->ev_base;
    const uint32_t *seg_cnt = d.act_count + (size_t)slot * d.n_blocks;
    // lane 0 claims `count` consecutive rows of segment `seg` for this warp
    auto claim = [&](int seg_smem, int seg, unsigned count) -> uint32_t {
        if (seg_smem >= 0) return s_base[seg_smem] + atomicAdd(&s_cnt[seg_smem], count);
        return segoff[seg] + atomicAdd(&cursor[seg], count);
    };
    for (int sg = blockIdx.x; sg < d.n_blocks; sg += gridDim.x)
    for (uint32_t base = 0, n_act = seg_cnt[sg]; base < n_act; base += kThreads) {
        if (tid < kSegSmem + 2) s_cnt[tid] = 0;
        __syncthreads();
        const uint32_t e = base + tid;
        int idx = 0, mag = 0, pol = 0, flags = 0;
        float tm0 = 0.f, th = 0.f;
        S b0 = (S)0, lpv = (S)0;
        if (e < n_act) {
            idx = (int)d.act_list[(size_t)sg * d.seg_px + e];
            const int r = d.rec[idx];
            const int cnt = r >> kRecShift;
            flags = r & 3;
            mag = cnt < 0 ? -cnt : cnt;
            pol = cnt < 0;
            // everything the patch may need, issued together so the loads overlap
            if (filter && mag) tm0 = d.tmem[idx];
            th = pol ? (d.per_pixel_thres ? d.neg_thres[idx] : (float)d.neg_nom)
                     : (d.per_pixel_thres ? d.pos_thres[idx] : (float)d.pos_nom);
            b0 = ((const S *)d.base)[idx];
            if (flags) lpv = ((const S *)d.lp)[idx];
        }
        // pass 1: block-level counts per segment
        {
            float tm = tm0;
            warp_walk(mag, pol, ts, filter, d.refr_f, tm, [&](int it, float, unsigned on, unsigned off, bool) {
                if (lane == 0) {
                    if (on && 2 * it < kSegSmem) atomicAdd(&s_cnt[2 * it], __popc(on));
                    if (off && 2 * it + 1 < kSegSmem) atomicAdd(&s_cnt[2 * it + 1], __popc(off));
                }
            });
            const unsigned son = __ballot_sync(0xffffffffu, flags & 1), soff = __ballot_sync(0xffffffffu, flags & 2);
            if (lane == 0) {
                if (son) atomicAdd(&s_cnt[kSegSmem], __popc(son));
                if (soff) atomicAdd(&s_cnt[kSegSmem + 1], __popc(soff));
            }
        }
        __syncthreads();
        if (tid < kSegSmem + 2) {
            const uint32_t n = s_cnt[tid];
            if (n) {
                const int seg = tid < kSegSmem ? tid : 2 * d.iter_cap + (tid - kSegSmem);
                s_base[tid] = segoff[seg] + atomicAdd(&cursor[seg], n);
            }
            s_cnt[tid] = 0;
        }
        __syncthreads();
        // pass 2: write rows, patch state
        {
            const float fx = (float)(idx % d.W), fy = (float)(idx / d.W);
            const float pv = pol ? -1.0f : 1.0f;
            float tm = tm0;
            const int fin = warp_walk(mag, pol, ts, filter, d.refr_f, tm,
                                      [&](int it, float t, unsigned on, unsigned off, bool pass) {
                uint32_t b_on = 0, b_off = 0;
                if (lane == 0) {
                    if (on) b_on = claim(2 * it < kSegSmem ? 2 * it : -1, 2 * it, __popc(on));
                    if (off) b_off = claim(2 * it + 1 < kSegSmem ? 2 * it + 1 : -1, 2 * it + 1, __popc(off));
                }
                b_on = __shfl_sync(0xffffffffu, b_on, 0);
                b_off = __shfl_sync(0xffffffffu, b_off, 0);
                if (pass) {
                    const uint64_t row = ev_base + (pol ? b_off + __popc(off & lt_mask) : b_on + __popc(on & lt_mask));
                    events[row] = make_float4(t, fx, fy, pv);
                }
            });
            if (filter && fin) d.tmem[idx] = tm;
            if (fin || flags) {
                S b = b0;
                const float prod = (float)fin * th;      // int32*float32 -> float32 (emulator.py:936-937)
                if (pol) b = b - (S)prod; else b = b + (S)prod;
                if (flags) b = lpv;                      // emulator.py:940-942
                ((S *)d.base)[idx] = b;
            }
            const unsigned son = __ballot_sync(0xffffffffu, flags & 1), soff = __ballot_sync(0xffffffffu, flags & 2);
            if (son | soff) {
                uint32_t b_on = 0, b_off = 0;
                if (lane == 0) {
                    if (son) b_on = claim(kSegSmem, 0, __popc(son));
                    if (soff) b_off = claim(kSegSmem + 1, 0, __popc(soff));
                }
                b_on = __shfl_sync(0xffffffffu, b_on, 0);
                b_off = __shfl_sync(0xffffffffu, b_off, 0);
                if (flags & 1) events[ev_base + b_on + __popc(son & lt_mask)] = make_float4(ts_last, fx, fy, 1.0f);
                if (flags & 2) events[ev_base + b_off + __popc(soff & lt_mask)] = make_float4(ts_last, fx, fy, -1.0f);
            }
        }
        __syncthreads();
    }
}


// =============================================================================================
// Fused multi-frame path (v2e_emu_step with T >= 2 frames, uint8 frames, plain pixel model, device RNG or no
// per-frame noise).
//
// The only frame-global quantity of the model is max_num_events_any_pixel (emulator.py:773-775): it sets the
// timestamps of the frame and decides whether the refractory filter runs at all (refractory_period_s > dt / max_n,
// emulator.py:830). Whenever the filter does NOT run, everything a pixel does is local: its event count is
// floor(|lp - base| / theta), its base moves by count * theta, timestamp_mem is not touched. So:
//   pass 1 (emu_fused_update_kernel): a thread keeps lp / base / thresholds / noise rate of its 4 pixels in
//           REGISTERS across all T frames, reads one byte per pixel and frame (prefetched 4 frames ahead), and
//           appends a 16-bit record (pixel, polarity, count, shot flags) per active pixel and frame to the list
//           segment of its (frame, 128-pixel unit). New state goes to alternate arrays.
//   pass 2 (emu_fused_count_kernel): walks the (sparse) records: per-frame (iteration, polarity) histogram and
//           frame maximum.
//   plan   (emu_fused_plan_kernel): per frame, checks the assumption (filter inactive, max_n small enough for the
//           record) and lays out the iteration-major rows of all T frames; if any frame breaks the assumption the
//           chunk is REJECTED: nothing is emitted or committed, and the caller replays the chunk frame by frame from
//           the untouched state (v2e_emu_collect does that itself for v2e_emu_step).
//   emit   (emu_fused_emit_kernel): records -> packed rows with the frame's linspace timestamps.
//   commit (emu_fused_commit_kernel): alternate lp / base -> the handle's state.
// Arithmetic per pixel and frame is the update + emit kernels' (same operations in the same order), so the rows,
// counters and state equal the per-frame path's bit for bit (tests/test_emulator_gpu.py).
// =============================================================================================
struct FusedFrame {                     // what pass 1 needs of one frame
    double eps_scale, shot_c;
    float dt_f;
    uint32_t frame_index, pref_lo, pad;
};
static_assert(sizeof(FusedFrame) == 32, "FusedFrame layout");
constexpr int kFusedGroup = 64;                     // 128-pixel units per block of the count / emit kernels
constexpr int kFusedMaxN = 31;                      // largest per-frame maximum the fused plan accepts
constexpr int kFusedFallback = 100;                 // abort_flag value: chunk rejected (internal)
constexpr int kBlkSeg = kSegSmem + 2;
// record: bits 0-6 pixel within the unit, 7 polarity (1 = OFF), 8-9 shot flags, 10-15 event count (clamped to 63)
__device__ __forceinline__ uint32_t make_rec16(int px_local, int neg, int flags, int mag) {
    return (uint32_t)px_local | ((uint32_t)neg << 7) | ((uint32_t)flags << 8) | ((uint32_t)(mag > 63 ? 63 : mag) << 10);
}

// rare paths of pass 1, kept out of line so that the frame loop stays small (instruction cache)
template <typename S>
__device__ __noinline__ int32_t fused_deep_count(S a, S b) {
    int32_t mag = div_floor_count<S>(a, b);
    return mag > kRecMaxCount ? kRecMaxCount : mag;
}
// (scalar arguments: a reference to the kernel-parameter struct would force a copy of it into local memory)
__device__ __noinline__ int fused_shot_flags(uint64_t seed, double shot_inten_m1, int per_pixel_thres, double pos_nom,
                                             double neg_nom, double shot_c, uint32_t gpx, uint32_t frame_index,
                                             uint32_t pref, int code, float thp, float thn) {
    const float r = shot_uniform(seed, gpx >> 2, frame_index, (int)(gpx & 3u), pref);
    EmuDev dd;
    dd.shot_inten_m1 = shot_inten_m1;
    dd.per_pixel_thres = per_pixel_thres;
    dd.pos_nom = pos_nom;
    dd.neg_nom = neg_nom;
    return shot_flags(dd, shot_c, (double)code, r, thp, thn);
}

// frame bytes of a quad that is not 4-byte aligned in its frame, or crosses the end of the frame
__device__ __noinline__ uint32_t fused_load_codes_slow(const uint8_t *pf, int valid) {
    uint32_t v = 0;
    for (int k = 0; k < valid; k++) v |= (uint32_t)pf[k] << (8 * k);
    return v;
}

// WARPS warps per block, MINB blocks per SM: the register budget / occupancy / tail trade-off is picked on the host
// (launch_fused_update). Units are dealt evenly to blocks and, inside a block, to warps.
template <typename S, bool FAST, int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB)
emu_fused_update_kernel(EmuDev d, const FusedFrame *__restrict__ ff, const uint8_t *__restrict__ frames, int T,
                        S *__restrict__ lp_out, S *__restrict__ base_out, uint16_t *__restrict__ rec_list,
                        uint32_t *__restrict__ rec_cnt) {
    const bool f_pp = FAST || d.per_pixel_thres, f_leak = FAST || d.leak_on, f_shot = FAST || d.shot_on;
    constexpr bool f_lp = sizeof(S) == 8;        // no hdr here: float64 state <=> the low-pass is on
    extern __shared__ __align__(16) unsigned char s_dyn[];
    const FusedFrame *s_ff = (const FusedFrame *)s_dyn;
    __shared__ double2 s_tab[256];               // x: lin_log(code) (float32 value widened), y: inten01(code) =
                                                 // (code + 20) / 275 (emulator_utils.py:48-54)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    {
        const uint4 *src = (const uint4 *)ff;
        uint4 *dst = (uint4 *)s_dyn;
        for (int i = tid; i < T * 2; i += WARPS * 32) dst[i] = src[i];
        for (int i = tid; i < 256; i += WARPS * 32) s_tab[i] = make_double2((double)d.lut[i], ((double)i + 20.0) / 275.0);
    }
    __syncthreads();
    if (*(volatile int32_t *)d.abort_flag) return;
    const int u0 = (int)(((long long)blockIdx.x * d.units) / gridDim.x);
    const int u1 = (int)(((long long)(blockIdx.x + 1) * d.units) / gridDim.x);
    const size_t n = (size_t)d.n;
    const bool use_rng = (f_leak || f_shot) && d.rng_mode == 1;
    const S tp_nom = (S)d.pos_nom, tn_nom = (S)d.neg_nom;
    // every frame's row of bytes at a quad is 4-byte aligned iff the frame size is a multiple of 4 (and the base is)
    const bool al = ((n & 3) == 0) && ((((uintptr_t)frames) & 3) == 0);
    for (int unit = u0 + warp; unit < u1; unit += WARPS) {
        const int i0 = unit * kUnitPx + lane * kVec;
        const int valid = i0 < d.n ? min(4, d.n - i0) : 0;          // pixels of this quad inside the frame
        const uint8_t *pf0 = frames + i0;
        auto load_codes = [&](int f) -> uint32_t {
            const uint8_t *pf = pf0 + (size_t)f * n;
            if (al && valid == 4) return __ldg((const uint32_t *)pf);
            return fused_load_codes_slow(pf, valid);
        };
        // the next frame's bytes are requested before this frame's arithmetic: a frame takes a warp thousands of
        // cycles, one frame of look-ahead hides the load
        uint32_t c_next = load_codes(0);
        // per-pixel state -> registers for the whole chunk
        S lp[4] = {(S)0, (S)0, (S)0, (S)0}, base[4] = {(S)0, (S)0, (S)0, (S)0};
        float thp[4], thn[4], lnr[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < 4; k++) { thp[k] = (float)d.pos_nom; thn[k] = (float)d.neg_nom; }
        if (valid) {
            if (f_lp) ld4((const S *)d.lp, i0, lp);
            ld4((const S *)d.base, i0, base);
            if (f_pp) { ld4(d.pos_thres, i0, thp); ld4(d.neg_thres, i0, thn); }
            if (f_leak) {
                ld4(d.noise_rate, i0, lnr);
#pragma unroll
                for (int k = 0; k < 4; k++) lnr[k] = d.leak_rate_f * lnr[k];      // emulator_utils.py:127, float32 product
            }
        }
        const uint32_t g0 = (uint32_t)i0 + d.px_off;
        uint16_t *seg = rec_list + (size_t)unit * kUnitPx;               // + f * units * kUnitPx per frame
        uint32_t *cntp = rec_cnt + unit;
        const size_t seg_stride = (size_t)d.units * kUnitPx;
#pragma unroll 1
        for (int f = 0; f < T; f++) {
            const uint32_t codes = c_next;
            if (f + 1 < T) c_next = load_codes(f + 1);
            const double eps_scale = s_ff[f].eps_scale;
            const float dt_f = s_ff[f].dt_f;
            const uint32_t frame_index = s_ff[f].frame_index, pref_lo = s_ff[f].pref_lo;
            uint32_t r16[4];
            float lr[4] = {0.f, 0.f, 0.f, 0.f};
            uint32_t pref[4] = {0u, 0u, 0u, 0u};
            if (use_rng) noise_px4(d.seed, g0, frame_index, lr, pref);
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int code = (int)((codes >> (8 * k)) & 0xffu);
                // photoreceptor low-pass (emulator_utils.py:57-109)
                const double2 tb = s_tab[code];
                if (f_lp) {
                    const double eps = fmin(tb.y * eps_scale, 1.0);             // clamp(max=1), eps is never NaN
                    lp[k] = (S)((1.0 - eps) * (double)lp[k] + eps * tb.x);
                } else {
                    lp[k] = (S)tb.x;
                }
                // leak (emulator_utils.py:114-134): float32 products, subtract in S
                if (f_leak) {
                    const float rate = lnr[k] * (1.0f - d.leak_jit_f * lr[k]);
                    const float delta = (dt_f * rate) * thp[k];
                    base[k] = base[k] - (S)delta;
                }
                // difference and event count (emulator.py:748-772, emulator_utils.py:137-173)
                const S diff = lp[k] - base[k];
                const bool neg = diff < (S)0;
                const float thf = neg ? thn[k] : thp[k];
                S b;
                if (sizeof(S) == 8 && !f_pp) b = neg ? tn_nom : tp_nom;
                else b = (S)thf;
                const S a = neg ? -diff : diff, b2 = b + b;
                const int ge2 = a >= b2;
                int32_t mag = (int)(a >= b) + ge2;
                if (ge2 && !(a - b2 < b)) mag = fused_deep_count<S>(a, b);          // >= 3 events: rare
                int flags = 0;
                if (f_shot && shot_candidate(pref[k], pref_lo))                        // rare
                    flags = fused_shot_flags(d.seed, d.shot_inten_m1, d.per_pixel_thres, d.pos_nom, d.neg_nom,
                                             s_ff[f].shot_c, g0 + k, frame_index, pref[k], code, thp[k], thn[k]);
                if (k >= valid) { mag = 0; flags = 0; }
                // the refractory filter does not run (checked by the plan): every event is emitted
                // (emulator.py:936-942: int32 * float32 -> float32, then the state's dtype). Selects, not
                // branches: x + 0.0 would turn a -0.0 into +0.0
                const S prod = (S)((float)mag * thf);
                const S moved = base[k] + (neg ? -prod : prod);          // x - p == x + (-p) exactly
                S bb = mag ? moved : base[k];
                bb = flags ? lp[k] : bb;
                base[k] = bb;
                r16[k] = (mag | flags) ? make_rec16(lane * kVec + k, neg, flags, mag) : 0u;      // active => non-zero
            }
            // compaction of this frame's active pixels into the (frame, unit) list segment
            uint32_t cnt = 0;
            if (__any_sync(0xffffffffu, (r16[0] | r16[1] | r16[2] | r16[3]) != 0u)) {
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const unsigned m = __ballot_sync(0xffffffffu, r16[k] != 0u);
                    if (r16[k]) seg[cnt + __popc(m & lt_mask)] = (uint16_t)r16[k];
                    cnt += __popc(m);
                }
            }
            if (lane == 0) *cntp = cnt;
            seg += seg_stride;
            cntp += d.units;
        }
        if (valid) {
            st4(lp_out, i0, lp);
            st4(base_out, i0, base);
        }
    }
}

// the records of up to 8 consecutive units of one frame as one list: off[k] = first list position of unit k
struct FusedWarpList {
    uint32_t off[9];
    uint32_t total;
    // unit of list position i and that unit's first position (selects: no dynamically indexed array)
    __device__ __forceinline__ int unit_of(uint32_t i, uint32_t &first) const {
        int k = 0;
        first = off[0];
#pragma unroll
        for (int m = 1; m < 8; m++)
            if (i >= off[m]) { k = m; first = off[m]; }
        return k;
    }
};
__device__ __forceinline__ void fused_warp_list(FusedWarpList &wl, const uint32_t *cnt, int nu, int lane) {
    uint32_t c = lane < nu ? cnt[lane] : 0u;
    uint32_t incl = c;
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    const uint32_t excl = incl - c;
#pragma unroll
    for (int m = 0; m < 8; m++) wl.off[m] = __shfl_sync(0xffffffffu, excl, m);
    wl.off[8] = wl.total = __shfl_sync(0xffffffffu, incl, 7);
}

// pass 2: histogram per (iteration, polarity) and maximum per frame from the records. Block = (frame, group of
// kFusedGroup units). The block's own per-segment counts are kept for the emit kernel (blk_cnt).
__global__ void __launch_bounds__(kThreads)
emu_fused_count_kernel(EmuDev d, int T, int groups, const uint16_t *__restrict__ rec_list,
                       const uint32_t *__restrict__ rec_cnt, uint32_t *__restrict__ blk_cnt) {
    __shared__ uint32_t s_hist[kBlkSeg];
    __shared__ int s_max;
    if (*(volatile int32_t *)d.abort_flag) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int f = blockIdx.x / groups, g = blockIdx.x - f * groups;
    if (tid < kBlkSeg) s_hist[tid] = 0;
    if (tid == 0) s_max = 0;
    __syncthreads();
    uint32_t *hist = d.hist_pre + (size_t)f * d.seg_stride;
    const int ue = min(d.units, (g + 1) * kFusedGroup);
    int local_max = 0;
    // a warp takes 8 consecutive units and walks their records as ONE list (a unit holds ~13 records at 0.1
    // events/px/frame: unit by unit two thirds of the lanes would idle)
    for (int ub = g * kFusedGroup + warp * 8; ub < ue; ub += kWarps * 8) {
        const int nu = min(8, ue - ub);
        FusedWarpList wl;
        fused_warp_list(wl, rec_cnt + (size_t)f * d.units + ub, nu, lane);
        for (uint32_t i0 = 0; i0 < wl.total; i0 += 32) {
            const uint32_t i = i0 + lane;
            uint32_t r = 0u;
            if (i < wl.total) {
                uint32_t first;
                const int k = wl.unit_of(i, first);
                r = (uint32_t)rec_list[((size_t)f * d.units + ub + k) * kUnitPx + (i - first)];
            }
            const int mag = (int)(r >> 10), neg = (int)((r >> 7) & 1u), flags = (int)((r >> 8) & 3u);
            local_max = max(local_max, mag);
            const int magc = min(mag, d.iter_cap);
            const int wmax = __reduce_max_sync(0xffffffffu, magc);
            for (int it = 0; it < wmax; it++) {
                const unsigned on = __ballot_sync(0xffffffffu, it < magc && !neg);
                const unsigned off = __ballot_sync(0xffffffffu, it < magc && neg);
                if (lane == 0) {
                    if (on) { if (2 * it < kSegSmem) atomicAdd(&s_hist[2 * it], __popc(on)); else atomicAdd(&hist[2 * it], __popc(on)); }
                    if (off) { if (2 * it + 1 < kSegSmem) atomicAdd(&s_hist[2 * it + 1], __popc(off)); else atomicAdd(&hist[2 * it + 1], __popc(off)); }
                }
            }
            const unsigned son = __ballot_sync(0xffffffffu, flags & 1), soff = __ballot_sync(0xffffffffu, flags & 2);
            if (lane == 0) {
                if (son) atomicAdd(&s_hist[kSegSmem], __popc(son));
                if (soff) atomicAdd(&s_hist[kSegSmem + 1], __popc(soff));
            }
        }
    }
    local_max = warp_reduce_max(local_max);
    if (lane == 0 && local_max > 0) atomicMax(&s_max, local_max);
    __syncthreads();
    if (tid == 0 && s_max > 0) atomicMax(&d.ctrl[f].max_n, s_max);
    if (tid < kBlkSeg) {
        const uint32_t v = s_hist[tid];
        blk_cnt[(size_t)blockIdx.x * kBlkSeg + tid] = v;
        if (v) atomicAdd(&hist[tid < kSegSmem ? tid : 2 * d.iter_cap + (tid - kSegSmem)], v);
    }
}

// plan of all T frames: one block. max_vec (nullable): the frame maxima reduced over the ranks of a pixel-sharded clip.
__global__ void __launch_bounds__(kThreads)
emu_fused_plan_kernel(EmuDev d, const FrameParams *__restrict__ fp, int T, uint64_t ev_base_start, uint64_t capacity,
                      const int32_t *__restrict__ max_vec, int slot0, int chain) {
    extern __shared__ uint32_t s_tot[];          // [T] rows of each frame
    __shared__ int s_bad;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_bad = 0x7fffffff;
    __syncthreads();
    for (int f = warp; f < T; f += kWarps) {
        FrameCtrl *c = d.ctrl + f;
        int32_t max_n = max_vec ? max_vec[f] : *(volatile int32_t *)&c->max_n;
        const FrameParams p = fp[f];
        bool bad = max_n > kFusedMaxN || max_n > d.iter_cap;
        if (d.refr_on && max_n > 0 && d.refr_d > p.dt / (double)max_n) bad = true;    // emulator.py:792, 830
        const uint32_t *h = d.hist_pre + (size_t)f * d.seg_stride;
        uint32_t *off = d.segoff + (size_t)f * d.seg_stride;
        const int nseg = bad ? 0 : 2 * max_n;
        const int s0 = 2 * lane, s1 = 2 * lane + 1;
        const uint32_t v0 = s0 < nseg ? h[s0] : 0u, v1 = s1 < nseg ? h[s1] : 0u;
        uint32_t incl = v0 + v1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        const uint32_t excl = incl - (v0 + v1);
        if (s0 < nseg) off[s0] = excl;
        if (s1 < nseg) off[s1] = excl + v0;
        const uint32_t sig = __shfl_sync(0xffffffffu, incl, 31);
        const uint32_t sig_on = __reduce_add_sync(0xffffffffu, v0);
        if (lane == 0) {
            const uint32_t shot_on = h[2 * d.iter_cap], shot_off = h[2 * d.iter_cap + 1];
            off[2 * d.iter_cap] = sig;
            off[2 * d.iter_cap + 1] = sig + shot_on;
            const uint32_t total = sig + shot_on + shot_off;
            c->max_n = max_n;
            c->filter_active = 0;
            c->n_on = sig_on + shot_on;
            c->n_off = (sig - sig_on) + shot_off;
            c->n_shot_on = shot_on;
            c->n_shot_off = shot_off;
            c->n_events = total;
            s_tot[f] = total;
            if (bad) atomicMin(&s_bad, f);
        }
    }
    __syncthreads();
    if (tid == 0 && !*(volatile int32_t *)d.abort_flag) {
        // d is shifted to the segment's first frame (slot0 of the step); a segment after the first continues at the
        // row the previous segment / frame of the step ended at
        uint64_t base = chain ? (uint64_t)*d.chain_base : ev_base_start;
        for (int f = 0; f < T; f++) {
            d.ctrl[f].ev_base = base;
            base += s_tot[f];
        }
        d.ctrl[T].ev_base = base;
        if (s_bad != 0x7fffffff) {
            if (atomicCAS(d.abort_flag, 0, kFusedFallback) == 0) d.abort_flag[1] = slot0 + s_bad;
        } else if (base > capacity) {
            if (atomicCAS(d.abort_flag, 0, V2E_E_CAPACITY) == 0) d.abort_flag[1] = slot0;
        } else {
            for (int f = 0; f < T; f++) d.ctrl[f].planned = 1;
            *d.chain_base = base;
        }
        __threadfence();
    }
}

__global__ void __launch_bounds__(kThreads)
emu_fused_emit_kernel(EmuDev d, const FrameParams *__restrict__ fp, int T, int groups,
                      const uint16_t *__restrict__ rec_list, const uint32_t *__restrict__ rec_cnt,
                      const uint32_t *__restrict__ blk_cnt, float4 *__restrict__ events) {
    __shared__ uint32_t s_cnt[kBlkSeg];
    __shared__ uint32_t s_base[kBlkSeg];
    if (*(volatile int32_t *)d.abort_flag) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int f = blockIdx.x / groups, g = blockIdx.x - f * groups;
    const FrameCtrl *c = d.ctrl + f;
    if (!c->planned || c->n_events == 0) return;
    const TsParams ts = make_ts(fp[f], c->max_n, d.refr_d);
    const float ts_last = linspace_f32(ts, ts.steps - 1);
    const uint32_t *segoff = d.segoff + (size_t)f * d.seg_stride;
    uint32_t *cursor = d.cursor + (size_t)f * d.seg_stride;
    const uint64_t ev_base = c->ev_base;
    if (tid < kBlkSeg) {
        const uint32_t nb = blk_cnt[(size_t)blockIdx.x * kBlkSeg + tid];
        s_cnt[tid] = 0;
        if (nb) {
            const int seg = tid < kSegSmem ? tid : 2 * d.iter_cap + (tid - kSegSmem);
            s_base[tid] = segoff[seg] + atomicAdd(&cursor[seg], nb);
        }
    }
    __syncthreads();
    auto claim = [&](int seg_smem, int seg, unsigned count) -> uint32_t {
        if (seg_smem >= 0) return s_base[seg_smem] + atomicAdd(&s_cnt[seg_smem], count);
        return segoff[seg] + atomicAdd(&cursor[seg], count);
    };
    const int ue = min(d.units, (g + 1) * kFusedGroup);
    for (int ub = g * kFusedGroup + warp * 8; ub < ue; ub += kWarps * 8) {
        const int nu = min(8, ue - ub);
        FusedWarpList wl;
        fused_warp_list(wl, rec_cnt + (size_t)f * d.units + ub, nu, lane);
        for (uint32_t i0 = 0; i0 < wl.total; i0 += 32) {
            const uint32_t i = i0 + lane;
            uint32_t r = 0u;
            int k = 0;
            if (i < wl.total) {
                uint32_t first;
                k = wl.unit_of(i, first);
                r = (uint32_t)rec_list[((size_t)f * d.units + ub + k) * kUnitPx + (i - first)];
            }
            const int mag = (int)(r >> 10), neg = (int)((r >> 7) & 1u), flags = (int)((r >> 8) & 3u);
            const int idx = (ub + k) * kUnitPx + (int)(r & 127u);
            const float fx = (float)(idx % d.W), fy = (float)(idx / d.W);
            const float pv = neg ? -1.0f : 1.0f;
            const int wmax = __reduce_max_sync(0xffffffffu, mag);
            for (int it = 0; it < wmax; it++) {
                const float t = linspace_f32(ts, it);
                const bool pass = it < mag;
                const unsigned on = __ballot_sync(0xffffffffu, pass && !neg);
                const unsigned off = __ballot_sync(0xffffffffu, pass && neg);
                uint32_t b_on = 0, b_off = 0;
                if (lane == 0) {
                    if (on) b_on = claim(2 * it < kSegSmem ? 2 * it : -1, 2 * it, __popc(on));
                    if (off) b_off = claim(2 * it + 1 < kSegSmem ? 2 * it + 1 : -1, 2 * it + 1, __popc(off));
                }
                b_on = __shfl_sync(0xffffffffu, b_on, 0);
                b_off = __shfl_sync(0xffffffffu, b_off, 0);
                if (pass) {
                    const uint64_t row = ev_base + (neg ? b_off + __popc(off & lt_mask) : b_on + __popc(on & lt_mask));
                    events[row] = make_float4(t, fx, fy, pv);
                }
            }
            const unsigned son = __ballot_sync(0xffffffffu, flags & 1), soff = __ballot_sync(0xffffffffu, flags & 2);
            if (son | soff) {
                uint32_t b_on = 0, b_off = 0;
                if (lane == 0) {
                    if (son) b_on = claim(kSegSmem, 0, __popc(son));
                    if (soff) b_off = claim(kSegSmem + 1, 0, __popc(soff));
                }
                b_on = __shfl_sync(0xffffffffu, b_on, 0);
                b_off = __shfl_sync(0xffffffffu, b_off, 0);
                if (flags & 1) events[ev_base + b_on + __popc(son & lt_mask)] = make_float4(ts_last, fx, fy, 1.0f);
                if (flags & 2) events[ev_base + b_off + __popc(soff & lt_mask)] = make_float4(ts_last, fx, fy, -1.0f);
            }
        }
    }
}

// accepted chunk: the alternate lp / base arrays become the state
__global__ void __launch_bounds__(kThreads)
emu_fused_commit_kernel(EmuDev d, const uint4 *__restrict__ lp_alt, const uint4 *__restrict__ base_alt, size_t n16) {
    if (*(volatile int32_t *)d.abort_flag) return;
    uint4 *lp = (uint4 *)d.lp, *base = (uint4 *)d.base;
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n16; i += (size_t)gridDim.x * kThreads) {
        lp[i] = lp_alt[i];
        base[i] = base_alt[i];
    }
}

// measurement floor: what an event bracket reports around a kernel that does nothing (v2e_emu_profile_read4)
__global__ void emu_null_kernel() {}

__global__ void emu_begin_step_kernel(EmuDev d, int slot, uint64_t ev_base) {
    d.ctrl[slot].ev_base = ev_base;
}
// the frame-by-frame kernels continue where a multi-frame chunk of the same step stopped writing
__global__ void emu_chain_step_kernel(EmuDev d, int slot) {
    d.ctrl[slot].ev_base = *d.chain_base;
}

__global__ void __launch_bounds__(kThreads) emu_plan_kernel(EmuDev d, FrameParams p, int slot) {
    plan_frame(d, p, slot);
}

}  // namespace

// =============================================================================================
// host side
// =============================================================================================
constexpr int kProfKinds = 4;            // update, filter, emit, null kernel (bracket floor)
struct V2eEmu {
    V2eEmuCfg cfg;
    EmuDev d;
    int first_done;
    int last_T;
    uint32_t frame_counter;     // frames counted so far (Philox counter word, rng_mode 1)
    uint32_t step_base;         // frame_counter at the start of the current step
    double last_dt;             // delta_time of the last single-frame phase_count
    double min_thres;           // smallest per-pixel threshold uploaded by v2e_emu_set_fields
    int profile;                // 1: bracket every kernel of v2e_emu_step with CUDA events
    cudaEvent_t *ev;            // [max_slots][3 kinds][2]
    int prof_frames;
    unsigned char *prof_used;   // [max_slots][kProfKinds]
    float *lut_dev;
    // optional models: per-frame inputs of the next step / phase_count (v2e_emu_set_pr_noise)
    const float *pr_randn_dev;  // [T][H*W] or null (device RNG)
    double *pr_vrms;            // [max_slots]
    int pr_T;                   // frames covered by pr_vrms (0: not set)
    int pr_T_last;              // what the last step consumed (a resume_emit step re-counts its later frames)
    int scidvs_started;         // scidvs_highpass exists (emulator.py:720-722)
    FrameCtrl *ctrl_host;       // pinned
    int32_t *abort_host;        // pinned [2]
    size_t state_elem;
    // fused multi-frame path (allocated on first use)
    int fused_enable;           // v2e_emu_set_option(h, 0, x)
    int fused_max_T;            // frames per fused chunk the record lists hold (0: not allocated)
    void *lp_alt, *base_alt;    // where pass 1 stores the new state until the chunk is accepted
    uint16_t *rec_list;         // [fused_max_T][units][128]
    uint32_t *rec_cnt;          // [fused_max_T][units]
    uint32_t *blk_cnt;          // [fused_max_T * groups][kBlkSeg]
    FusedFrame *ff_dev;         // [max_slots]
    FrameParams *fp_dev;        // [max_slots]
    int32_t *max_vec;           // [max_slots] frame maxima, contiguous (all-reduced over ranks when sharded)
    int last_fused;             // the last step went through the fused path: 1 = v2e_emu_step, 2 = phase functions
    int fused_T;                // (phase functions) frames of that step the fused kernels covered
    // schedule of the last v2e_emu_step: segments of frames [a, b), kind 0 = multi-frame kernels, 1 = frame by frame
    struct Seg { int kind, a, b; } *sched;
    int n_seg;
    struct {                    // arguments of that step, for the frame-by-frame replay of a rejected chunk
        const void *frames; int dtype, T; double t_previous; float *events; uint64_t capacity, ev_base_start;
        double *t_frames;       // [max_slots]
    } ls;
    long long n_fused_chunks, n_fused_rejected;
    int last_reject_frame, last_reject_max_n;      // diagnostics: where and why the last chunk was rejected
    long long n_frames_multi, n_frames_single;     // frames of scheduled steps that ended up in multi-frame / single-frame segments
    int fused_skip, fused_penalty;                 // back-off: chunks to run frame by frame before the next attempt
    // pixel-sharded centre-surround model: plan of the current frame (v2e_emu_cs_begin) and the exchange buffers
    int cs_K;                   // halo rows = Euler steps per chunk (0: not sharded)
    double *cs_send, *cs_recv;  // [2][K][W]
    int cs_num_steps;
    double cs_alpha_p; float cs_alpha_h;
    FrameParams cs_p;
    int cs_pending;             // v2e_emu_cs_begin ran, v2e_emu_cs_update not yet
};

thread_local char g_err[512] = "";
static int fail(int code, const char *fmt, const char *detail = "") {
    snprintf(g_err, sizeof(g_err), fmt, detail);
    return code;
}
#define CU(call)                                                            \
    do {                                                                    \
        cudaError_t e_ = (call);                                            \
        if (e_ != cudaSuccess) return fail(V2E_E_CUDA, #call ": %s", cudaGetErrorString(e_)); \
    } while (0)

int v2e_set_error(int code, const char *fmt, const char *detail) { return fail(code, fmt, detail); }
extern "C" const char *v2e_last_error(void) { return g_err; }
extern "C" int v2e_version(void) { return 200; }
extern "C" int v2e_abi_info(int *version, int *emu_cfg_size, int *frame_info_size, int *unet_weights_size) {
    if (version) *version = 200;
    if (emu_cfg_size) *emu_cfg_size = (int)sizeof(V2eEmuCfg);
    if (frame_info_size) *frame_info_size = (int)sizeof(V2eFrameInfo);
    if (unet_weights_size) *unet_weights_size = (int)sizeof(V2eUNetWeights);
    return V2E_OK;
}

static FrameParams make_params(const V2eEmu *h, double t_frame, double t_prev, uint32_t frame_index,
                               uint64_t capacity) {
    FrameParams p;
    memset(&p, 0, sizeof(p));
    p.t_prev = t_prev;
    p.t_frame = t_frame;
    p.dt = t_frame - t_prev;                                    // emulator.py:656
    if (h->cfg.cutoff_hz > 0) {
        double tau = 1.0 / (M_PI * 2 * h->cfg.cutoff_hz);       // emulator_utils.py:80
        p.eps_scale = p.dt / tau;
    }
    p.dt_f = (float)p.dt;
    p.frame_index = frame_index;
    p.shot_c = (h->cfg.shot_noise_rate_hz / 2) * p.dt;
    {
        // probability = shot_c * ((f-1)*inten01 + 1) * nominal/threshold; for x >= 0 the intensity term
        // is <= max(1, f) on 0 <= x <= 255 and thresholds are clamped at 0.01 by the caller (emulator.py:464, 471)
        double inten_max = h->cfg.shot_inten_factor > 1 ? h->cfg.shot_inten_factor : 1.0;   // 0 <= x <= 255
        double pre_max = 1.0;
        if (h->cfg.per_pixel_thres) {
            double nom = h->cfg.pos_thres_nominal > h->cfg.neg_thres_nominal ? h->cfg.pos_thres_nominal
                                                                               : h->cfg.neg_thres_nominal;
            pre_max = nom / h->min_thres;
        }
        p.shot_bound = fabs(p.shot_c) * inten_max * pre_max * 1.0001 + 1e-300;
        // rounded outwards: (double)r < shot_bound implies r < shot_lo_f, (double)r > 1-shot_bound implies r > shot_hi_f
        float lo = (float)p.shot_bound;
        if ((double)lo < p.shot_bound) lo = nextafterf(lo, INFINITY);
        float hi = (float)(1.0 - p.shot_bound);
        if ((double)hi > 1.0 - p.shot_bound) hi = nextafterf(hi, -INFINITY);
        p.shot_lo_f = lo;
        p.shot_hi_f = hi;
        const double pl = ceil(p.shot_bound * 4096.0);
        p.pref_lo = pl >= 2048.0 ? 2048u : (uint32_t)pl;
    }
    p.capacity = capacity;
    if (h->cfg.photoreceptor_noise && h->cfg.cutoff_hz > 0) {
        const double eps = p.dt / (1.0 / (M_PI * 2 * h->cfg.cutoff_hz));   // emulator_utils.py:80, 97: a Python float
        p.pr_ome_f = (float)(1.0 - eps);
        p.pr_eps_f = (float)eps;
    }
    p.scidvs_first = (h->cfg.scidvs && !h->scidvs_started) ? 1 : 0;
    return p;
}

extern "C" int v2e_emu_create(const V2eEmuCfg *cfg, V2eEmu **out) {
    if (!cfg || !out) return fail(V2E_E_INVALID, "null argument");
    if (cfg->width <= 0 || cfg->height <= 0) return fail(V2E_E_INVALID, "bad frame size");
    if ((int64_t)cfg->width * cfg->height > (1ll << 30)) return fail(V2E_E_INVALID, "frame too large");
    if (cfg->iter_cap < 1 || cfg->iter_cap > kRecMaxCount) return fail(V2E_E_INVALID, "iter_cap out of range");
    if (cfg->max_frames_per_step < 1) return fail(V2E_E_INVALID, "max_frames_per_step < 1");
    if (cfg->csdvs && !(cfg->cutoff_hz > 0 || cfg->hdr))
        return fail(V2E_E_UNSUPPORTED, "csdvs needs a float64 photoreceptor state (cutoff_hz > 0)");
    if (cfg->csdvs && !(cfg->cs_tau_p_s > 0 && cfg->cs_tau_h_s > 0)) return fail(V2E_E_INVALID, "csdvs time constants must be positive");
    if (cfg->photoreceptor_noise && !(cfg->shot_noise_rate_hz > 0 && cfg->cutoff_hz > 0))   // emulator.py:196-204
        return fail(V2E_E_INVALID, "photoreceptor_noise needs shot_noise_rate_hz > 0 and cutoff_hz > 0");
    V2eEmu *h = new V2eEmu();
    memset(h, 0, sizeof(*h));
    h->cfg = *cfg;
    EmuDev &d = h->d;
    d.W = cfg->width;
    d.H = cfg->height;
    d.n = cfg->width * cfg->height;
    d.n_pad = (d.n + kVec - 1) / kVec * kVec;
    d.per_pixel_thres = cfg->per_pixel_thres;
    d.hdr = cfg->hdr;
    d.state_f64 = (cfg->cutoff_hz > 0 || cfg->hdr) ? 1 : 0;
    d.csdvs = cfg->csdvs;
    d.leak_on = cfg->leak_rate_hz > 0;
    d.lowpass_on = cfg->cutoff_hz > 0;
    d.scidvs = cfg->scidvs ? 1 : 0;
    d.pr_noise = cfg->photoreceptor_noise ? 1 : 0;
    // emulator.py:893: with photoreceptor noise the shot events come from the noise, none are injected
    d.shot_on = cfg->shot_noise_rate_hz > 0 && !d.pr_noise;
    d.refr_on = cfg->refractory_period_s > 0;
    d.rng_mode = cfg->rng_mode;
    d.iter_cap = cfg->iter_cap;
    d.seg_stride = 2 * cfg->iter_cap + 2;
    d.max_slots = cfg->max_frames_per_step;
    d.pos_nom = cfg->pos_thres_nominal;
    d.neg_nom = cfg->neg_thres_nominal;
    d.leak_rate_f = (float)cfg->leak_rate_hz;
    d.leak_jit_f = (float)cfg->leak_jitter_fraction;
    d.refr_f = (float)cfg->refractory_period_s;
    d.refr_d = cfg->refractory_period_s;
    d.shot_inten_m1 = cfg->shot_inten_factor - 1;
    d.seed = cfg->seed;
    h->state_elem = d.state_f64 ? 8 : 4;
    h->min_thres = 0.01;
    h->fused_enable = 1;
    h->ls.t_frames = new double[cfg->max_frames_per_step]();
    h->sched = new V2eEmu::Seg[(size_t)cfg->max_frames_per_step + 2]();
    d.px_off = cfg->rng_pixel_offset;
    d.units = (d.n + kUnitPx - 1) / kUnitPx;
    // state arrays are staged in whole 128-pixel units by the update kernel's bulk copies
    size_t np = (size_t)d.units * kUnitPx;
#define ALLOC(ptr, bytes)                                                     \
    do {                                                                      \
        cudaError_t e_ = cudaMalloc((void **)&(ptr), (bytes));                \
        if (e_ == cudaSuccess) e_ = cudaMemset((ptr), 0, (bytes));            \
        if (e_ != cudaSuccess) { v2e_emu_destroy(h); return fail(V2E_E_CUDA, "cudaMalloc: %s", cudaGetErrorString(e_)); } \
    } while (0)
    ALLOC(d.lp, np * h->state_elem);
    ALLOC(d.base, np * h->state_elem);
    d.lp_out = d.lp;
    d.base_out = d.base;
    ALLOC(d.rec, np * sizeof(int16_t));

    if (d.per_pixel_thres) { ALLOC(d.pos_thres, np * 4); ALLOC(d.neg_thres, np * 4); }
    if (d.leak_on) ALLOC(d.noise_rate, np * 4);
    if (d.refr_on) ALLOC(d.tmem, np * 4);
    if (d.scidvs) { ALLOC(d.hp, np * h->state_elem); ALLOC(d.prev_photo, np * h->state_elem); ALLOC(d.tau_arr, np * 4); }
    if (d.pr_noise) ALLOC(d.noise_arr, np * 4);
    if (d.scidvs || d.pr_noise) {
        ALLOC(d.pr_eff, np * h->state_elem);
        h->pr_vrms = new double[cfg->max_frames_per_step]();
    }
    d.own_lo = 0;
    d.own_hi = d.n;
    d.cs_y_lo = 0;
    d.cs_y_hi = d.H;
    d.cs_ring = 2;
    if (cfg->own_rows > 0) {
        if (cfg->own_row0 < 0 || cfg->own_row0 + cfg->own_rows > d.H) { v2e_emu_destroy(h); return fail(V2E_E_INVALID, "own rows outside the handle"); }
        d.own_lo = cfg->own_row0 * d.W;
        d.own_hi = (cfg->own_row0 + cfg->own_rows) * d.W;
        d.cs_y_lo = cfg->own_row0;
        d.cs_y_hi = cfg->own_row0 + cfg->own_rows;
    }
    if (d.csdvs) {
        ALLOC(d.cs_cur, sizeof(int32_t));
        d.cs_cap = 8192;
        ALLOC(d.cs_max, (size_t)d.cs_cap * sizeof(unsigned long long));
        // float32 conv2d summation order of the reference's CPU backend: decided by the size of the WHOLE frame
        const long long full_px = cfg->full_frame_px ? (long long)cfg->full_frame_px : (long long)d.n;
        d.cs_seq_order = full_px >= 20000;
        if (cfg->cs_halo_rows > 0) {
            const int K = cfg->cs_halo_rows;
            if (K > d.cs_y_hi - d.cs_y_lo) { v2e_emu_destroy(h); return fail(V2E_E_INVALID, "cs_halo_rows larger than the band"); }
            h->cs_K = K;
            d.cs_ring = K + 1;
            d.cs_stride = np;
            ALLOC(d.cs_bufs, (size_t)d.cs_ring * np * 8);
            ALLOC(d.cs_done, sizeof(int32_t));
            ALLOC(h->cs_send, (size_t)2 * K * d.W * 8);
            ALLOC(h->cs_recv, (size_t)2 * K * d.W * 8);
        } else {
            ALLOC(d.surround, np * 8);
            ALLOC(d.surround2, np * 8);
        }
    }
    ALLOC(h->lut_dev, 256 * 4);
    d.lut = h->lut_dev;
    size_t slots = (size_t)d.max_slots;
    ALLOC(d.ctrl, (slots + 1) * sizeof(FrameCtrl));
    ALLOC(d.hist_pre, slots * d.seg_stride * 4);
    ALLOC(d.hist_post, slots * d.seg_stride * 4);
    ALLOC(d.segoff, slots * d.seg_stride * 4);
    ALLOC(d.cursor, slots * d.seg_stride * 4);
    {
        // one wave of the update kernel: 3 resident blocks per SM (2 stages x 28 KB of shared memory each),
        // every block the same number of 128-pixel units
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        d.n_blocks = 3 * sms;
        if (d.n_blocks > (d.units + 3) / 4) d.n_blocks = (d.units + 3) / 4;     // small frames: >= 4 units per block
        if (d.n_blocks < 1) d.n_blocks = 1;
        d.upb = (d.units + d.n_blocks - 1) / d.n_blocks;
        d.seg_px = d.upb * kUnitPx;
    }
    ALLOC(d.act_count, slots * d.n_blocks * sizeof(uint32_t));
    ALLOC(d.act_list, (size_t)d.n_blocks * d.seg_px * sizeof(uint32_t));
    ALLOC(d.abort_flag, 2 * sizeof(int32_t));
    ALLOC(d.chain_base, sizeof(unsigned long long));
#undef ALLOC
    if (cudaMallocHost((void **)&h->ctrl_host, (slots + 1) * sizeof(FrameCtrl)) != cudaSuccess ||
        cudaMallocHost((void **)&h->abort_host, 2 * sizeof(int32_t)) != cudaSuccess) {
        v2e_emu_destroy(h);
        return fail(V2E_E_CUDA, "cudaMallocHost failed");
    }
    *out = h;
    return V2E_OK;
}

extern "C" int v2e_emu_destroy(V2eEmu *h) {
    if (!h) return V2E_OK;
    EmuDev &d = h->d;
    delete[] h->pr_vrms;
    delete[] h->ls.t_frames;
    delete[] h->sched;
    void *cs_ptrs[] = {d.cs_bufs, d.cs_done, h->cs_send, h->cs_recv};
    for (void *p : cs_ptrs) if (p) cudaFree(p);
    void *fused_ptrs[] = {h->lp_alt, h->base_alt, h->rec_list, h->rec_cnt, h->blk_cnt, h->ff_dev, h->fp_dev, h->max_vec};
    for (void *p : fused_ptrs) if (p) cudaFree(p);
    void *ptrs[] = {d.hp, d.prev_photo, d.tau_arr, d.noise_arr, d.pr_eff,
                    d.lp, d.base, d.rec, d.pos_thres, d.neg_thres, d.noise_rate, d.tmem, d.surround,
                    h->lut_dev, d.ctrl, d.hist_pre, d.hist_post, d.segoff, d.cursor, d.abort_flag, d.chain_base, d.act_list, d.act_count, d.surround2, d.cs_cur, d.cs_max};
    for (void *p : ptrs) if (p) cudaFree(p);
    if (h->ctrl_host) cudaFreeHost(h->ctrl_host);
    if (h->abort_host) cudaFreeHost(h->abort_host);
    if (h->ev) {
        for (int i = 0; i < d.max_slots * kProfKinds * 2; i++) cudaEventDestroy(h->ev[i]);
        delete[] h->ev;
        delete[] h->prof_used;
    }
    delete h;
    return V2E_OK;
}

extern "C" int v2e_emu_set_linlog_lut(V2eEmu *h, const float *lut, void *stream) {
    if (!h || !lut) return fail(V2E_E_INVALID, "null argument");
    CU(cudaMemcpyAsync(h->lut_dev, lut, 256 * 4, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    return V2E_OK;
}

extern "C" int v2e_emu_set_fields(V2eEmu *h, const float *pos, const float *neg, const float *nr) {
    if (!h) return fail(V2E_E_INVALID, "null handle");
    size_t bytes = (size_t)h->d.n * 4;
    if (h->d.per_pixel_thres) {
        if (!pos || !neg) return fail(V2E_E_INVALID, "per-pixel thresholds required");
        CU(cudaMemcpy(h->d.pos_thres, pos, bytes, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(h->d.neg_thres, neg, bytes, cudaMemcpyHostToDevice));
        float mn = pos[0];
        for (int i = 0; i < h->d.n; i++) { mn = pos[i] < mn ? pos[i] : mn; mn = neg[i] < mn ? neg[i] : mn; }
        if (!(mn > 0)) return fail(V2E_E_INVALID, "thresholds must be positive");
        h->min_thres = (double)mn;
    }
    if (h->d.leak_on) {
        if (!nr) return fail(V2E_E_INVALID, "noise_rate field required when leak_rate_hz > 0");
        CU(cudaMemcpy(h->d.noise_rate, nr, bytes, cudaMemcpyHostToDevice));
    }
    return V2E_OK;
}

extern "C" int v2e_emu_set_scidvs_tau(V2eEmu *h, const float *tau_host) {
    if (!h || !tau_host) return fail(V2E_E_INVALID, "null argument");
    if (!h->d.scidvs) return fail(V2E_E_STATE, "scidvs is not enabled for this handle");
    CU(cudaMemcpy(h->d.tau_arr, tau_host, (size_t)h->d.n * 4, cudaMemcpyHostToDevice));
    return V2E_OK;
}

extern "C" int v2e_emu_set_pr_noise(V2eEmu *h, const float *pr_randn_dev, const double *vrms_host, int T) {
    if (!h || !vrms_host) return fail(V2E_E_INVALID, "null argument");
    if (!h->d.pr_noise) return fail(V2E_E_STATE, "photoreceptor_noise is not enabled for this handle");
    if (T < 1 || T > h->d.max_slots) return fail(V2E_E_INVALID, "bad T");
    if (h->d.rng_mode == 0 && !pr_randn_dev) return fail(V2E_E_INVALID, "the randn field is required in replay mode");
    h->pr_randn_dev = pr_randn_dev;
    memcpy(h->pr_vrms, vrms_host, sizeof(double) * (size_t)T);
    h->pr_T = T;
    return V2E_OK;
}

// one block per list segment while they are all co-resident (148 SMs x 8 blocks), grid-stride beyond
static inline int list_grid(const EmuDev &d) { return d.n_blocks < 1184 ? d.n_blocks : 1184; }
static inline int grid_for(const EmuDev &d) { return (d.n_pad / kVec + kThreads - 1) / kThreads; }

template <typename S>
static int launch_first(V2eEmu *h, const FrameParams &p, const void *frame, int dt, cudaStream_t st) {
    int g = grid_for(h->d);
    switch (dt) {
        case V2E_U8: emu_first_frame_kernel<S, V2E_U8><<<g, kThreads, 0, st>>>(h->d, p, frame); break;
        case V2E_F32: emu_first_frame_kernel<S, V2E_F32><<<g, kThreads, 0, st>>>(h->d, p, frame); break;
        case V2E_F64: emu_first_frame_kernel<S, V2E_F64><<<g, kThreads, 0, st>>>(h->d, p, frame); break;
        default: return fail(V2E_E_INVALID, "bad frame dtype");
    }
    return V2E_OK;
}

extern "C" int v2e_emu_first_frame(V2eEmu *h, const void *frame, int dtype, double t_frame,
                                   double t_previous, void *stream) {
    if (!h || !frame) return fail(V2E_E_INVALID, "null argument");
    FrameParams p = make_params(h, t_frame, t_previous, 0, 0);
    int rc = h->d.state_f64 ? launch_first<double>(h, p, frame, dtype, (cudaStream_t)stream)
                            : launch_first<float>(h, p, frame, dtype, (cudaStream_t)stream);
    if (rc) return rc;
    if (h->d.csdvs) CU(cudaMemsetAsync(h->d.cs_cur, 0, sizeof(int32_t), (cudaStream_t)stream));
    CU(cudaGetLastError());
    h->first_done = 1;
    return V2E_OK;
}

template <typename S, int RNG>
static int launch_update_r(V2eEmu *h, const FrameParams &p, const void *frame, int dt, const float *lr,
                           const float *sr, int slot, int do_plan, int lp_done, cudaStream_t st) {
    int g = h->d.n_blocks;
    const EmuDev &d = h->d;
    const size_t sm = (size_t)StageLayout<S>::block_bytes;
    {
        // opt in to > 48 KB of dynamic shared memory once per instantiation
        static PerDeviceOnce once;
        if (once.first()) {
            CU(cudaFuncSetAttribute(emu_update_kernel<double, V2E_U8, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)StageLayout<double>::block_bytes));
            CU(cudaFuncSetAttribute(emu_update_kernel<S, V2E_U8, RNG, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
            CU(cudaFuncSetAttribute(emu_update_kernel<S, V2E_F32, RNG, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
            CU(cudaFuncSetAttribute(emu_update_kernel<S, V2E_F64, RNG, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        }
    }
    if (sizeof(S) == 8 && RNG == 1 && dt == V2E_U8 && d.per_pixel_thres && d.leak_on && d.lowpass_on && d.shot_on &&
        !d.hdr && !d.csdvs && !lp_done) {
        emu_update_kernel<double, V2E_U8, 1, true><<<g, kThreads, sm, st>>>(h->d, p, frame, lr, sr, slot, do_plan, 0);
        return V2E_OK;
    }
    switch (dt) {
        case V2E_U8: emu_update_kernel<S, V2E_U8, RNG, false><<<g, kThreads, sm, st>>>(h->d, p, frame, lr, sr, slot, do_plan, lp_done); break;
        case V2E_F32: emu_update_kernel<S, V2E_F32, RNG, false><<<g, kThreads, sm, st>>>(h->d, p, frame, lr, sr, slot, do_plan, lp_done); break;
        case V2E_F64: emu_update_kernel<S, V2E_F64, RNG, false><<<g, kThreads, sm, st>>>(h->d, p, frame, lr, sr, slot, do_plan, lp_done); break;
        default: return fail(V2E_E_INVALID, "bad frame dtype");
    }
    return V2E_OK;
}
template <typename S>
static int launch_update(V2eEmu *h, const FrameParams &p, const void *frame, int dt, const float *lr,
                         const float *sr, int slot, int do_plan, int lp_done, cudaStream_t st) {
    return h->d.rng_mode == 1 ? launch_update_r<S, 1>(h, p, frame, dt, lr, sr, slot, do_plan, lp_done, st)
                              : launch_update_r<S, 0>(h, p, frame, dt, lr, sr, slot, do_plan, lp_done, st);
}

static int launch_shot(V2eEmu *h, const FrameParams &p, const void *frame, int dt, const float *sr,
                       int slot, cudaStream_t st) {
    int g = grid_for(h->d);
    switch (dt) {
        case V2E_U8: emu_shot_kernel<V2E_U8><<<g, kThreads, 0, st>>>(h->d, p, frame, sr, slot); break;
        case V2E_F32: emu_shot_kernel<V2E_F32><<<g, kThreads, 0, st>>>(h->d, p, frame, sr, slot); break;
        case V2E_F64: emu_shot_kernel<V2E_F64><<<g, kThreads, 0, st>>>(h->d, p, frame, sr, slot); break;
        default: return fail(V2E_E_INVALID, "bad frame dtype");
    }
    return V2E_OK;
}

struct ProfScope {
    V2eEmu *h; int slot, kind; cudaStream_t st;
    ProfScope(V2eEmu *h_, int slot_, int kind_, cudaStream_t st_) : h(h_), slot(slot_), kind(kind_), st(st_) {
        if (h->profile) { cudaEventRecord(h->ev[(slot * kProfKinds + kind) * 2], st); h->prof_used[slot * kProfKinds + kind] = 1; }
    }
    ~ProfScope() { if (h->profile) cudaEventRecord(h->ev[(slot * kProfKinds + kind) * 2 + 1], st); }
};

static size_t frame_elem(int dt) { return dt == V2E_U8 ? 1 : (dt == V2E_F32 ? 4 : 8); }

// One cooperative launch for Euler steps [s0, s1) (emu_csdvs_iter_kernel). Returns false when the device / occupancy
// does not allow a cooperative grid (the per-step kernels are used then).
static bool cs_launch_iter(V2eEmu *h, double alpha_p, float alpha_h, int s0, int s1, int sharded, int slot, cudaStream_t st) {
    static int coop = -1, blocks_per_sm = 0, sms = 148;
    if (coop < 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, emu_csdvs_iter_kernel, kCsThreads, 0) != cudaSuccess)
            blocks_per_sm = 0;
        const char *e = getenv("V2E_CS_COOP");
        if (e && atoi(e) == 0) coop = 0;
    }
    if (!coop || blocks_per_sm < 1) return false;
    const EmuDev &d = h->d;
    int grid = sms * (blocks_per_sm > 2 ? 2 : blocks_per_sm);            // few, fat blocks: a cheap grid barrier
    const int need = (d.n + kCsThreads - 1) / kCsThreads;
    if (grid > need) grid = need;
    EmuDev dd = d;
    void *args[] = {(void *)&dd, (void *)&alpha_p, (void *)&alpha_h, (void *)&s0, (void *)&s1, (void *)&sharded, (void *)&slot};
    if (cudaLaunchCooperativeKernel((const void *)emu_csdvs_iter_kernel, dim3(grid), dim3(kCsThreads), args, 0, st) == cudaSuccess)
        return true;
    cudaGetLastError();         // clear; fall back to one launch per step from now on
    coop = 0;
    return false;
}

// Euler-step plan of one frame of the centre-surround model (emulator.py:1068-1096)
static int cs_plan(const V2eEmu *h, const FrameParams &p, int *num_steps, double *alpha_p, float *alpha_h) {
    const double tau_p = h->cfg.cs_tau_p_s, tau_h = h->cfg.cs_tau_h_s;
    const double min_tau = tau_p < tau_h ? tau_p : tau_h;
    const int n = (int)ceil((p.dt / min_tau) * 5);                          // emulator.py:1076-1078
    if (n < 1) return fail(V2E_E_INVALID, "csdvs: delta_time must be positive");
    if (n > h->d.cs_cap) return fail(V2E_E_UNSUPPORTED, "csdvs: more Euler steps per frame than cs_cap (8192)");
    const double adt = p.dt / n;
    const double ap = adt / tau_p, ah = adt / tau_h;
    if (ap >= 1 || ah >= 1)                                                  // emulator.py:1091-1096 quits
        return fail(V2E_E_INVALID, "CSDVS update alpha (of IIR update) is too large; simulation would explode");
    *num_steps = n;
    *alpha_p = ap;
    *alpha_h = (float)ah;
    return V2E_OK;
}

// enqueue the counting kernels of one frame into `slot`
static int enqueue_count(V2eEmu *h, const FrameParams &p, const void *frame, int dtype, const float *lr,
                         const float *sr, int shot_pending, int slot, cudaStream_t st, const float *pr_randn = nullptr) {
    const EmuDev &d = h->d;
    if (d.pr_noise && d.rng_mode == 0 && !pr_randn) return fail(V2E_E_STATE, "v2e_emu_set_pr_noise must precede this call");
    if (d.rng_mode == 0 && d.leak_on && !lr) return fail(V2E_E_INVALID, "leak_randn field required in replay mode");
    const bool shot_in_update = d.shot_on && (d.rng_mode == 1 || sr != nullptr);
    if (d.shot_on && !shot_in_update && !shot_pending)
        return fail(V2E_E_INVALID, "shot_rand field required in replay mode (or shot_pending)");
    const int plan_in_update = (!d.refr_on && !shot_pending) ? 1 : 0;
    int rc;
    int lp_done = 0;
    if (d.csdvs) {
        // emulator.py:686-708: low-pass for the whole field, then the surround's Euler steps
        const int g = grid_for(d);
        switch (dtype) {
            case V2E_U8: emu_lp_kernel<V2E_U8><<<g, kThreads, 0, st>>>(d, p, frame); break;
            case V2E_F32: emu_lp_kernel<V2E_F32><<<g, kThreads, 0, st>>>(d, p, frame); break;
            case V2E_F64: emu_lp_kernel<V2E_F64><<<g, kThreads, 0, st>>>(d, p, frame); break;
            default: return fail(V2E_E_INVALID, "bad frame dtype");
        }
        lp_done = 1;
    }
    if (d.scidvs || d.pr_noise) {
        // low-pass (unless the surround path just did it), noise IIR, nonlinear high-pass -> pr_eff
        const int g = grid_for(d);
#define FRONT(S_)                                                                                                  \
        switch (dtype) {                                                                                            \
            case V2E_U8: emu_front_kernel<S_, V2E_U8><<<g, kThreads, 0, st>>>(d, p, frame, pr_randn, lp_done); break;   \
            case V2E_F32: emu_front_kernel<S_, V2E_F32><<<g, kThreads, 0, st>>>(d, p, frame, pr_randn, lp_done); break; \
            case V2E_F64: emu_front_kernel<S_, V2E_F64><<<g, kThreads, 0, st>>>(d, p, frame, pr_randn, lp_done); break; \
            default: return fail(V2E_E_INVALID, "bad frame dtype");                                                 \
        }
        if (d.state_f64) { FRONT(double) } else { FRONT(float) }
#undef FRONT
        lp_done = 1;
    }
    if (d.csdvs) {
        if (h->cs_K) return fail(V2E_E_STATE, "a pixel-sharded centre-surround handle is stepped with v2e_emu_cs_*");
        int num_steps = 0;
        double alpha_p = 0;
        float alpha_h = 0;
        if ((rc = cs_plan(h, p, &num_steps, &alpha_p, &alpha_h))) return rc;
        CU(cudaMemsetAsync(d.cs_max, 0, (size_t)num_steps * sizeof(unsigned long long), st));
        if (!cs_launch_iter(h, alpha_p, alpha_h, 0, num_steps, 0, slot, st)) {
            const int gs = (d.n + kThreads - 1) / kThreads;
            for (int k = 0; k < num_steps; k++)
                emu_csdvs_step_kernel<<<gs, kThreads, 0, st>>>(d, alpha_p, alpha_h, k, k, 0);
            emu_csdvs_finish_kernel<<<1, 1, 0, st>>>(d, num_steps, slot);
        }
    }
    {
        ProfScope ps(h, slot, 0, st);
        rc = d.state_f64 ? launch_update<double>(h, p, frame, dtype, lr, sr, slot, plan_in_update, lp_done, st)
                         : launch_update<float>(h, p, frame, dtype, lr, sr, slot, plan_in_update, lp_done, st);
    }
    if (rc) return rc;
    if (d.refr_on) {
        ProfScope ps(h, slot, 1, st);
        emu_filter_kernel<<<list_grid(d), kThreads, 0, st>>>(d, p, slot, !shot_pending);
    }
    return V2E_OK;
}

static int enqueue_emit(V2eEmu *h, const FrameParams &p, int slot, float *events, cudaStream_t st) {
    const EmuDev &d = h->d;
    ProfScope ps(h, slot, 2, st);
    if (d.state_f64) emu_emit_kernel<double><<<list_grid(d), kThreads, 0, st>>>(d, p, slot, (float4 *)events);
    else emu_emit_kernel<float><<<list_grid(d), kThreads, 0, st>>>(d, p, slot, (float4 *)events);
    return V2E_OK;
}
static void enqueue_null_bracket(V2eEmu *h, int slot, cudaStream_t st) {
    if (!h->profile) return;
    ProfScope ps(h, slot, 3, st);
    emu_null_kernel<<<1, 32, 0, st>>>();
}

static int reset_slots(V2eEmu *h, int first, int count, cudaStream_t st, bool clear_abort = true) {
    EmuDev &d = h->d;
    size_t off = (size_t)first * d.seg_stride * 4, bytes = (size_t)count * d.seg_stride * 4;
    CU(cudaMemsetAsync((char *)d.hist_pre + off, 0, bytes, st));
    CU(cudaMemsetAsync((char *)d.hist_post + off, 0, bytes, st));
    CU(cudaMemsetAsync((char *)d.cursor + off, 0, bytes, st));
    CU(cudaMemsetAsync(d.ctrl + first, 0, (size_t)(count + 1) * sizeof(FrameCtrl), st));
    CU(cudaMemsetAsync(d.act_count + (size_t)first * d.n_blocks, 0, (size_t)count * d.n_blocks * sizeof(uint32_t), st));
    if (clear_abort) CU(cudaMemsetAsync(d.abort_flag, 0, 2 * sizeof(int32_t), st));
    return V2E_OK;
}


// ---- fused multi-frame path, host side ------------------------------------------------------------
constexpr uint64_t kChainBase = ~0ull;      // step_classic: start at the row the multi-frame chunk ended at
static int fused_groups(const EmuDev &d) { return (d.units + kFusedGroup - 1) / kFusedGroup; }

static bool fused_config_ok(const V2eEmu *h, int dtype) {
    const EmuDev &d = h->d;
    return dtype == V2E_U8 && !d.hdr && !d.csdvs && !d.scidvs && !d.pr_noise &&
           (d.rng_mode == 1 || (!d.leak_on && !d.shot_on)) && (d.state_f64 ? d.lowpass_on : !d.lowpass_on);
}

static int fused_alloc(V2eEmu *h) {
    if (h->fused_max_T) return V2E_OK;
    const EmuDev &d = h->d;
    // record lists: 2 bytes per pixel and frame of capacity (sparsely written); bounded at 1.5 GB
    size_t per_frame = (size_t)d.units * kUnitPx * sizeof(uint16_t);
    int maxT = (int)((size_t)1536 * 1024 * 1024 / per_frame);
    if (maxT > d.max_slots) maxT = d.max_slots;
    if (maxT < 2) { h->fused_max_T = -1; return V2E_OK; }
    const size_t np = (size_t)d.units * kUnitPx;
#define FALLOC(ptr, bytes)                                                                  \
    do {                                                                                    \
        cudaError_t e_ = cudaMalloc((void **)&(ptr), (bytes));                              \
        if (e_ != cudaSuccess) return fail(V2E_E_CUDA, "cudaMalloc (fused path): %s", cudaGetErrorString(e_)); \
    } while (0)
    FALLOC(h->lp_alt, np * h->state_elem);
    FALLOC(h->base_alt, np * h->state_elem);
    FALLOC(h->rec_list, (size_t)maxT * per_frame);
    FALLOC(h->rec_cnt, (size_t)maxT * d.units * sizeof(uint32_t));
    FALLOC(h->blk_cnt, (size_t)maxT * fused_groups(d) * kBlkSeg * sizeof(uint32_t));
    FALLOC(h->ff_dev, (size_t)d.max_slots * sizeof(FusedFrame));
    FALLOC(h->fp_dev, (size_t)d.max_slots * sizeof(FrameParams));
    FALLOC(h->max_vec, (size_t)d.max_slots * sizeof(int32_t));
#undef FALLOC
    CU(cudaMemset(h->lp_alt, 0, np * h->state_elem));
    CU(cudaMemset(h->base_alt, 0, np * h->state_elem));
    h->fused_max_T = maxT;
    return V2E_OK;
}

// Block shape of pass 1. The kernel is bound by dependent-instruction latency, so what matters is (resident warps)
// against (units per warp, an integer): 0 = 8 warps x 3 blocks/SM (24 warps, 80 registers), 1 = 4 x 5 (20 warps,
// 96 registers), 2 = 4 x 7 (28 warps, 72 registers), 3 = 8 x 2 (16 warps, 128 registers). V2E_FUSED_CFG overrides.
static int fused_cfg() {
    static int cfg = -1;
    if (cfg < 0) {
        const char *e = getenv("V2E_FUSED_CFG");
        cfg = e ? atoi(e) : 1;
        if (cfg < 0 || cfg > 3) cfg = 1;
    }
    return cfg;
}
template <typename S, bool FAST, int WARPS, int MINB>
static void launch_fused_update_cfg(V2eEmu *h, const EmuDev &d, const FusedFrame *ff, const uint8_t *frames, int T, size_t sm,
                                    cudaStream_t st) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int blocks = sms * MINB;
    const int min_units = 2 * WARPS;                       // small frames: at least two units per warp
    if (blocks > (d.units + min_units - 1) / min_units) blocks = (d.units + min_units - 1) / min_units;
    if (blocks < 1) blocks = 1;
    emu_fused_update_kernel<S, FAST, WARPS, MINB><<<blocks, WARPS * 32, sm, st>>>(d, ff, frames, T, (S *)h->lp_alt,
                                                                                   (S *)h->base_alt, h->rec_list, h->rec_cnt);
}
template <typename S, bool FAST>
static void launch_fused_update_f(V2eEmu *h, const EmuDev &d, const FusedFrame *ff, const uint8_t *frames, int T, size_t sm,
                                  cudaStream_t st) {
    switch (fused_cfg()) {
        case 0: launch_fused_update_cfg<S, FAST, 8, 3>(h, d, ff, frames, T, sm, st); break;
        case 2: launch_fused_update_cfg<S, FAST, 4, 7>(h, d, ff, frames, T, sm, st); break;
        case 3: launch_fused_update_cfg<S, FAST, 8, 2>(h, d, ff, frames, T, sm, st); break;
        default: launch_fused_update_cfg<S, FAST, 4, 5>(h, d, ff, frames, T, sm, st); break;
    }
}
template <typename S>
static int launch_fused_update(V2eEmu *h, const EmuDev &d, const FusedFrame *ff, const uint8_t *frames, int T, cudaStream_t st) {
    const size_t sm = (size_t)T * sizeof(FusedFrame);
    const bool fast = sizeof(S) == 8 && d.rng_mode == 1 && d.per_pixel_thres && d.leak_on && d.shot_on;
    if (sm > 40 * 1024) return fail(V2E_E_INVALID, "fused path: too many frames per step");
    if (fast) launch_fused_update_f<S, true>(h, d, ff, frames, T, sm, st);
    else launch_fused_update_f<S, false>(h, d, ff, frames, T, sm, st);
    return V2E_OK;
}

// uploads the per-frame parameters of a chunk; returns them in `fp_host` too
static int fused_upload_params(V2eEmu *h, int T, const double *t_frames, double t_previous, uint32_t frame_base,
                               uint64_t capacity, cudaStream_t st) {
    static thread_local FusedFrame *ffh = nullptr;
    static thread_local FrameParams *fph = nullptr;
    static thread_local int cap = 0;
    if (cap < T) {
        delete[] ffh; delete[] fph;
        cap = T > 64 ? T : 64;
        ffh = new FusedFrame[cap];
        fph = new FrameParams[cap];
    }
    for (int f = 0; f < T; f++) {
        const double tp = f == 0 ? t_previous : t_frames[f - 1];
        if (t_frames[f] < tp) return fail(V2E_E_INVALID, "frame times must be non-decreasing");
        fph[f] = make_params(h, t_frames[f], tp, frame_base + (uint32_t)f, capacity);
        memset(&ffh[f], 0, sizeof(FusedFrame));
        ffh[f].eps_scale = fph[f].eps_scale;
        ffh[f].shot_c = fph[f].shot_c;
        ffh[f].dt_f = fph[f].dt_f;
        ffh[f].frame_index = fph[f].frame_index;
        ffh[f].pref_lo = fph[f].pref_lo;
    }
    // pageable sources: the runtime stages them before the call returns, so the buffers can be reused at once
    CU(cudaMemcpyAsync(h->ff_dev, ffh, (size_t)T * sizeof(FusedFrame), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(h->fp_dev, fph, (size_t)T * sizeof(FrameParams), cudaMemcpyHostToDevice, st));
    return V2E_OK;
}

// the handle's device view shifted to frame slot `a` of the step: the multi-frame kernels index frames from 0
static EmuDev shifted_dev(const EmuDev &d, int a) {
    EmuDev s = d;
    s.ctrl = d.ctrl + a;
    s.hist_pre = d.hist_pre + (size_t)a * d.seg_stride;
    s.hist_post = d.hist_post + (size_t)a * d.seg_stride;
    s.segoff = d.segoff + (size_t)a * d.seg_stride;
    s.cursor = d.cursor + (size_t)a * d.seg_stride;
    return s;
}

// frames [a, a + T) of `frames` (the step's frame 0 at `frames`)
static int enqueue_fused_count(V2eEmu *h, const void *frames, int T, cudaStream_t st, int a = 0) {
    const EmuDev d = shifted_dev(h->d, a);
    const uint8_t *fr = (const uint8_t *)frames + (size_t)a * d.n;
    int rc;
    {
        ProfScope ps(h, 0, 0, st);
        rc = d.state_f64 ? launch_fused_update<double>(h, d, h->ff_dev + a, fr, T, st)
                         : launch_fused_update<float>(h, d, h->ff_dev + a, fr, T, st);
    }
    if (rc) return rc;
    {
        ProfScope ps(h, 0, 1, st);
        emu_fused_count_kernel<<<T * fused_groups(d), kThreads, 0, st>>>(d, T, fused_groups(d), h->rec_list, h->rec_cnt, h->blk_cnt);
    }
    return V2E_OK;
}

static int enqueue_fused_emit(V2eEmu *h, int T, float *events, uint64_t capacity, uint64_t ev_base_start,
                              const int32_t *max_vec, bool commit, cudaStream_t st, int a = 0, int chain = 0) {
    const EmuDev d = shifted_dev(h->d, a);
    {
        ProfScope ps(h, 1, 1, st);       // slot 1: v2e_emu_profile_read sums count + plan under "filter"
        emu_fused_plan_kernel<<<1, kThreads, (size_t)T * sizeof(uint32_t), st>>>(d, h->fp_dev + a, T, ev_base_start, capacity,
                                                                                 max_vec, a, chain);
    }
    {
        ProfScope ps(h, 0, 2, st);
        emu_fused_emit_kernel<<<T * fused_groups(d), kThreads, 0, st>>>(d, h->fp_dev + a, T, fused_groups(d), h->rec_list,
                                                                         h->rec_cnt, h->blk_cnt, (float4 *)events);
    }
    if (commit) {
        ProfScope ps(h, 1, 2, st);       // emit + commit under "emit"
        const size_t n16 = (size_t)d.units * kUnitPx * h->state_elem / 16;
        emu_fused_commit_kernel<<<296, kThreads, 0, st>>>(d, (const uint4 *)h->lp_alt, (const uint4 *)h->base_alt, n16);
    }
    return V2E_OK;
}

static void remember_step(V2eEmu *h, const void *frames, int dtype, int T, const double *t_frames, double t_previous,
                          float *events, uint64_t capacity, uint64_t ev_base_start) {
    h->ls.frames = frames; h->ls.dtype = dtype; h->ls.T = T; h->ls.t_previous = t_previous;
    h->ls.events = events; h->ls.capacity = capacity; h->ls.ev_base_start = ev_base_start;
    if (t_frames != h->ls.t_frames) memcpy(h->ls.t_frames, t_frames, sizeof(double) * (size_t)T);
}

static int step_classic(V2eEmu *h, const void *frames, int dtype, int T, const double *t_frames, double t_previous,
                        const float *leak_randn, const float *shot_rand, float *events, uint64_t capacity,
                        uint64_t ev_base_start, int first, int resume_emit, void *stream, int last = -1);

// Runs segments [from, n_seg) of the handle's schedule over the remembered step (h->ls); Philox frame indices are
// step_base + frame. The first segment of the step starts at ls.ev_base_start, every other one where the previous
// segment / frame ended (chain_base, device side). A capacity abort or a rejection anywhere is sticky: every later
// kernel leaves at once; v2e_emu_collect sorts it out.
static int run_schedule(V2eEmu *h, int from, cudaStream_t st) {
    int rc;
    for (int i = from; i < h->n_seg; i++) {
        const V2eEmu::Seg g = h->sched[i];
        const bool step_start = g.a == 0;
        if (g.kind == 0) {
            const int Tf = g.b - g.a;
            if ((rc = reset_slots(h, g.a, Tf, st, false))) return rc;
            if ((rc = enqueue_fused_count(h, h->ls.frames, Tf, st, g.a))) return rc;
            if ((rc = enqueue_fused_emit(h, Tf, h->ls.events, h->ls.capacity, h->ls.ev_base_start, nullptr, true, st, g.a,
                                         step_start ? 0 : 1))) return rc;
        } else {
            h->frame_counter = h->step_base;
            if ((rc = step_classic(h, h->ls.frames, h->ls.dtype, h->ls.T, h->ls.t_frames, h->ls.t_previous, nullptr, nullptr,
                                   h->ls.events, h->ls.capacity, step_start ? h->ls.ev_base_start : kChainBase, g.a, 0,
                                   (void *)st, g.b))) return rc;
        }
    }
    CU(cudaGetLastError());
    h->frame_counter = h->step_base + (uint32_t)h->ls.T;
    h->last_T = h->ls.T;
    return V2E_OK;
}

extern "C" int v2e_emu_set_option(V2eEmu *h, int option, int value) {
    if (!h) return fail(V2E_E_INVALID, "null handle");
    if (option == 0) { h->fused_enable = value ? 1 : 0; return V2E_OK; }
    return fail(V2E_E_INVALID, "unknown option");
}
extern "C" int v2e_emu_fused_stats(V2eEmu *h, long long *chunks, long long *rejected) {
    if (!h) return fail(V2E_E_INVALID, "null handle");
    if (chunks) *chunks = h->n_fused_chunks;
    if (rejected) *rejected = h->n_fused_rejected;
    return V2E_OK;
}
extern "C" int v2e_emu_fused_frames(V2eEmu *h, long long *frames_multi, long long *frames_single) {
    if (!h) return fail(V2E_E_INVALID, "null handle");
    if (frames_multi) *frames_multi = h->n_frames_multi;
    if (frames_single) *frames_single = h->n_frames_single;
    return V2E_OK;
}
extern "C" int v2e_emu_fused_last_reject(V2eEmu *h, int *frame, int *max_n) {
    if (!h) return fail(V2E_E_INVALID, "null handle");
    if (frame) *frame = h->last_reject_frame;
    if (max_n) *max_n = h->last_reject_max_n;
    return V2E_OK;
}
extern "C" int32_t *v2e_emu_max_vec_dev(V2eEmu *h) { return h ? h->max_vec : nullptr; }

__global__ void emu_gather_max_kernel(EmuDev d, int T, int32_t *max_vec) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < T) max_vec[f] = d.ctrl[f].max_n;
}

extern "C" int v2e_emu_fused_count(V2eEmu *h, const void *frames, int dtype, int T, const double *t_frames,
                                   double t_previous, void *stream) {
    if (!h || !frames || !t_frames) return fail(V2E_E_INVALID, "null argument");
    if (!h->first_done) return fail(V2E_E_STATE, "v2e_emu_first_frame must run first");
    if (T < 1 || T > h->d.max_slots) return fail(V2E_E_INVALID, "bad T");
    if (!fused_config_ok(h, dtype)) return fail(V2E_E_UNSUPPORTED, "configuration does not qualify for the fused path");
    int rc;
    if ((rc = fused_alloc(h))) return rc;
    if (h->fused_max_T < T) return fail(V2E_E_UNSUPPORTED, "fused path: T exceeds the record lists");
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = reset_slots(h, 0, T, st))) return rc;
    if (h->profile) { memset(h->prof_used, 0, (size_t)h->d.max_slots * kProfKinds); h->prof_frames = T; }
    h->step_base = h->frame_counter;
    h->frame_counter += (uint32_t)T;
    if ((rc = fused_upload_params(h, T, t_frames, t_previous, h->step_base, 0, st))) return rc;
    if ((rc = enqueue_fused_count(h, frames, T, st))) return rc;
    emu_gather_max_kernel<<<(T + 127) / 128, 128, 0, st>>>(h->d, T, h->max_vec);
    CU(cudaGetLastError());
    remember_step(h, frames, dtype, T, t_frames, t_previous, nullptr, 0, 0);
    h->last_T = T;
    h->last_fused = 2;
    h->fused_T = T;
    h->n_fused_chunks++;
    return V2E_OK;
}

extern "C" int v2e_emu_fused_emit(V2eEmu *h, float *events, uint64_t capacity, uint64_t ev_base_start, void *stream) {
    if (!h || (!events && capacity)) return fail(V2E_E_INVALID, "null argument");
    if (h->last_fused != 2) return fail(V2E_E_STATE, "v2e_emu_fused_count must precede v2e_emu_fused_emit");
    if (((uintptr_t)events & 15) != 0) return fail(V2E_E_INVALID, "events_out must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const EmuDev &d = h->d;
    const int T = h->ls.T;
    // a second call after V2E_E_CAPACITY: same records, new plan
    CU(cudaMemsetAsync(d.abort_flag, 0, 2 * sizeof(int32_t), st));
    CU(cudaMemsetAsync(d.cursor, 0, (size_t)T * d.seg_stride * 4, st));
    h->ls.events = events; h->ls.capacity = capacity; h->ls.ev_base_start = ev_base_start;
    int rc = enqueue_fused_emit(h, T, events, capacity, ev_base_start, h->max_vec, true, st);
    if (rc) return rc;
    CU(cudaGetLastError());
    return V2E_OK;
}

// frames [first, last) of the step (last < 0: to the end)
static int step_classic(V2eEmu *h, const void *frames, int dtype, int T, const double *t_frames,
                            double t_previous, const float *leak_randn, const float *shot_rand,
                            float *events, uint64_t capacity, uint64_t ev_base_start, int first,
                            int resume_emit, void *stream, int last) {
    if (!h || !frames || !t_frames || (!events && capacity)) return fail(V2E_E_INVALID, "null argument");
    if (!h->first_done) return fail(V2E_E_STATE, "v2e_emu_first_frame must run before v2e_emu_step");
    if (T < 1 || T > h->d.max_slots || first < 0 || first >= T) return fail(V2E_E_INVALID, "bad T / first");
    if (((uintptr_t)events & 15) != 0) return fail(V2E_E_INVALID, "events_out must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const EmuDev &d = h->d;
    const size_t fbytes = (size_t)d.n * frame_elem(dtype);
    if (last < 0 || last > T) last = T;
    if (first >= last) return fail(V2E_E_INVALID, "bad frame range");
    int rc;
    if (resume_emit) {
        // frame `first` was counted but not emitted (capacity abort): clear the abort and the slots
        // after it, keep slot `first`'s histograms, re-plan it against the new capacity.
        if (first + 1 < last && (rc = reset_slots(h, first + 1, last - first - 1, st))) return rc;
        CU(cudaMemsetAsync(d.abort_flag, 0, 2 * sizeof(int32_t), st));
    } else {
        // continuing after a multi-frame segment of the same step: its capacity abort (if any) must stay sticky
        if ((rc = reset_slots(h, first, last - first, st, ev_base_start != kChainBase))) return rc;
    }
    if (resume_emit && h->pr_T == 0) h->pr_T = h->pr_T_last;
    if (h->profile && first == 0) { memset(h->prof_used, 0, (size_t)d.max_slots * kProfKinds); h->prof_frames = T - first; }
    if (!resume_emit) {
        h->step_base = h->frame_counter;
        h->frame_counter += (uint32_t)T;
    }
    if (ev_base_start == kChainBase) emu_chain_step_kernel<<<1, 1, 0, st>>>(d, first);
    else emu_begin_step_kernel<<<1, 1, 0, st>>>(d, first, ev_base_start);
    for (int f = first; f < last; f++) {
        double tp = f == 0 ? t_previous : t_frames[f - 1];
        if (t_frames[f] < tp) return fail(V2E_E_INVALID, "frame times must be non-decreasing");
        FrameParams p = make_params(h, t_frames[f], tp, h->step_base + (uint32_t)f, capacity);
        const char *frame = (const char *)frames + (size_t)f * fbytes;
        const float *lr = leak_randn ? leak_randn + (size_t)f * d.n : nullptr;
        const float *sr = shot_rand ? shot_rand + (size_t)f * d.n : nullptr;
        if (resume_emit && f == first) {
            emu_plan_kernel<<<1, kThreads, 0, st>>>(d, p, f);   // only the plan has to be redone
        } else {
            const float *prn = nullptr;
            if (d.pr_noise) {
                if (h->pr_T < T) return fail(V2E_E_STATE, "v2e_emu_set_pr_noise must cover every frame of the step");
                p.pr_vrms_f = (float)h->pr_vrms[f];
                prn = h->pr_randn_dev ? h->pr_randn_dev + (size_t)f * d.n : nullptr;
            }
            if ((rc = enqueue_count(h, p, frame, dtype, lr, sr, 0, f, st, prn))) return rc;
            h->scidvs_started = 1;
        }
        if ((rc = enqueue_emit(h, p, f, events, st))) return rc;
        enqueue_null_bracket(h, f, st);
    }
    CU(cudaGetLastError());
    h->last_T = T;
    h->pr_T_last = h->pr_T;
    h->pr_T = 0;
    return V2E_OK;
}


extern "C" int v2e_emu_step(V2eEmu *h, const void *frames, int dtype, int T, const double *t_frames,
                            double t_previous, const float *leak_randn, const float *shot_rand,
                            float *events, uint64_t capacity, uint64_t ev_base_start, int first,
                            int resume_emit, void *stream) {
    if (!h || !frames || !t_frames || (!events && capacity)) return fail(V2E_E_INVALID, "null argument");
    if (!h->first_done) return fail(V2E_E_STATE, "v2e_emu_first_frame must run before v2e_emu_step");
    if (T < 1 || T > h->d.max_slots || first < 0 || first >= T) return fail(V2E_E_INVALID, "bad T / first");
    if (((uintptr_t)events & 15) != 0) return fail(V2E_E_INVALID, "events_out must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const EmuDev &d = h->d;
    int rc;
    if (resume_emit && h->last_fused == 1 && h->n_seg > 0) {
        // capacity abort at frame `first` of a scheduled step (the abort is sticky: nothing after it ran). The segment
        // that holds `first` is finished into the larger buffer -- a multi-frame segment still has its records and is
        // planned again, a frame-by-frame segment resumes at its counted-but-not-emitted frame -- then the rest of the
        // schedule runs.
        int i = 0;
        while (i < h->n_seg && !(h->sched[i].a <= first && first < h->sched[i].b)) i++;
        if (i == h->n_seg || (h->sched[i].kind == 0 && h->sched[i].a != first))
            return fail(V2E_E_STATE, "resume_emit: frame is not where the scheduled step stopped");
        remember_step(h, frames, dtype, T, t_frames, t_previous, events, capacity, h->ls.ev_base_start);
        CU(cudaMemsetAsync(d.abort_flag, 0, 2 * sizeof(int32_t), st));
        const V2eEmu::Seg g = h->sched[i];
        if (g.kind == 0) {
            CU(cudaMemsetAsync(d.cursor + (size_t)g.a * d.seg_stride, 0, (size_t)(g.b - g.a) * d.seg_stride * 4, st));
            if ((rc = enqueue_fused_emit(h, g.b - g.a, events, capacity, ev_base_start, nullptr, true, st, g.a, 0))) return rc;
        } else {
            h->frame_counter = h->step_base;
            if ((rc = step_classic(h, frames, dtype, T, t_frames, t_previous, nullptr, nullptr, events, capacity, ev_base_start,
                                   first, 1, stream, g.b))) return rc;
        }
        return run_schedule(h, i + 1, st);
    }
    bool want_fused = h->fused_enable && T >= 2 && first == 0 && !resume_emit && !leak_randn && !shot_rand &&
                      fused_config_ok(h, dtype);
    // back-off: input whose chunks keep breaking the assumption in many frames pays for the wasted speculative pass;
    // after such a chunk the next 1, 2, 4, ... 64 chunks go frame by frame before the multi-frame path is tried again
    if (want_fused && h->fused_skip > 0) { h->fused_skip--; want_fused = false; }
    if (want_fused) {
        if ((rc = fused_alloc(h))) return rc;
        if (h->fused_max_T >= T) {
            h->step_base = h->frame_counter;
            remember_step(h, frames, dtype, T, t_frames, t_previous, events, capacity, ev_base_start);
            if (h->profile) { memset(h->prof_used, 0, (size_t)d.max_slots * kProfKinds); h->prof_frames = T; }
            if ((rc = fused_upload_params(h, T, t_frames, t_previous, h->step_base, capacity, st))) return rc;
            CU(cudaMemsetAsync(d.abort_flag, 0, 2 * sizeof(int32_t), st));
            h->sched[0] = {0, 0, T};
            h->n_seg = 1;
            h->last_fused = 1;
            h->n_fused_chunks++;
            return run_schedule(h, 0, st);
        }
    }
    h->n_seg = 0;
    h->last_fused = 0;
    return step_classic(h, frames, dtype, T, t_frames, t_previous, leak_randn, shot_rand, events, capacity,
                        ev_base_start, first, resume_emit, stream);
}

extern "C" int v2e_emu_collect(V2eEmu *h, V2eFrameInfo *info, int T, int *frames_done,
                               uint64_t *rows_total, void *stream) {
    if (!h || !info || T < 1 || T > h->d.max_slots) return fail(V2E_E_INVALID, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    CU(cudaMemcpyAsync(h->ctrl_host, h->d.ctrl, (size_t)(T + 1) * sizeof(FrameCtrl), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h->abort_host, h->d.abort_flag, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int round = 0; h->abort_host[0] == kFusedFallback; round++) {
        // A multi-frame segment was rejected on the device at frame fb (refractory filter active there, or more than
        // kFusedMaxN events of one pixel): nothing of it was emitted or committed, nothing after it ran.
        const int fb = h->abort_host[1];
        h->n_fused_rejected++;
        h->last_reject_frame = fb;
        h->last_reject_max_n = (fb >= 0 && fb < T) ? h->ctrl_host[fb].max_n : -1;
        if (h->last_fused == 2) {                 // phase functions: the caller replays (identically on every rank)
            h->last_fused = 0;
            h->frame_counter = h->step_base;
            if (frames_done) *frames_done = fb;
            return fail(V2E_E_FALLBACK, "fused chunk rejected: replay it frame by frame");
        }
        // Re-schedule the segment: its count pass left every frame's maximum (exact up to fb, a prediction after it --
        // the state was speculative). Frames that break the assumption go frame by frame, the runs between them
        // through the multi-frame kernels again (each run still verifies itself: a wrong prediction costs another
        // round, never a wrong row). Same frames, same Philox frame indices, rows chained on the device.
        int i = 0;
        while (i < h->n_seg && !(h->sched[i].kind == 0 && h->sched[i].a <= fb && fb < h->sched[i].b)) i++;
        if (i == h->n_seg || round > T) return fail(V2E_E_STATE, "rejected frame outside the schedule");
        const V2eEmu::Seg g = h->sched[i];
        std::vector<V2eEmu::Seg> neu;
        int n_bad = 0;
        for (int f = g.a; f < g.b;) {
            auto bad = [&](int q) {
                const int m = h->ctrl_host[q].max_n;
                const double dt = h->ls.t_frames[q] - (q == 0 ? h->ls.t_previous : h->ls.t_frames[q - 1]);
                return q == fb || m > kFusedMaxN || m > h->d.iter_cap || (h->d.refr_on && m > 0 && h->d.refr_d > dt / (double)m);
            };
            int e = f;
            if (bad(f)) { while (e < g.b && bad(e)) { e++; n_bad++; } neu.push_back({1, f, e}); }
            else {
                while (e < g.b && !bad(e)) e++;
                if (e - f >= 2) neu.push_back({0, f, e});
                else if (!neu.empty() && neu.back().kind == 1) neu.back().b = e;     // a lone good frame joins its neighbours
                else neu.push_back({1, f, e});
            }
            f = e;
        }
        // merge adjacent frame-by-frame segments
        std::vector<V2eEmu::Seg> merged;
        for (const auto &q : neu) {
            if (!merged.empty() && merged.back().kind == 1 && q.kind == 1) merged.back().b = q.b;
            else merged.push_back(q);
        }
        if ((size_t)h->n_seg - 1 + merged.size() > (size_t)h->d.max_slots + 2) return fail(V2E_E_STATE, "schedule overflow");
        std::vector<V2eEmu::Seg> all(h->sched, h->sched + i);
        all.insert(all.end(), merged.begin(), merged.end());
        all.insert(all.end(), h->sched + i + 1, h->sched + h->n_seg);
        for (size_t k = 0; k < all.size(); k++) h->sched[k] = all[k];
        h->n_seg = (int)all.size();
        if (4 * n_bad > g.b - g.a) {              // the assumption fails in many frames of this input: back off
            h->fused_penalty = h->fused_penalty ? (h->fused_penalty < 64 ? 2 * h->fused_penalty : 64) : 1;
            h->fused_skip = h->fused_penalty;
        }
        CU(cudaMemsetAsync(h->d.abort_flag, 0, 2 * sizeof(int32_t), st));
        int rc = run_schedule(h, i, st);
        if (rc) return rc;
        CU(cudaMemcpyAsync(h->ctrl_host, h->d.ctrl, (size_t)(T + 1) * sizeof(FrameCtrl), cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(h->abort_host, h->d.abort_flag, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    int status = h->abort_host[0], done = status ? h->abort_host[1] : T;
    // a whole chunk accepted (a rejected chunk can also end as one segment: frame by frame, which is no reset)
    if (!status && h->last_fused == 1 && h->n_seg == 1 && h->sched[0].kind == 0) h->fused_penalty = 0;
    if (!status && h->last_fused == 1 && h->n_seg > 0) {
        for (int k = 0; k < h->n_seg; k++)
            (h->sched[k].kind == 0 ? h->n_frames_multi : h->n_frames_single) += h->sched[k].b - h->sched[k].a;
        h->n_seg = 0;                                  // counted once
        h->last_fused = 0;
    }
    uint64_t rows = 0;
    for (int f = 0; f < T; f++) {
        const FrameCtrl &c = h->ctrl_host[f];
        V2eFrameInfo &o = info[f];
        o.max_n = c.max_n;
        o.filter_active = c.filter_active;
        o.n_on = c.n_on; o.n_off = c.n_off;
        o.n_shot_on = c.n_shot_on; o.n_shot_off = c.n_shot_off;
        o.n_events = c.n_events;
        o.cs_steps = c.cs_steps;
        o.ev_base = c.ev_base;
        if (f < done) rows = c.ev_base + c.n_events;
    }
    if (frames_done) *frames_done = done;
    if (rows_total) *rows_total = rows;
    if (status == V2E_E_CAPACITY) return fail(V2E_E_CAPACITY, "event buffer too small");
    if (status == V2E_E_ITER_CAP) return fail(V2E_E_ITER_CAP, "a pixel exceeded iter_cap events in one frame");
    return V2E_OK;
}

extern "C" int v2e_emu_time_fused(V2eEmu *h, const void *frames, int dtype, int T, const double *t_frames,
                                  double t_previous, float *events, uint64_t capacity, int K, float *us_chunk,
                                  float *us_update, void *stream) {
    if (!h || !frames || !t_frames || !events || K < 1 || !us_chunk) return fail(V2E_E_INVALID, "bad argument");
    if (!h->first_done) return fail(V2E_E_STATE, "v2e_emu_first_frame must run first");
    if (T < 2 || T > h->d.max_slots) return fail(V2E_E_INVALID, "bad T");
    if (!fused_config_ok(h, dtype)) return fail(V2E_E_UNSUPPORTED, "configuration does not qualify for the fused path");
    int rc;
    if ((rc = fused_alloc(h))) return rc;
    if (h->fused_max_T < T) return fail(V2E_E_UNSUPPORTED, "fused path: T exceeds the record lists");
    cudaStream_t st = (cudaStream_t)stream;
    cudaEvent_t e[4];
    for (int i = 0; i < 4; i++) cudaEventCreate(&e[i]);
    rc = fused_upload_params(h, T, t_frames, t_previous, h->frame_counter, capacity, st);
    const int prof = h->profile;
    h->profile = 0;
    for (int k = -1; k < K && !rc; k++) {          // k = -1: warm-up
        if (k == 0) cudaEventRecord(e[0], st);
        rc = reset_slots(h, 0, T, st);
        if (!rc) rc = enqueue_fused_count(h, frames, T, st);
        if (!rc) rc = enqueue_fused_emit(h, T, events, capacity, 0, nullptr, false, st);
    }
    cudaEventRecord(e[1], st);
    if (!rc) rc = reset_slots(h, 0, T, st);
    cudaEventRecord(e[2], st);
    for (int k = 0; k < K && !rc; k++)
        rc = h->d.state_f64 ? launch_fused_update<double>(h, h->d, h->ff_dev, (const uint8_t *)frames, T, st)
                            : launch_fused_update<float>(h, h->d, h->ff_dev, (const uint8_t *)frames, T, st);
    cudaEventRecord(e[3], st);
    h->profile = prof;
    if (!rc) rc = reset_slots(h, 0, T, st);
    cudaError_t ce = cudaStreamSynchronize(st);
    float ms0 = 0.f, ms1 = 0.f;
    cudaEventElapsedTime(&ms0, e[0], e[1]);
    cudaEventElapsedTime(&ms1, e[2], e[3]);
    for (int i = 0; i < 4; i++) cudaEventDestroy(e[i]);
    if (rc) return rc;
    if (ce != cudaSuccess) return fail(V2E_E_CUDA, "v2e_emu_time_fused: %s", cudaGetErrorString(ce));
    *us_chunk = ms0 * 1e3f / (float)K;
    if (us_update) *us_update = ms1 * 1e3f / (float)K;
    return V2E_OK;
}

// ---- single-frame phases (slot 0) ---------------------------------------------------------------
extern "C" int v2e_emu_phase_count(V2eEmu *h, const void *frame, int dtype, double t_frame,
                                   double t_previous, const float *lr, const float *sr, int shot_pending,
                                   uint64_t capacity, uint64_t ev_base_start, void *stream) {
    if (!h || !frame) return fail(V2E_E_INVALID, "null argument");
    if (!h->first_done) return fail(V2E_E_STATE, "v2e_emu_first_frame must run first");
    if (t_frame < t_previous) return fail(V2E_E_INVALID, "frame times must be non-decreasing");
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if ((rc = reset_slots(h, 0, 1, st))) return rc;
    emu_begin_step_kernel<<<1, 1, 0, st>>>(h->d, 0, ev_base_start);
    FrameParams p = make_params(h, t_frame, t_previous, h->frame_counter++, capacity);
    h->last_dt = p.dt;
    const float *prn = nullptr;
    if (h->d.pr_noise) {
        if (h->pr_T < 1) return fail(V2E_E_STATE, "v2e_emu_set_pr_noise must precede v2e_emu_phase_count");
        p.pr_vrms_f = (float)h->pr_vrms[0];
        prn = h->pr_randn_dev;
        h->pr_T = 0;
    }
    if ((rc = enqueue_count(h, p, frame, dtype, lr, sr, shot_pending, 0, st, prn))) return rc;
    h->scidvs_started = 1;
    CU(cudaGetLastError());
    h->last_T = 1;
    return V2E_OK;
}

// ---- pixel-sharded operation: update only, reduce max_n over ranks, then filter / plan ----------------
extern "C" int v2e_emu_phase_update(V2eEmu *h, const void *frame, int dtype, double t_frame, double t_previous,
                                    const float *lr, const float *sr, uint64_t capacity, uint64_t ev_base_start,
                                    void *stream) {
    if (!h || !frame) return fail(V2E_E_INVALID, "null argument");
    if (!h->first_done) return fail(V2E_E_STATE, "v2e_emu_first_frame must run first");
    if (t_frame < t_previous) return fail(V2E_E_INVALID, "frame times must be non-decreasing");
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if ((rc = reset_slots(h, 0, 1, st))) return rc;
    emu_begin_step_kernel<<<1, 1, 0, st>>>(h->d, 0, ev_base_start);
    FrameParams p = make_params(h, t_frame, t_previous, h->frame_counter++, capacity);
    h->last_dt = p.dt;
    // shot_pending = 1 makes enqueue_count run the update kernel alone when there is no refractory
    // period; with one, the filter must wait for the reduced max, so launch the update kernel directly
    const EmuDev &d = h->d;
    if (d.rng_mode == 0 && d.leak_on && !lr) return fail(V2E_E_INVALID, "leak_randn field required in replay mode");
    if (d.csdvs) return fail(V2E_E_UNSUPPORTED, "centre-surround model: a pixel-sharded handle is stepped with v2e_emu_cs_* (cs_halo_rows > 0)");
    if (d.scidvs || d.pr_noise) return fail(V2E_E_UNSUPPORTED, "pixel sharding with scidvs / photoreceptor_noise is not built");
    rc = d.state_f64 ? launch_update<double>(h, p, frame, dtype, lr, sr, 0, 0, 0, st)
                     : launch_update<float>(h, p, frame, dtype, lr, sr, 0, 0, 0, st);
    if (rc) return rc;
    CU(cudaGetLastError());
    h->last_T = 1;
    return V2E_OK;
}

extern "C" int32_t *v2e_emu_max_n_dev(V2eEmu *h) { return h ? &h->d.ctrl[0].max_n : nullptr; }

// ---- pixel-sharded centre-surround model (see include/v2e_b200.h) ----------------------------------
extern "C" int v2e_emu_cs_begin(V2eEmu *h, const void *frame, int dtype, double t_frame, double t_previous,
                                uint64_t capacity, uint64_t ev_base_start, int *num_steps, void *stream) {
    if (!h || !frame || !num_steps) return fail(V2E_E_INVALID, "null argument");
    if (!h->first_done) return fail(V2E_E_STATE, "v2e_emu_first_frame must run first");
    if (!h->d.csdvs || !h->cs_K) return fail(V2E_E_STATE, "not a pixel-sharded centre-surround handle (cs_halo_rows)");
    if (h->d.scidvs || h->d.pr_noise) return fail(V2E_E_UNSUPPORTED, "pixel sharding with scidvs / photoreceptor_noise is not built");
    if (t_frame < t_previous) return fail(V2E_E_INVALID, "frame times must be non-decreasing");
    cudaStream_t st = (cudaStream_t)stream;
    const EmuDev &d = h->d;
    int rc;
    if ((rc = reset_slots(h, 0, 1, st))) return rc;
    emu_begin_step_kernel<<<1, 1, 0, st>>>(d, 0, ev_base_start);
    FrameParams p = make_params(h, t_frame, t_previous, h->frame_counter++, capacity);
    h->last_dt = p.dt;
    if ((rc = cs_plan(h, p, &h->cs_num_steps, &h->cs_alpha_p, &h->cs_alpha_h))) return rc;
    const int g = grid_for(d);
    switch (dtype) {
        case V2E_U8: emu_lp_kernel<V2E_U8><<<g, kThreads, 0, st>>>(d, p, frame); break;
        case V2E_F32: emu_lp_kernel<V2E_F32><<<g, kThreads, 0, st>>>(d, p, frame); break;
        case V2E_F64: emu_lp_kernel<V2E_F64><<<g, kThreads, 0, st>>>(d, p, frame); break;
        default: return fail(V2E_E_INVALID, "bad frame dtype");
    }
    CU(cudaMemsetAsync(d.cs_max, 0, (size_t)h->cs_num_steps * sizeof(unsigned long long), st));
    CU(cudaMemsetAsync(d.cs_done, 0, sizeof(int32_t), st));
    CU(cudaGetLastError());
    h->cs_p = p;
    h->cs_pending = 1;
    *num_steps = h->cs_num_steps;
    h->last_T = 1;
    h->last_fused = 0;
    return V2E_OK;
}
extern "C" double *v2e_emu_cs_send_dev(V2eEmu *h) { return h ? h->cs_send : nullptr; }
extern "C" double *v2e_emu_cs_recv_dev(V2eEmu *h) { return h ? h->cs_recv : nullptr; }
extern "C" uint64_t *v2e_emu_cs_max_dev(V2eEmu *h) { return h ? (uint64_t *)h->d.cs_max : nullptr; }
extern "C" int v2e_emu_cs_pack(V2eEmu *h, void *stream) {
    if (!h || !h->cs_K) return fail(V2E_E_STATE, "not a pixel-sharded centre-surround handle");
    emu_csdvs_pack_kernel<<<148, 256, 0, (cudaStream_t)stream>>>(h->d, h->cs_send, h->cs_K);
    CU(cudaGetLastError());
    return V2E_OK;
}
extern "C" int v2e_emu_cs_unpack(V2eEmu *h, void *stream) {
    if (!h || !h->cs_K) return fail(V2E_E_STATE, "not a pixel-sharded centre-surround handle");
    emu_csdvs_unpack_kernel<<<148, 256, 0, (cudaStream_t)stream>>>(h->d, h->cs_recv, h->cs_recv + (size_t)h->cs_K * h->d.W, h->cs_K);
    CU(cudaGetLastError());
    return V2E_OK;
}
extern "C" int v2e_emu_cs_unpack_from(V2eEmu *h, const double *rows_above_dev, const double *rows_below_dev, void *stream) {
    if (!h || !h->cs_K) return fail(V2E_E_STATE, "not a pixel-sharded centre-surround handle");
    emu_csdvs_unpack_kernel<<<148, 256, 0, (cudaStream_t)stream>>>(h->d, rows_above_dev, rows_below_dev, h->cs_K);
    CU(cudaGetLastError());
    return V2E_OK;
}
extern "C" int v2e_emu_cs_chunk(V2eEmu *h, int s0, int s1, void *stream) {
    if (!h || !h->cs_pending) return fail(V2E_E_STATE, "v2e_emu_cs_begin must precede v2e_emu_cs_chunk");
    if (s0 < 0 || s1 <= s0 || s1 > h->cs_num_steps || s1 - s0 > h->cs_K) return fail(V2E_E_INVALID, "bad chunk of Euler steps");
    const EmuDev &d = h->d;
    if (!cs_launch_iter(h, h->cs_alpha_p, h->cs_alpha_h, s0, s1, 1, 0, (cudaStream_t)stream)) {
        const int gs = (d.n + kThreads - 1) / kThreads;
        for (int s = s0; s < s1; s++)
            emu_csdvs_step_kernel<<<gs, kThreads, 0, (cudaStream_t)stream>>>(d, h->cs_alpha_p, h->cs_alpha_h, s, s - s0, 1);
    }
    CU(cudaGetLastError());
    return V2E_OK;
}
extern "C" int v2e_emu_cs_advance(V2eEmu *h, int s0, int s1, void *stream) {
    if (!h || !h->cs_pending) return fail(V2E_E_STATE, "v2e_emu_cs_begin must precede v2e_emu_cs_advance");
    emu_csdvs_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(h->d, s0, s1, 0);
    CU(cudaGetLastError());
    return V2E_OK;
}
extern "C" int v2e_emu_cs_update(V2eEmu *h, const void *frame, int dtype, const float *lr, const float *sr, void *stream) {
    if (!h || !frame) return fail(V2E_E_INVALID, "null argument");
    if (!h->cs_pending) return fail(V2E_E_STATE, "v2e_emu_cs_begin must precede v2e_emu_cs_update");
    const EmuDev &d = h->d;
    if (d.rng_mode == 0 && d.leak_on && !lr) return fail(V2E_E_INVALID, "leak_randn field required in replay mode");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = d.state_f64 ? launch_update<double>(h, h->cs_p, frame, dtype, lr, sr, 0, 0, 1, st)
                         : launch_update<float>(h, h->cs_p, frame, dtype, lr, sr, 0, 0, 1, st);
    if (rc) return rc;
    CU(cudaGetLastError());
    h->cs_pending = 0;
    return V2E_OK;
}

extern "C" int v2e_emu_phase_filter(V2eEmu *h, double t_frame, double t_previous, uint64_t capacity, int do_plan,
                                    void *stream) {
    if (!h) return fail(V2E_E_INVALID, "null handle");
    cudaStream_t st = (cudaStream_t)stream;
    FrameParams p = make_params(h, t_frame, t_previous, 0, capacity);
    const EmuDev &d = h->d;
    if (d.refr_on) emu_filter_kernel<<<list_grid(d), kThreads, 0, st>>>(d, p, 0, do_plan);
    else if (do_plan) emu_plan_kernel<<<1, kThreads, 0, st>>>(d, p, 0);
    CU(cudaGetLastError());
    return V2E_OK;
}

extern "C" int v2e_emu_read_counts(V2eEmu *h, int32_t *max_n, uint32_t *counts, int counts_cap, void *stream) {
    if (!h || !max_n) return fail(V2E_E_INVALID, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    CU(cudaMemcpyAsync(h->ctrl_host, h->d.ctrl, sizeof(FrameCtrl), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    int32_t m = h->ctrl_host[0].max_n;
    *max_n = m;
    if (m > h->d.iter_cap) return fail(V2E_E_ITER_CAP, "a pixel exceeded iter_cap events in one frame");
    if (counts && m > 0) {
        if (2 * m > counts_cap) return fail(V2E_E_INVALID, "counts buffer too small");
        // which histogram applies: the refractory filter is active iff
        // refractory_period_s > delta_time / max_n (emulator.py:792, 830), same doubles as make_ts()
        const uint32_t *src = h->d.hist_pre;
        if (h->d.refr_on && h->d.refr_d > h->last_dt / (double)m) src = h->d.hist_post;
        CU(cudaMemcpy(counts, src, (size_t)2 * m * 4, cudaMemcpyDeviceToHost));
    }
    return V2E_OK;
}

extern "C" int v2e_emu_phase_shot(V2eEmu *h, const void *frame, int dtype, double t_frame, double t_previous,
                                  const float *sr, uint64_t capacity, void *stream) {
    if (!h || !frame || !sr) return fail(V2E_E_INVALID, "null argument");
    FrameParams p = make_params(h, t_frame, t_previous, 0, capacity);
    int rc = launch_shot(h, p, frame, dtype, sr, 0, (cudaStream_t)stream);
    if (rc) return rc;
    CU(cudaGetLastError());
    return V2E_OK;
}

extern "C" int v2e_emu_phase_emit(V2eEmu *h, double t_frame, double t_previous, float *events,
                                  uint64_t capacity, void *stream) {
    if (!h) return fail(V2E_E_INVALID, "null handle");
    if (((uintptr_t)events & 15) != 0) return fail(V2E_E_INVALID, "events_out must be 16-byte aligned");
    FrameParams p = make_params(h, t_frame, t_previous, 0, capacity);
    int rc = enqueue_emit(h, p, 0, events, (cudaStream_t)stream);
    if (rc) return rc;
    CU(cudaGetLastError());
    return V2E_OK;
}

extern "C" int v2e_emu_profile(V2eEmu *h, int enable) {
    if (!h) return fail(V2E_E_INVALID, "null handle");
    if (enable && !h->ev) {
        int n = h->d.max_slots * kProfKinds * 2;
        h->ev = new cudaEvent_t[n];
        for (int i = 0; i < n; i++) CU(cudaEventCreate(&h->ev[i]));
        h->prof_used = new unsigned char[h->d.max_slots * kProfKinds]();
    }
    h->profile = enable ? 1 : 0;
    return V2E_OK;
}

static int profile_read_n(V2eEmu *h, float *ms_sum, int *launches, int kinds, void *stream) {
    if (!h || !h->ev || !ms_sum || !launches) return fail(V2E_E_INVALID, "profiling not enabled");
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    for (int k = 0; k < kinds; k++) { ms_sum[k] = 0.f; launches[k] = 0; }
    for (int s = 0; s < h->d.max_slots; s++)
        for (int k = 0; k < kinds; k++)
            if (h->prof_used[s * kProfKinds + k]) {
                float ms = 0.f;
                CU(cudaEventElapsedTime(&ms, h->ev[(s * kProfKinds + k) * 2], h->ev[(s * kProfKinds + k) * 2 + 1]));
                ms_sum[k] += ms;
                launches[k] += 1;
            }
    return V2E_OK;
}
extern "C" int v2e_emu_profile_read(V2eEmu *h, float *ms_sum3, int *launches3, void *stream) {
    return profile_read_n(h, ms_sum3, launches3, 3, stream);
}
extern "C" int v2e_emu_profile_read4(V2eEmu *h, float *ms_sum4, int *launches4, void *stream) {
    return profile_read_n(h, ms_sum4, launches4, 4, stream);
}

// Average duration of the update kernel: K back-to-back launches on the given frame and the handle's CURRENT
// state, between ONE pair of CUDA events (no per-launch bracket, whose own cost is several microseconds). The
// launches store lp / base into scratch arrays, so every one of them does exactly the work of the real launch
// (same loads, same stores, same event density) and the handle's state is untouched; the per-frame scratch
// (records, active list, histograms of slot 0) is reset by the next v2e_emu_step as usual.
extern "C" int v2e_emu_time_update(V2eEmu *h, const void *frame_dev, int dtype, double t_frame, double t_previous,
                                   int K, float *us_per_launch, void *stream) {
    if (!h || !frame_dev || !us_per_launch || K < 1) return fail(V2E_E_INVALID, "bad argument");
    if (!h->first_done) return fail(V2E_E_STATE, "v2e_emu_first_frame must run first");
    if (h->d.rng_mode != 1 || h->d.csdvs || h->d.scidvs || h->d.pr_noise)
        return fail(V2E_E_UNSUPPORTED, "v2e_emu_time_update: device RNG, plain pixel model only");
    cudaStream_t st = (cudaStream_t)stream;
    EmuDev &d = h->d;
    const size_t bytes = (size_t)d.units * kUnitPx * h->state_elem;
    void *lp2 = nullptr, *base2 = nullptr;
    CU(cudaMalloc(&lp2, bytes));
    if (cudaMalloc(&base2, bytes) != cudaSuccess) { cudaFree(lp2); return fail(V2E_E_CUDA, "cudaMalloc failed"); }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    int rc = reset_slots(h, 0, 1, st);
    d.lp_out = lp2;
    d.base_out = base2;
    FrameParams p = make_params(h, t_frame, t_previous, h->frame_counter, 0);
    for (int i = 0; i < 2 && !rc; i++)          // warm-up
        rc = d.state_f64 ? launch_update<double>(h, p, frame_dev, dtype, nullptr, nullptr, 0, 0, 0, st)
                         : launch_update<float>(h, p, frame_dev, dtype, nullptr, nullptr, 0, 0, 0, st);
    cudaEventRecord(e0, st);
    for (int i = 0; i < K && !rc; i++)
        rc = d.state_f64 ? launch_update<double>(h, p, frame_dev, dtype, nullptr, nullptr, 0, 0, 0, st)
                         : launch_update<float>(h, p, frame_dev, dtype, nullptr, nullptr, 0, 0, 0, st);
    cudaEventRecord(e1, st);
    d.lp_out = d.lp;
    d.base_out = d.base;
    cudaError_t ce = cudaStreamSynchronize(st);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(lp2);
    cudaFree(base2);
    if (!rc) rc = reset_slots(h, 0, 1, st);
    if (rc) return rc;
    if (ce != cudaSuccess) return fail(V2E_E_CUDA, "v2e_emu_time_update: %s", cudaGetErrorString(ce));
    *us_per_launch = ms * 1e3f / (float)K;
    return V2E_OK;
}

extern "C" int v2e_emu_state_is_f64(V2eEmu *h) { return h ? h->d.state_f64 : 0; }

extern "C" void *v2e_emu_state_ptr(V2eEmu *h, int which) {
    if (!h) return nullptr;
    switch (which) {
        case 0: return h->d.lp;
        case 1: return h->d.base;
        case 2: return h->d.pos_thres;
        case 3: return h->d.neg_thres;
        case 4: return h->d.noise_rate;
        case 5: return h->d.tmem;
        case 6: {
            if (!h->d.surround && !h->d.cs_bufs) return nullptr;
            int32_t cur = 0;
            cudaDeviceSynchronize();
            cudaMemcpy(&cur, h->d.cs_cur, sizeof(cur), cudaMemcpyDeviceToHost);
            if (h->d.cs_bufs) return h->d.cs_bufs + (size_t)cur * h->d.cs_stride;
            return cur ? h->d.surround2 : h->d.surround;
        }
        case 7: return h->d.hp;
        case 8: return h->d.noise_arr;
        case 9: return h->d.tau_arr;
    }
    return nullptr;
}

extern "C" int v2e_emu_get_state(V2eEmu *h, int which, void *dst, int *elem_size) {
    if (!h || !dst) return fail(V2E_E_INVALID, "null argument");
    void *src = v2e_emu_state_ptr(h, which);
    if (!src) return fail(V2E_E_STATE, "state array not allocated for this configuration");
    int es = (which <= 1 || which == 7) ? (int)h->state_elem : (which == 6 ? 8 : 4);
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(dst, src, (size_t)h->d.n * es, cudaMemcpyDeviceToHost));
    if (elem_size) *elem_size = es;
    return V2E_OK;
}
