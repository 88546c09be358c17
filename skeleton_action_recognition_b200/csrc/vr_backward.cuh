// vr_backward.cuh -- gradients of the VirtualRadar layer with respect to its two radar parameters
// (`wavelength`, `radar_location`; reference layers/virtual_radar.py:40-41, 65-69: the constructor's
// train_wavelength / train_radar_location flags make them trainable nn.Parameters and PyTorch autograd
// differentiates forward(), :79-134).  Two kernels:
//
//   vr_stft_adjoint_kernel   grad_out (N, 256, F) and the saved complex baseband signal z (N, T, 2)
//                            -> dL/dz (N, T, 2): per frame, X = FFT(hann * zp); G = g * X / (|X| (|X| + 1e-6))
//                            (log-magnitude and fftshift, :126-133); dL/dzp = hann * conj(FFT(conj(G))) (the
//                            adjoint of the windowed DFT, :124-125); overlap-add through the reflect padding, in
//                            owner form: a CTA owns a segment of samples and adds every contribution to it in a fixed
//                            order (adj_seg_frames), so dL/dz is bitwise reproducible and independent of the batch.
//   vr_synth_adjoint_kernel  dL/dz and x -> dL/dwavelength, dL/dradar_location (and, on request, dL/dx): per (sequence, time step, body,
//                            bone) the forward geometry is recomputed (range and phase with the forward's exact
//                            float32 rounding, the rest in float64) and the analytic derivatives of
//                            z = sum amp * exp(j theta) are accumulated in float64; the block partials of the
//                            parameter gradients are added in block order by the last block (synth_adjoint_reduce).
//
// theta = 4 pi d / lambda reaches 1e4..1e5 rad, so dtheta/dlambda = -theta/lambda is of order 1e7..1e8: the
// reference's float32 autograd result carries relative errors of 1e-3 and more; these kernels are checked
// against the float64 autograd of the oracle (tests/test_backward_gpu.py).
#pragma once
#include "vr_kernels.cuh"
#include "vr_pad_frames.cuh"

namespace vr {

struct BwdParams {
    const float* x;              // (N,3,T,V,M)
    const float* iq;             // (N,T,2) saved by the forward (vr_forward_debug_f32)
    const float* gout;           // (N,256,F)
    float* gz;                   // (N,T,2) dL/dz: every sample written once by the adjoint STFT
    double* gparams;             // [dL/dlambda, dL/dLx, dL/dLy, dL/dLz]: the launch's total is added by its last block
    double* part;                // this launch's slot of g_param_partials: 4 partials per block
    unsigned* count;             // and its counter of finished blocks (0 between launches)
    int seg_len, segs;           // adjoint STFT: samples per segment, segments per sequence (adjoint_plan)
    float* gx;                   // optional dL/dx (N / views,3,T,V,M), zeroed before the launch; nullptr = not wanted
    const float* lam_ptr;        // 1 wavelength and 1 location, or (VR_FLAG_PER_SEQUENCE) N and N x 3
    const float* loc_ptr;
    long long ps_segs;           // VR_FLAG_PER_SEQUENCE: segments per sequence of the per-sequence reduction (part = their
                                 // partials, gparams = N x 4 gradients); 0 = one reduction over the batch
    long long N, T;
    int V, M, E, F, hop, VM;
    int fma_range;
    float inv_E;
    const double* coef;          // vr_synth_adjoint_ups_kernel: (N, ups_T-1, 4, 3*V*M) cubics of vr_pad_frames_kernel; T = ups_K * ups_T
    double ups_ratio;
    int ups_T;
    uint16_t src[NG * MAX_EG], dst[NG * MAX_EG];
    int views;                   // VR_FLAG_VIEWS: radars per sequence R (vr_synth_adjoint_ps_kernel); x and coef hold N / R
                                 // sequences, output n reads sequence n / R.  (Last: the other fields keep their offsets.)
};

// ---- owner-form plan of the adjoint STFT -----------------------------------------------------------------------------
// The samples of a sequence are cut into segments of seg_len samples; one CTA at a time owns a segment.  Frame f covers the
// padded positions u in [f hop, f hop + 256); sample t sits at u = t + 128, and through the reflect padding also at u = 128 - t
// (1 <= t <= 128) and u = 128 + 2 (T - 1) - t (T - 129 <= t <= T - 2).  A segment transforms every frame that reaches one of
// its samples by any of the three, including halo frames its neighbours transform as well, and adds each sample's
// contributions frame by frame in increasing order, direct position before the mirrors: the order depends on neither the
// segment cut nor the batch.
constexpr int ADJ_SEG_MAX = 4096;          // samples per segment: the float2 accumulators live in shared memory (32 KB,
                                           // 56 KB per CTA with the FFT buffers: four CTAs per SM)
constexpr int ADJ_SEG_MIN = 1024;          // a cut costs 256 / hop - 1 halo frames; below this it would cost more than 1/5

// the frames [lo, hi] that reach samples [s0, s1) (lo > hi: none)
__host__ __device__ inline void adj_seg_frames(long long s0, long long s1, long long T, int F, int hop, int& lo, int& hi) {
    long long ulo = s0 + 128, uhi = s1 - 1 + 128;                                           // direct positions
    const long long a = s0 > 1 ? s0 : 1, b = s1 - 1 < 128 ? s1 - 1 : 128;                   // left mirror
    if (a <= b) { ulo = ulo < 128 - b ? ulo : 128 - b; uhi = uhi > 128 - a ? uhi : 128 - a; }
    const long long c = s0 > T - 129 ? s0 : T - 129, d = s1 - 1 < T - 2 ? s1 - 1 : T - 2;  // right mirror
    if (c <= d) { ulo = ulo < 126 + 2 * T - d ? ulo : 126 + 2 * T - d; uhi = uhi > 126 + 2 * T - c ? uhi : 126 + 2 * T - c; }
    const long long f0 = ulo - 255 <= 0 ? 0 : (ulo - 255 + hop - 1) / hop, f1 = uhi / hop;
    lo = (int)f0;
    hi = (int)(f1 < F - 1 ? f1 : F - 1);
}

// The host's choice: enough segments that the batch fills the machine (about four CTAs per SM), none shorter than
// ADJ_SEG_MIN unless it is the whole sequence, none longer than ADJ_SEG_MAX.  The result does not depend on it.
inline void adjoint_plan(long long N, long long T, int sm_count, int& seg_len, int& segs) {
    const long long want = (4ll * sm_count + N - 1) / N;
    long long s = (T + ADJ_SEG_MIN - 1) / ADJ_SEG_MIN;
    s = want < s ? want : s;
    const long long smin = (T + ADJ_SEG_MAX - 1) / ADJ_SEG_MAX;
    s = s > smin ? s : smin;
    s = s > 1 ? s : 1;
    long long len = (T + s - 1) / s;
    len = (len + 31) / 32 * 32;
    if (len > ADJ_SEG_MAX) len = ADJ_SEG_MAX;
    seg_len = (int)len;
    segs = (int)((T + len - 1) / len);
}

// Per-sequence parameter gradients (VR_FLAG_PER_SEQUENCE): steps per segment of the reduction (one per lane of a warp), and
// the segments of a T-step sequence.  Depends on nothing but T.
constexpr int PS_SEG = 32;
inline long long ps_segments(long long T) { return (T + PS_SEG - 1) / PS_SEG; }

#ifdef __CUDACC__
// 256-point forward DFT (e^{-j...}) of one frame by one warp.  In: v[q] = sample lane + 32 q.  Out: v holds
// the bins bwd_bin(lane, j), j = 0..7.  Same radix 8 x 8 x 4 decomposition as the forward kernel's STFT.
__device__ __forceinline__ int bwd_bin(int lane, int j) {
    const int k1 = lane >> 2, b4 = lane & 3;
    return k1 + 8 * (b4 + 4 * (j >> 2)) + 64 * (j & 3);
}
__device__ __forceinline__ void bwd_fft256(c2 (&v)[8], float2* __restrict__ xch, const float4* __restrict__ tw1,
                                           const float4* __restrict__ tw2, int lane) {
    const int k1 = lane >> 2, b4 = lane & 3;
    dft8(v);
#pragma unroll
    for (int q = 1; q < 8; ++q) v[q] = pcmul(v[q], tw1[(q - 1) * 32 + lane]);
    __syncwarp();
#pragma unroll
    for (int q = 0; q < 8; ++q) xch[q * XCH_STRIDE + lane] = v[q];
    __syncwarp();
#pragma unroll
    for (int a = 0; a < 8; ++a) v[a] = xch[k1 * XCH_STRIDE + 4 * a + b4];
    dft8(v);
#pragma unroll
    for (int c = 1; c < 8; ++c) v[c] = pcmul(v[c], tw2[(c - 1) * 4 + b4]);
    __syncwarp();
#pragma unroll
    for (int c = 0; c < 8; ++c) xch[k1 * XCH_STRIDE + 4 * c + b4] = v[c];
    __syncwarp();
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
        const int c = b4 + 4 * hh;
        const float4* src4 = reinterpret_cast<const float4*>(&xch[k1 * XCH_STRIDE + 4 * c]);
        const float4 p01 = src4[0], p23 = src4[1];
        dft4(make_float2(p01.x, p01.y), make_float2(p01.z, p01.w), make_float2(p23.x, p23.y),
             make_float2(p23.z, p23.w), v[4 * hh], v[4 * hh + 1], v[4 * hh + 2], v[4 * hh + 3]);
    }
    __syncwarp();
}
__device__ __forceinline__ int bwd_reflect(int t, int T) {       // nnAudio center=True, pad_mode='reflect'
    t = t < 0 ? -t : t;
    return t >= T ? 2 * (T - 1) - t : t;
}

constexpr int BWD_WARPS = 8;

// One CTA per (sequence, segment) job.  Round after round, warp w transforms frame lo + round * BWD_WARPS + w and parks its
// Hann-weighted contributions in its slot of shared memory (tr); after a barrier the segment's samples that the round reaches
// take them from the slots in frame order into their float2 accumulators (acc, dynamic shared memory: seg_len entries).
// Each sample of gz is written once at the end of its job; a sample no frame covers (hop > 256) gets exactly 0.
__global__ void __launch_bounds__(BWD_WARPS * 32) vr_stft_adjoint_kernel(const __grid_constant__ BwdParams p) {
    __shared__ float4 tw1[7 * 32 + 7 * 4];
    __shared__ float hann[NFFT];
    // per warp: the FFT exchange buffer, also the parking place of G between the two FFTs and, after the second, the
    // frame's contribution slot that the gather reads (every use is separated from the next by a __syncwarp inside
    // bwd_fft256 or the round's __syncthreads)
    __shared__ float2 xch_all[BWD_WARPS][8 * XCH_STRIDE];
    static_assert(8 * XCH_STRIDE >= NFFT, "a frame's 256 values fit the exchange buffer");
    extern __shared__ float2 acc[];
    float4* tw2 = tw1 + 7 * 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < 7 * 32 + 7 * 4; i += blockDim.x) {
        const int e = i < 7 * 32 ? (i & 31) * ((i >> 5) + 1) : 8 * ((i - 7 * 32) & 3) * (((i - 7 * 32) >> 2) + 1);
        float sn, cs;
        sincospif((float)(e & 255) * (2.0f / NFFT), &sn, &cs);
        tw1[i] = make_float4(cs, -sn, sn, cs);
    }
    for (int i = tid; i < NFFT; i += blockDim.x) hann[i] = fmaf(-0.5f, cospif((float)i * (2.0f / NFFT)), 0.5f);
    __syncthreads();
    float2* xch = xch_all[warp];
    float2* tr = xch_all[warp];
    const int T = (int)p.T, hop = p.hop, h = NFFT / 2;
    const long long jobs = p.N * (long long)p.segs;
    for (long long job = blockIdx.x; job < jobs; job += gridDim.x) {
        const long long n = job / p.segs;
        const int s0 = (int)(job - n * p.segs) * p.seg_len;
        const int s1 = s0 + p.seg_len < T ? s0 + p.seg_len : T;
        int flo, fhi;
        adj_seg_frames(s0, s1, T, p.F, hop, flo, fhi);
        for (int i = tid; i < s1 - s0; i += blockDim.x) acc[i] = make_float2(0.f, 0.f);
        const float2* z = reinterpret_cast<const float2*>(p.iq) + n * T;
        const float* gn = p.gout + n * (long long)NFFT * p.F;
        for (int f0 = flo; f0 <= fhi; f0 += BWD_WARPS) {
            const int nf = fhi - f0 + 1 < BWD_WARPS ? fhi - f0 + 1 : BWD_WARPS;
            if (warp < nf) {
                const int f = f0 + warp;
                const int fstart = f * hop - h;
                c2 v[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int nidx = lane + 32 * q;
                    v[q] = pscale(__ldg(z + bwd_reflect(fstart + nidx, T)), hann[nidx]);
                }
                bwd_fft256(v, xch, tw1, tw2, lane);
                // log-magnitude + fftshift backward: G = g X / (|X| (|X| + 1e-6)); park conj(G) by bin
                const float* g = gn + f;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int kbin = bwd_bin(lane, j);
                    const int row = (kbin + NFFT / 2) & (NFFT - 1);
                    const float a = sqrtf(v[j].x * v[j].x + v[j].y * v[j].y);
                    const float s = a > 0.f ? __ldg(g + (size_t)row * p.F) / (a * (a + 1e-6f)) : 0.f;
                    tr[kbin] = make_float2(s * v[j].x, -s * v[j].y);
                }
                __syncwarp();
#pragma unroll
                for (int q = 0; q < 8; ++q) v[q] = tr[lane + 32 * q];
                bwd_fft256(v, xch, tw1, tw2, lane);
#pragma unroll
                for (int j = 0; j < 8; ++j) {                        // the frame's contribution at padded position f hop + nidx
                    const int nidx = bwd_bin(lane, j);
                    const float w = hann[nidx];
                    tr[nidx] = make_float2(w * v[j].x, -w * v[j].y);
                }
            }
            __syncthreads();
            // the samples this round reaches: direct t = u - 128 for u in [ulo, uhi], and the mirrors
            const int ulo = f0 * hop, uhi = (f0 + nf - 1) * hop + NFFT - 1;
            int tlo = ulo - h, thi = uhi - h;
            if (ulo < h) thi = thi > h - ulo ? thi : h - ulo;
            if (uhi >= T + h) { const int m = 2 * (T - 1) + h - (uhi < T + NFFT - 1 ? uhi : T + NFFT - 1); tlo = tlo < m ? tlo : m; }
            tlo = tlo > s0 ? tlo : s0;
            thi = thi < s1 - 1 ? thi : s1 - 1;
            for (int t = tlo + tid; t <= thi; t += blockDim.x) {
                float2 a = acc[t - s0];
                const bool left = t >= 1 && t <= h, right = t >= T - 1 - h && t <= T - 2;
                for (int w = 0; w < nf; ++w) {
                    const int fb = (f0 + w) * hop;
                    const float2* c = xch_all[w];
                    int j = t + h - fb;
                    if ((unsigned)j < (unsigned)NFFT) { a.x += c[j].x; a.y += c[j].y; }
                    j = h - t - fb;
                    if (left && (unsigned)j < (unsigned)NFFT) { a.x += c[j].x; a.y += c[j].y; }
                    j = h + 2 * (T - 1) - t - fb;
                    if (right && (unsigned)j < (unsigned)NFFT) { a.x += c[j].x; a.y += c[j].y; }
                }
                acc[t - s0] = a;
            }
            __syncthreads();
        }
        float2* gz = reinterpret_cast<float2*>(p.gz) + n * T;
        for (int i = tid; i < s1 - s0; i += blockDim.x) gz[s0 + i] = acc[i];
    }
}

// exact float32 range and phase of a joint, as the forward computes them (SURVEY Appendix A)
__device__ __forceinline__ void bwd_range_phase(float jx, float jy, float jz, bool fma_range, float lam, float lam_rcp,
                                                float& d, float& th) {
    const float d2 = fma_range ? __fmaf_rn(jz, jz, __fmaf_rn(jy, jy, __fmul_rn(jx, jx)))
                               : __fadd_rn(__fadd_rn(__fmul_rn(jx, jx), __fmul_rn(jy, jy)), __fmul_rn(jz, jz));
    d = sqrt_rn_fast(d2);
    th = div_rn_fast(__fmul_rn(12.566370614359172f, d), lam, lam_rcp);
}

// The adjoint of one (sequence, time step, body): mean bone length, then per bone the forward geometry (range and phase
// with the forward's exact float32 rounding, the rest in float64) and the analytic derivatives of
// z = sum amp * exp(j theta), accumulated in float64.  `pos(v, m, c)` is coordinate c of joint v of body m at this step:
// read from x, or evaluated from the up-sampling spline -- equal positions and equal (gI, gQ) give equal results.
// gx0 (optional): this step's x-plane row of dL/dx.
template <class Pos>
__device__ __forceinline__ void synth_adjoint_body(const BwdParams& p, const Pos& pos, int m, double gI, double gQ,
                                                   float lam, float lam_rcp, float Lx, float Ly, float Lz,
                                                   double& g_lam, double& g_lx, double& g_ly, double& g_lz,
                                                   float* gx0, long long ps) {
    const double PI = 3.14159265358979323846;
    // mean bone length (:110-113), float32 like the forward
    float sumB = 0.f;
    for (int e = 0; e < p.E; ++e) {
        const int si = p.src[e], di = p.dst[e];
        const float bx = __fsub_rn(pos(di, m, 0), pos(si, m, 0)), by = __fsub_rn(pos(di, m, 1), pos(si, m, 1)),
                    bz = __fsub_rn(pos(di, m, 2), pos(si, m, 2));
        const float bb = p.fma_range ? __fmaf_rn(bz, bz, __fmaf_rn(by, by, __fmul_rn(bx, bx)))
                                     : __fadd_rn(__fadd_rn(__fmul_rn(bx, bx), __fmul_rn(by, by)), __fmul_rn(bz, bz));
        sumB = __fadd_rn(sumB, sqrt_rn_fast(bb));
    }
    if (sumB == 0.f) return;                                           // absent body: contributes exactly 0
    const double cbar = (double)__fmul_rn(sumB, p.inv_E);
    const double c = cbar * cbar, K = sqrt(PI) * cbar;
    double G_c = 0.0;                                                  // dL/d(mean bone length), over this body's bones
    for (int e = 0; e < p.E; ++e) {
        const int si = p.src[e], di = p.dst[e];
        const float sx = pos(si, m, 0), sy = pos(si, m, 1), sz = pos(si, m, 2);
        const float dx = pos(di, m, 0), dy = pos(di, m, 1), dz = pos(di, m, 2);
        // range, phase: the forward's float32 values
        float rng, th;
        bwd_range_phase(__fsub_rn(sx, Lx), __fsub_rn(sy, Ly), __fsub_rn(sz, Lz), p.fma_range != 0, lam, lam_rcp, rng, th);
        double sn, cs;
        sincos((double)th, &sn, &cs);
        // aspect cosine and amplitude, float64 from the float32 inputs
        const double Bx = (double)dx - sx, By = (double)dy - sy, Bz = (double)dz - sz;
        const double Ax = (double)Lx - 0.5 * ((double)sx + dx), Ay = (double)Ly - 0.5 * ((double)sy + dy),
                     Az = (double)Lz - 0.5 * ((double)sz + dz);
        const double na = sqrt(Ax * Ax + Ay * Ay + Az * Az), nb = sqrt(Bx * Bx + By * By + Bz * Bz);
        const double dot = Ax * Bx + Ay * By + Az * Bz;
        const double q = na * nb + 1e-6;
        const double u = dot / q;
        const double den = 1.0 + (c - 1.0) * u * u;
        const double amp = K / den;
        const double dL_dth = amp * (gQ * cs - gI * sn);
        const double dL_damp = gI * cs + gQ * sn;
        g_lam += dL_dth * (-(double)th / (double)lam);
        double gsx = 0.0, gsy = 0.0, gsz = 0.0, gdx = 0.0, gdy = 0.0, gdz = 0.0;   // dL/dS, dL/dD of this bone
        if (rng > 0.f) {
            const double kth = dL_dth * (4.0 * PI / (double)lam) / (double)rng;
            g_lx += kth * ((double)Lx - sx); g_ly += kth * ((double)Ly - sy); g_lz += kth * ((double)Lz - sz);
            gsx = kth * ((double)sx - Lx); gsy = kth * ((double)sy - Ly); gsz = kth * ((double)sz - Lz);
        }
        const double kamp = dL_damp * (-K * 2.0 * u * (c - 1.0) / (den * den));
        if (na > 0.0) {
            const double r2 = dot * nb / (na * q * q);
            const double ax = kamp * (Bx / q - r2 * Ax), ay = kamp * (By / q - r2 * Ay), az = kamp * (Bz / q - r2 * Az);   // dL/dA
            g_lx += ax; g_ly += ay; g_lz += az;
            gsx -= 0.5 * ax; gsy -= 0.5 * ay; gsz -= 0.5 * az;
            gdx -= 0.5 * ax; gdy -= 0.5 * ay; gdz -= 0.5 * az;
        }
        if (gx0) {
            if (nb > 0.0) {
                const double r3 = dot * na / (nb * q * q);
                const double bx = kamp * (Ax / q - r3 * Bx), by = kamp * (Ay / q - r3 * By), bz = kamp * (Az / q - r3 * Bz);  // dL/dB via u
                gsx -= bx; gsy -= by; gsz -= bz;
                gdx += bx; gdy += by; gdz += bz;
            }
            G_c += dL_damp * sqrt(PI) * (1.0 / den - 2.0 * c * u * u / (den * den));
            float* gs = gx0 + si * p.M + m;
            float* gd = gx0 + di * p.M + m;
            gs[0] += (float)gsx; gs[ps] += (float)gsy; gs[2 * ps] += (float)gsz;
            gd[0] += (float)gdx; gd[ps] += (float)gdy; gd[2 * ps] += (float)gdz;
        }
    }
    if (gx0) {                                                         // through the mean bone length (:110-113)
        for (int e = 0; e < p.E; ++e) {
            const int si = p.src[e], di = p.dst[e];
            const double Bx = (double)pos(di, m, 0) - pos(si, m, 0), By = (double)pos(di, m, 1) - pos(si, m, 1),
                         Bz = (double)pos(di, m, 2) - pos(si, m, 2);
            const double nb = sqrt(Bx * Bx + By * By + Bz * Bz);
            if (nb > 0.0) {
                const double kc = G_c * (double)p.inv_E / nb;
                float* gs = gx0 + si * p.M + m;
                float* gd = gx0 + di * p.M + m;
                gs[0] -= (float)(kc * Bx); gs[ps] -= (float)(kc * By); gs[2 * ps] -= (float)(kc * Bz);
                gd[0] += (float)(kc * Bx); gd[ps] += (float)(kc * By); gd[2 * ps] += (float)(kc * Bz);
            }
        }
    }
}

// The parameter gradients' partial sums: PARAM_SLOTS slots of static memory, handed out round-robin per launch by the host
// (like the forward's ticket pool), so that launches in flight on different streams do not share one.  A slot holds 4
// partials per block and a counter of finished blocks.  Budget: PARAM_MAX_BLOCKS * 4 doubles per slot (80 KB),
// PARAM_SLOTS slots (2.5 MB); the host caps the grid at PARAM_MAX_BLOCKS.
constexpr int PARAM_SLOTS = 32;
constexpr int PARAM_MAX_BLOCKS = 2560;
__device__ double g_param_partials[PARAM_SLOTS][PARAM_MAX_BLOCKS * 4];
__device__ unsigned g_param_count[PARAM_SLOTS];

// sum over the block's 128 threads in a fixed order: warp shuffles, then the four warps' sums in pairs
__device__ __forceinline__ void block_sum4(double (&vals)[4], double (&red)[4][4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        double v = vals[i];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) red[i][threadIdx.x >> 5] = v;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) vals[i] = (red[i][0] + red[i][1]) + (red[i][2] + red[i][3]);
    __syncthreads();
}

// Block reduction of the four parameter gradients into the block's partials; the last block to finish adds the partials in
// block order, adds the total to gparams and re-arms the counter.  No float atomics: the result depends only on the
// inputs and the grid, and the grid only on (N, T, sm_count).  128 threads per block.
__device__ __forceinline__ void synth_adjoint_reduce(const BwdParams& p, double g_lam, double g_lx, double g_ly, double g_lz) {
    __shared__ double red[4][4];
    __shared__ bool last;
    double vals[4] = {g_lam, g_lx, g_ly, g_lz};
    block_sum4(vals, red);
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (threadIdx.x == i) p.part[blockIdx.x * 4 + i] = vals[i];
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(p.count, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[i] += __ldcg(p.part + b * 4 + i);
    }
    block_sum4(acc, red);
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (threadIdx.x == i) p.gparams[i] += acc[i];
    if (threadIdx.x == 0) *p.count = 0u;
}

// The adjoint of time step t of output n, joint positions read from x sequence xn (and dL/dx added to its row when p.gx is
// set); xn = n but with VR_FLAG_VIEWS.
__device__ __forceinline__ void synth_adjoint_step(const BwdParams& p, long long n, long long xn, int t, float lam, float lam_rcp,
                                                   float Lx, float Ly, float Lz,
                                                   double& g_lam, double& g_lx, double& g_ly, double& g_lz) {
    const int T = (int)p.T;
    const long long idx = n * T + t;
    const double gI = (double)__ldg(p.gz + idx * 2), gQ = (double)__ldg(p.gz + idx * 2 + 1);
    if (gI == 0.0 && gQ == 0.0) return;
    const float* x0 = p.x + (xn * 3 * T + t) * (long long)p.VM;      // x-plane row of this time step
    const long long ps = (long long)T * p.VM;                         // floats between coordinate planes
    const int M = p.M;
    auto pos = [&](int v, int m, int c) { return __ldg(x0 + v * M + m + c * ps); };
    float* gx0 = p.gx ? p.gx + (xn * 3 * T + t) * (long long)p.VM : nullptr;  // this thread's own rows of dL/dx
    for (int m = 0; m < p.M; ++m)
        synth_adjoint_body(p, pos, m, gI, gQ, lam, lam_rcp, Lx, Ly, Lz, g_lam, g_lx, g_ly, g_lz, gx0, ps);
}

// The same at up-sampled step i of output n (T = ups_K * ups_T): the joint positions come from the per-interval cubics of
// raw sequence xn (pf_locate + pf_eval on p.coef), bit-identical to what vr_pad_frames_f32 writes.  Parameter gradients only.
__device__ __forceinline__ void synth_adjoint_ups_step(const BwdParams& p, long long n, long long xn, long long i, float lam,
                                                       float lam_rcp,
                                                       float Lx, float Ly, float Lz,
                                                       double& g_lam, double& g_lx, double& g_ly, double& g_lz) {
    const long long idx = n * p.T + i;
    const double gI = (double)__ldg(p.gz + idx * 2), gQ = (double)__ldg(p.gz + idx * 2 + 1);
    if (gI == 0.0 && gQ == 0.0) return;
    const int C3 = 3 * p.VM;
    int j;
    double tt;
    pf_locate(i, p.ups_ratio, p.ups_T, j, tt);
    const double* cf = p.coef + ((size_t)xn * (p.ups_T - 1) + j) * 4 * C3;  // a0..a3 of interval j, C3 apart
    const int M = p.M, VM = p.VM;
    auto pos = [&](int v, int m, int c) {
        const double* a = cf + c * VM + v * M + m;
        return pf_eval(tt, __ldg(a), __ldg(a + C3), __ldg(a + 2 * C3), __ldg(a + 3 * C3));
    };
    for (int m = 0; m < p.M; ++m)
        synth_adjoint_body(p, pos, m, gI, gQ, lam, lam_rcp, Lx, Ly, Lz, g_lam, g_lx, g_ly, g_lz, nullptr, 0);
}

__global__ void __launch_bounds__(128) vr_synth_adjoint_kernel(const __grid_constant__ BwdParams p) {
    const int T = (int)p.T;
    const long long total = p.N * (long long)T;
    const float lam = __ldg(p.lam_ptr);
    const float Lx = __ldg(p.loc_ptr), Ly = __ldg(p.loc_ptr + 1), Lz = __ldg(p.loc_ptr + 2);
    const float lam_rcp = rcp_refined(lam);
    double g_lam = 0.0, g_lx = 0.0, g_ly = 0.0, g_lz = 0.0;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long n = idx / T;
        synth_adjoint_step(p, n, n, (int)(idx - n * T), lam, lam_rcp, Lx, Ly, Lz, g_lam, g_lx, g_ly, g_lz);
    }
    synth_adjoint_reduce(p, g_lam, g_lx, g_ly, g_lz);
}

// The same adjoint at the up-sampled steps of vr_forward_upsampled_f32.  (Staging the positions of a block's steps in shared
// memory first was measured slower on a B200: 54.7 vs 38.6 ms per fwd+bwd step at N = 256, k = 250 -- occupancy drops to
// two blocks per SM.)
__global__ void __launch_bounds__(128) vr_synth_adjoint_ups_kernel(const __grid_constant__ BwdParams p) {
    const long long KT = p.T;
    const long long total = p.N * KT;
    const float lam = __ldg(p.lam_ptr);
    const float Lx = __ldg(p.loc_ptr), Ly = __ldg(p.loc_ptr + 1), Lz = __ldg(p.loc_ptr + 2);
    const float lam_rcp = rcp_refined(lam);
    double g_lam = 0.0, g_lx = 0.0, g_ly = 0.0, g_lz = 0.0;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long n = idx / KT;
        synth_adjoint_ups_step(p, n, n, idx - n * KT, lam, lam_rcp, Lx, Ly, Lz, g_lam, g_lx, g_ly, g_lz);
    }
    synth_adjoint_reduce(p, g_lam, g_lx, g_ly, g_lz);
}

// ---- per-sequence parameter gradients (VR_FLAG_PER_SEQUENCE) ----------------------------------------------------------
// Output n reads placement n.  Its steps are cut into PS_SEG-step segments; one warp at a time owns an (x sequence,
// segment) unit, lane k runs the per-step adjoint above for step k of the segment, the warp adds the four gradients with a
// fixed butterfly of shuffles and lane 0 stores the unit's 4 partials (p.part, the scratch tail of the caller's gradient
// buffer).  vr_param_fold_kernel then adds each output's partials in segment order into gparams[4 n ..].  The cut depends
// on T alone and every sum runs in a fixed order, so an output's gradients are the same bits wherever it sits in the
// batch, whatever the batch size, grid or SM count.  No atomics, no counters.  (A block of 128 threads per 256-step
// segment, reduced with block_sum4, measured 1.19x the scalar path's forward + backward step at T = 300, N = 256 and 4096,
// on a B200, against 1.01-1.02x for a warp per 32 steps: 300 = 256 + 44 steps, and the second segment leaves 84 of the 128
// threads idle, where a warp per 32 steps idles at most 31 lanes per sequence; profiles/r03d_rejected_variants.md.)
// VIEWS (VR_FLAG_VIEWS(R), R = p.views > 1 views per x sequence) selects how the views are spread:
//   VIEWS_ROWS (dL/dx wanted): the unit is (x sequence xn, segment) and its warp runs the R views r = 0 .. R-1 in order, each
//     with output xn R + r's dL/d(iq) row and placement on the positions of x sequence xn.  Lane k owns the dL/dx row of
//     (xn, step k) and adds the views' contributions to it in view order: one owner per row, no atomics.
//   VIEWS_OUTPUTS (parameter gradients only): the unit is (output n, segment), as without views, reading x sequence n / R;
//     R times the units of VIEWS_ROWS, and no serial view loop.
// Either way each view's partials go where the repeated batch's unit of that output would put them, so the parameter
// gradients are its bits.  VIEWS_NONE is the plain per-sequence kernel, operation for operation (the same SASS as before
// views existed): the view loop keeps its index and placement live and costs registers (128 / 48 against 122 / 40
// without UPS), which R = 1 has no use for.
constexpr int VIEWS_NONE = 0, VIEWS_OUTPUTS = 1, VIEWS_ROWS = 2;
template <bool UPS, int VIEWS>
__global__ void __launch_bounds__(128) vr_synth_adjoint_ps_kernel(const __grid_constant__ BwdParams p) {
    const int lane = threadIdx.x & 31;
    const int R = VIEWS == VIEWS_ROWS ? p.views : 1;
    const long long segs = p.ps_segs, units = (VIEWS == VIEWS_ROWS ? p.N / R : p.N) * segs;
    const long long wstride = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long u = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); u < units; u += wstride) {
        const long long un = u / segs;                   // VIEWS_ROWS: the x sequence; otherwise the output
        const long long s = u - un * segs;
        const long long t = s * PS_SEG + lane;
        for (int r = 0; r < R; ++r) {
            const long long n = VIEWS == VIEWS_ROWS ? un * R + r : un;
            const long long xn = VIEWS == VIEWS_OUTPUTS ? n / p.views : un;
            const float lam = __ldg(p.lam_ptr + n);
            const float Lx = __ldg(p.loc_ptr + 3 * n), Ly = __ldg(p.loc_ptr + 3 * n + 1), Lz = __ldg(p.loc_ptr + 3 * n + 2);
            const float lam_rcp = rcp_refined(lam);
            double g[4] = {0.0, 0.0, 0.0, 0.0};
            if (t < p.T) {
                if (UPS) synth_adjoint_ups_step(p, n, xn, t, lam, lam_rcp, Lx, Ly, Lz, g[0], g[1], g[2], g[3]);
                else synth_adjoint_step(p, n, xn, (int)t, lam, lam_rcp, Lx, Ly, Lz, g[0], g[1], g[2], g[3]);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
                for (int o = 16; o > 0; o >>= 1) g[i] += __shfl_xor_sync(0xffffffffu, g[i], o);
            if (lane == 0) {
                double* q = p.part + (VIEWS == VIEWS_ROWS ? n * segs + s : u) * 4;
                q[0] = g[0]; q[1] = g[1]; q[2] = g[2]; q[3] = g[3];
            }
        }
    }
}

// gparams[i] += the segment partials of sequence i / 4, component i % 4, added in segment order
__global__ void __launch_bounds__(128) vr_param_fold_kernel(const double* __restrict__ part, double* __restrict__ gparams,
                                                            long long N, long long segs) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 4 * N) return;
    const double* q = part + (i >> 2) * segs * 4 + (i & 3);
    double a = 0.0;
    for (long long s = 0; s < segs; ++s) a += q[s * 4];
    gparams[i] += a;
}
#endif  // __CUDACC__

}  // namespace vr
