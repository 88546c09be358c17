// vr_pad_frames.cuh -- temporal up-sampling of joint trajectories to the radar sampling rate
// (SURVEY 8 row a13; reference utils.py:134-140 `Dataset.pad_frames` followed by the FloatTensor cast of
// `Dataset.__getitem__`, utils.py:128-132):
//
//   smooth = scipy.ndimage.gaussian_filter1d(x, sigma, axis=time)      float32 in -> float64 accumulate -> float32 out
//   spline = scipy.interpolate.interp1d(linspace(0,1,T), smooth, 'cubic', axis=time)   not-a-knot cubic, float64
//   out    = float32(spline(linspace(0,1,k*T)))
//
// One CTA owns the trajectories of `nc` adjacent (joint, body) columns of one (sequence, coordinate)
// plane.  It (1) smooths them with the reflect-padded Gaussian in FP64, accumulating in scipy's order
// (centre tap, then symmetric pairs from the outermost inwards) and rounding to float32 exactly where
// scipy does; (2) solves the not-a-knot cubic spline for its second derivatives, one thread per
// trajectory (the end conditions reduce the system to tridiagonal: 6 M1 = rhs1, 6 M(T-2) = rhs(T-2));
// (3) evaluates the k*T output frames in FP64 from shared memory and writes float32 rows, coalesced.
// The intermediate float64 arrays never leave shared memory.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace vr {

constexpr int PF_MAX_RADIUS = 40;

struct PadParams {
    const float* x;              // (N,3,T,V,M)
    float* out;                  // (N,3,k*T,V,M), or nullptr when only the spline is wanted (coef below)
    double* coef;                // optional (N, T-1, 4, 3*V*M): the cubic a0..a3 of every input interval and column,
                                 // consumed by the fused up-sampling + radar kernel (vr_forward_upsampled_f32)
    long long planes;            // N*3
    int T, VM, K, nc, ncb;       // frames in, columns per plane, up-sampling factor, columns per CTA, column blocks per plane
    int radius;
    double ratio;                // (T-1)/(K*T-1): input-sample position of output frame i is i*ratio
    double w[PF_MAX_RADIUS + 1]; // Gaussian weights, w[0] = centre
};

#ifdef __CUDACC__
// The cubic of input interval [j, j+1] in the local variable tt = s - j (unit sample spacing), from the
// smoothed samples y and the spline's second derivatives m.  One definition for every kernel that
// evaluates the spline: value(tt) = fma(tt, fma(tt, fma(tt, a3, a2), a1), a0), rounded to float32.
__device__ __forceinline__ void pf_cubic(double y0, double y1, double m0, double m1,
                                         double& a0, double& a1, double& a2, double& a3) {
    a0 = y0;
    a1 = (y1 - y0) - (2.0 * m0 + m1) * (1.0 / 6.0);
    a2 = 0.5 * m0;
    a3 = (m1 - m0) * (1.0 / 6.0);
}
__device__ __forceinline__ float pf_eval(double tt, double a0, double a1, double a2, double a3) {
    return (float)fma(tt, fma(tt, fma(tt, a3, a2), a1), a0);
}
// position of output frame i on the input grid: interval j and offset tt inside it
__device__ __forceinline__ void pf_locate(long long i, double ratio, int T, int& j, double& tt) {
    const double s = (double)i * ratio;
    j = (int)s;
    j = j > T - 2 ? T - 2 : j;
    tt = s - (double)j;
}

__device__ __forceinline__ int pf_reflect(int t, int T) {     // scipy 'reflect': d c b a | a b c d | d c b a
    while (t < 0 || t >= T) t = t < 0 ? -t - 1 : 2 * T - t - 1;
    return t;
}

__global__ void __launch_bounds__(1024, 1) vr_pad_frames_kernel(const __grid_constant__ PadParams p) {
    extern __shared__ __align__(16) unsigned char pf_smem[];
    const int T = p.T, nc = p.nc;
    double* Msh = reinterpret_cast<double*>(pf_smem);            // [T][nc] second derivatives (unit sample spacing)
    double* cp = Msh + (size_t)T * nc;                           // [T]     Thomas coefficients (same for every column)
    float* ys = reinterpret_cast<float*>(cp + T);                // [T][nc] smoothed trajectories, float32 like scipy's output
    const int tid = threadIdx.x;
    const long long KT = (long long)p.K * T;

    for (long long unit = blockIdx.x; unit < p.planes * p.ncb; unit += gridDim.x) {
        const long long plane = unit / p.ncb;
        const int col0 = (int)(unit - plane * p.ncb) * nc;
        const int ncl = (p.VM - col0 < nc) ? (p.VM - col0) : nc;     // columns of this block
        const float* xp = p.x + plane * (long long)T * p.VM + col0;
        float* op = p.out + plane * KT * p.VM + col0;
        __syncthreads();                                         // previous unit's evaluation has finished with shared memory

        // (1) Gaussian smoothing along time, float64 accumulate in scipy's order, float32 result
        for (int idx = tid; idx < T * ncl; idx += blockDim.x) {
            const int t = idx / ncl, c = idx - t * ncl;
            double acc = __dmul_rn((double)__ldg(xp + (size_t)t * p.VM + c), p.w[0]);
            for (int jj = p.radius; jj >= 1; --jj) {
                const double a = (double)__ldg(xp + (size_t)pf_reflect(t - jj, T) * p.VM + c);
                const double b = (double)__ldg(xp + (size_t)pf_reflect(t + jj, T) * p.VM + c);
                acc = __dadd_rn(acc, __dmul_rn(__dadd_rn(a, b), p.w[jj]));
            }
            ys[t * nc + c] = (float)acc;
        }
        if (tid == 0) {                                          // c'_i of the Thomas algorithm for rows 2..T-3 (diagonal 4, off-diagonals 1)
            double c = 0.0;
            for (int i = 2; i <= T - 3; ++i) { c = 1.0 / (4.0 - c); cp[i] = c; }
        }
        __syncthreads();

        // (2) not-a-knot cubic spline: second derivatives M_i, one thread per trajectory
        if (tid < ncl) {
            const int c = tid;
            auto rhs = [&](int i) {
                return 6.0 * (((double)ys[(i - 1) * nc + c] - 2.0 * (double)ys[i * nc + c]) + (double)ys[(i + 1) * nc + c]);
            };
            const double M1 = rhs(1) / 6.0, Mn = rhs(T - 2) / 6.0;
            Msh[1 * nc + c] = M1;
            Msh[(T - 2) * nc + c] = Mn;
            double d = 0.0;                                      // forward sweep: d'_i stored in place
            for (int i = 2; i <= T - 3; ++i) {
                double r = rhs(i);
                if (i == 2) r -= M1;
                if (i == T - 3) r -= Mn;
                d = (r - d) * cp[i];
                Msh[i * nc + c] = d;
            }
            double next = 0.0;                                   // back substitution: M_i = d'_i - c'_i M_{i+1}
            for (int i = T - 3; i >= 2; --i) {
                const double m = Msh[i * nc + c] - (i == T - 3 ? 0.0 : cp[i] * next);
                Msh[i * nc + c] = m;
                next = m;
            }
            Msh[0 * nc + c] = 2.0 * Msh[1 * nc + c] - Msh[2 * nc + c];
            Msh[(T - 1) * nc + c] = 2.0 * Msh[(T - 2) * nc + c] - Msh[(T - 3) * nc + c];
        }
        __syncthreads();

        // (2b) spline-only mode: hand the per-interval cubics to the fused radar kernel
        if (p.coef) {
            const int C3 = 3 * p.VM;
            const long long n = plane / 3;
            const int cplane = (int)(plane - n * 3);
            double* cf = p.coef + (size_t)n * (T - 1) * 4 * C3 + cplane * p.VM + col0;
            for (int idx = tid; idx < (T - 1) * ncl; idx += blockDim.x) {
                const int j = idx / ncl, c = idx - j * ncl;
                double a0, a1, a2, a3;
                pf_cubic((double)ys[j * nc + c], (double)ys[(j + 1) * nc + c], Msh[j * nc + c], Msh[(j + 1) * nc + c], a0, a1, a2, a3);
                double* o = cf + (size_t)j * 4 * C3 + c;
                o[0] = a0; o[C3] = a1; o[2 * C3] = a2; o[3 * C3] = a3;
            }
        }

        // (3) evaluate the K*T output frames, float64, and write float32 rows.  The plane's output is one
        // contiguous run when the block holds all columns, so a flat index gives coalesced stores; (row, column)
        // advance incrementally (no divisions) and the cubic of the current input interval is kept in
        // registers while consecutive output frames fall into it (K frames per interval).
        if (p.out) {
            const int rows_per_step = (int)blockDim.x / ncl;     // threads beyond rows_per_step * ncl sit this phase out,
            const int c = tid % ncl;                             // so that every thread stays on one column
            int jc = -1;
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            for (long long i = tid / ncl; i < KT && tid < rows_per_step * ncl; i += rows_per_step) {
                int j;
                double tt;
                pf_locate(i, p.ratio, T, j, tt);
                if (j != jc) {
                    pf_cubic((double)ys[j * nc + c], (double)ys[(j + 1) * nc + c], Msh[j * nc + c], Msh[(j + 1) * nc + c], a0, a1, a2, a3);
                    jc = j;
                }
                op[i * p.VM + c] = pf_eval(tt, a0, a1, a2, a3);
            }
        }
    }
}
#endif  // __CUDACC__

// ------------------------------------------------------------------------------------------------
// Backward pass of vr_pad_frames_kernel: dL/d(out) (N,3,k*T,V,M) -> dL/dx (N,3,T,V,M), both float32.
//
// Definition: the gradient is the transpose of the float64 linear operator the forward evaluates (Gaussian ->
// not-a-knot spline solve -> per-interval cubics -> Horner evaluation at the k*T positions).  The two float32
// roundings of the forward (the smoothed samples ys and the output) pass the gradient through unchanged, as autograd
// treats a dtype cast.  Everything is float64 and rounded to float32 once, at the end; no atomics, so the result is
// bitwise reproducible.  Stages, in reverse order of the forward's:
//   (1) evaluation: ga_q[j] = sum over the output rows i of interval j of tt_i^q g_i, q = 0..3, with the forward's own
//       pf_locate (the last row is clamped into interval T-2 there too).  The rows of an interval are contiguous: one warp,
//       lanes = columns, walks them in order (coalesced, fixed summation order);
//   (2) pf_cubic: (ga0..ga3) of interval j -> gy_j, gy_{j+1}, gM_j, gM_{j+1} (even intervals first, then odd ones: no two
//       intervals of a pass share an end point);
//   (3) the spline solve run backwards, one thread per column: end extrapolations, back substitution, forward sweep, the
//       direct rows M1 = rhs1 / 6 and M(T-2) = rhs(T-2) / 6, and the second differences of the right-hand sides;
//   (4) the reflect-padded Gaussian transposed: dL/dx[s] gathers w[|u - t|] gys[t] over every u that pf_reflect folds
//       onto s (a radius larger than T folds several times, exactly as the forward does).
// Shared memory: 16 bytes per (frame, column).  The Thomas coefficients c'_i reach their float64 fixed point at i = 15;
// the host computes them (the forward's recurrence) into `cp` and the kernel reads c'_i = cp[min(i, PF_CP_N - 1)].
constexpr int PF_CP_N = 32;

struct PadBwdParams {
    const float* g;              // (N,3,k*T,V,M) dL/d(out)
    float* gx;                   // (N,3,T,V,M)   dL/dx, overwritten
    long long planes;            // N*3
    int T, VM, K, nc, ncb;
    int radius;
    double ratio;                // as PadParams::ratio
    double w[PF_MAX_RADIUS + 1];
    double cp[PF_CP_N];          // c'_i of the forward's Thomas sweep, i < PF_CP_N (entries 0, 1 unused)
};

#ifdef __CUDACC__
// first output row of interval j (rows i with pf_locate(i) == j are [pf_first_row(j), pf_first_row(j+1)))
__device__ __forceinline__ long long pf_first_row(int j, double ratio, int T, long long KT) {
    if (j <= 0) return 0;
    if (j > T - 2) return KT;
    long long i = (long long)((double)j / ratio);
    i = i < 2 ? 0 : i - 2;
    int jj;
    double tt;
    for (;; ++i) {                                               // pf_locate is monotone in i: the first row not below j
        pf_locate(i, ratio, T, jj, tt);
        if (jj >= j) break;
    }
    while (i > 0) {
        pf_locate(i - 1, ratio, T, jj, tt);
        if (jj < j) break;
        --i;
    }
    return i;
}

__global__ void __launch_bounds__(1024, 1) vr_pad_frames_backward_kernel(const __grid_constant__ PadBwdParams p) {
    extern __shared__ __align__(16) unsigned char pf_smem[];
    const int T = p.T, nc = p.nc;
    double* Y = reinterpret_cast<double*>(pf_smem);               // [T][nc] dL/dys
    double* G = Y + (size_t)T * nc;                               // [T][nc] dL/dM, then dL/d(rhs), then dL/dx
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const long long KT = (long long)p.K * T;
    auto cp = [&](int i) { return p.cp[i < PF_CP_N ? i : PF_CP_N - 1]; };

    for (long long unit = blockIdx.x; unit < p.planes * p.ncb; unit += gridDim.x) {
        const long long plane = unit / p.ncb;
        const int col0 = (int)(unit - plane * p.ncb) * nc;
        const int ncl = (p.VM - col0 < nc) ? (p.VM - col0) : nc;
        const int ngr = (ncl + 31) >> 5;                          // 32-column groups
        const float* gp = p.g + plane * KT * p.VM + col0;
        __syncthreads();                                          // previous unit's gather has finished with shared memory
        for (int idx = tid; idx < 2 * T * nc; idx += blockDim.x) Y[idx] = 0.0;
        __syncthreads();

        // (1) + (2): interval sums, mapped through pf_cubic; even intervals, then odd ones
        for (int parity = 0; parity < 2; ++parity) {
            const int nint = (T - 1 - parity + 1) / 2;            // intervals j = parity, parity + 2, ... <= T - 2
            for (int task = warp; task < nint * ngr; task += nwarps) {
                const int j = parity + 2 * (task / ngr);
                const int c = (task - (task / ngr) * ngr) * 32 + lane;
                const long long lo = pf_first_row(j, p.ratio, T, KT), hi = pf_first_row(j + 1, p.ratio, T, KT);
                double ga0 = 0.0, ga1 = 0.0, ga2 = 0.0, ga3 = 0.0;
                if (c < ncl) {
                    const float* gc = gp + c;
                    long long i = lo;
                    for (; i + 4 <= hi; i += 4) {                 // four loads in flight ahead of the FP64 chain
                        float v[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) v[u] = __ldg(gc + (i + u) * p.VM);
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            int jj;
                            double tt;
                            pf_locate(i + u, p.ratio, T, jj, tt);
                            const double gv = (double)v[u], t2 = tt * tt;
                            ga0 += gv; ga1 += tt * gv; ga2 += t2 * gv; ga3 += (t2 * tt) * gv;
                        }
                    }
                    for (; i < hi; ++i) {
                        int jj;
                        double tt;
                        pf_locate(i, p.ratio, T, jj, tt);
                        const double gv = (double)__ldg(gc + i * p.VM), t2 = tt * tt;
                        ga0 += gv; ga1 += tt * gv; ga2 += t2 * gv; ga3 += (t2 * tt) * gv;
                    }
                    // a0 = y0, a1 = (y1 - y0) - (2 m0 + m1) / 6, a2 = m0 / 2, a3 = (m1 - m0) / 6
                    Y[j * nc + c] += ga0 - ga1;
                    Y[(j + 1) * nc + c] += ga1;
                    G[j * nc + c] += (0.5 * ga2 - (2.0 / 6.0) * ga1) - (1.0 / 6.0) * ga3;
                    G[(j + 1) * nc + c] += (1.0 / 6.0) * (ga3 - ga1);
                }
            }
            __syncthreads();
        }

        // (3) the not-a-knot solve backwards, one thread per column (in place in G)
        if (tid < ncl) {
            const int c = tid;
            double* g = G + c;
            // M(T-1) = 2 M(T-2) - M(T-3), M0 = 2 M1 - M2 (the forward's last two statements, reversed)
            g[(T - 2) * nc] += 2.0 * g[(T - 1) * nc];
            g[(T - 3) * nc] -= g[(T - 1) * nc];
            g[1 * nc] += 2.0 * g[0];
            g[2 * nc] -= g[0];
            g[0] = 0.0;
            g[(T - 1) * nc] = 0.0;
            // back substitution M_i = d_i - c'_i M_{i+1}, i = T-4 .. 2 (and M(T-3) = d(T-3)): g[i] becomes dL/dd_i
            for (int i = 2; i <= T - 4; ++i) g[(i + 1) * nc] -= cp(i) * g[i * nc];
            // forward sweep d_i = (r_i - d_{i-1}) c'_i, i = 2 .. T-3: g[i] becomes dL/dr_i = dL/d(rhs_i);
            // r_2 -= M1, r(T-3) -= M(T-2)
            for (int i = T - 3; i >= 2; --i) {
                const double gr = g[i * nc] * cp(i);
                g[i * nc] = gr;
                if (i > 2) g[(i - 1) * nc] -= gr;
            }
            if (T >= 5) {
                g[1 * nc] -= g[2 * nc];
                g[(T - 2) * nc] -= g[(T - 3) * nc];
            }
            // M1 = rhs1 / 6, M(T-2) = rhs(T-2) / 6
            g[1 * nc] /= 6.0;
            g[(T - 2) * nc] /= 6.0;
        }
        __syncthreads();
        // rhs_i = 6 ((ys_{i-1} - 2 ys_i) + ys_{i+1}), i = 1 .. T-2 (G[0] = G[T-1] = 0)
        for (int idx = tid; idx < T * ncl; idx += blockDim.x) {
            const int t = idx / ncl, c = idx - t * ncl;
            const double gm = t > 0 ? G[(t - 1) * nc + c] : 0.0, gq = t < T - 1 ? G[(t + 1) * nc + c] : 0.0;
            Y[t * nc + c] += 6.0 * ((gm + gq) - 2.0 * G[t * nc + c]);
        }
        __syncthreads();

        // (4) transposed Gaussian: ys[t] = sum_{|u - t| <= r} w[|u - t|] x[pf_reflect(u)]; dL/dx[s] sums over the u that
        // fold onto s -- they lie in {s + 2Tm} and {2Tm - 1 - s} (the folds map each family onto itself)
        float* gxp = p.gx + plane * (long long)T * p.VM + col0;
        const int r = p.radius, mlim = r / (2 * T) + 1;
        for (int idx = tid; idx < T * ncl; idx += blockDim.x) {
            const int s = idx / ncl, c = idx - s * ncl;
            double acc = 0.0;
            for (int m = -mlim; m <= mlim; ++m) {
                for (int fam = 0; fam < 2; ++fam) {
                    const int u = fam == 0 ? s + 2 * T * m : 2 * T * m - 1 - s;
                    if (u < -r || u > T - 1 + r || pf_reflect(u, T) != s) continue;
                    const int t0 = u - r > 0 ? u - r : 0, t1 = u + r < T - 1 ? u + r : T - 1;
                    for (int t = t0; t <= t1; ++t) acc += p.w[t > u ? t - u : u - t] * Y[t * nc + c];
                }
            }
            gxp[(size_t)s * p.VM + c] = (float)acc;
        }
    }
}
#endif  // __CUDACC__

// ------------------------------------------------------------------------------------------------
// The notebook's variant: `utils.pad_frames` (reference utils.py:82-89), used by virtual_radar_example.ipynb
// cells 2-4 on (T, V, C) arrays of ONE body:
//
//   smooth = scipy.ndimage.gaussian_filter1d(data, sigma, axis=1)     along the JOINT axis (a quirk that is kept,
//                                                                    SURVEY Appendix D); same dtype out as in
//   spline = scipy.interpolate.interp1d(linspace(0,1,T), smooth, 'cubic', axis=-3)     not-a-knot cubic in time, float64
//   out    = spline(linspace(0,1,k*T))                                float64; the notebook then casts with torch.Tensor
//
// x: (N, T, V, C) float64 or float32 (both occur: the mocap files are float64, the NTU example float32).  Output
// float32 -- the cast of torch.Tensor(...) -- in one of two layouts: ROWS (N, k*T, V, C), whose permuted view is exactly
// the notebook's coordinate-innermost tensor, or PLANES (N, C, k*T, V), the layer's own input layout, for the fused
// call that skips the layout copy (the range rounding mode then has to be passed explicitly: VR_FLAG_RANGE_FMA).
// One CTA owns `nc` adjacent (joint, coordinate) columns of one sequence; everything between the Gaussian and the
// evaluation stays in shared memory as float64: 16 bytes per (frame, column) + 8 per frame, i.e. T <= 8500 frames in
// (the reference's three inputs have 300, 2751 and 8192).
struct PadNbParams {
    const void* x;               // (N, T, V, C), TIN
    float* out;
    long long N;
    int T, V, C, K, nc, ncb, planar;
    int nrs;                     // row slices per (sequence, column block): a single long sequence still fills the machine
    long long rows_per_slice;
    int radius;
    double ratio;
    double w[PF_MAX_RADIUS + 1];
};

#ifdef __CUDACC__
template <typename TIN>
__global__ void __launch_bounds__(1024, 1) vr_pad_frames_nb_kernel(const __grid_constant__ PadNbParams p) {
    extern __shared__ __align__(16) unsigned char pf_smem[];
    const int T = p.T, nc = p.nc, VC = p.V * p.C;
    double* Msh = reinterpret_cast<double*>(pf_smem);            // [T][nc] second derivatives
    double* ys = Msh + (size_t)T * nc;                           // [T][nc] smoothed trajectories (rounded to TIN like scipy's output)
    double* cp = ys + (size_t)T * nc;                            // [T]     Thomas coefficients
    const int tid = threadIdx.x;
    const long long KT = (long long)p.K * T;

    for (long long unit = blockIdx.x; unit < p.N * p.ncb * p.nrs; unit += gridDim.x) {
        // unit = (sequence, column block, row slice); the Gaussian and the spline solve are repeated per row slice (the host
        // only slices when they are cheap next to the evaluation: one NTU sequence x550 is 2 column blocks x 165 000 rows)
        const long long nb_unit = unit / p.nrs;
        const int rs = (int)(unit - nb_unit * p.nrs);
        const long long n = nb_unit / p.ncb;
        const int col0 = (int)(nb_unit - n * p.ncb) * nc;
        const int ncl = (VC - col0 < nc) ? (VC - col0) : nc;
        const TIN* xp = static_cast<const TIN*>(p.x) + n * (long long)T * VC;
        const long long row_lo = rs * p.rows_per_slice;
        const long long row_hi = (row_lo + p.rows_per_slice < KT) ? row_lo + p.rows_per_slice : KT;
        __syncthreads();

        // (1) Gaussian along the joints of every frame: scipy's correlate1d order (centre tap, then symmetric pairs
        // from the outermost inwards), float64 accumulation, result rounded to the input dtype
        for (int idx = tid; idx < T * ncl; idx += blockDim.x) {
            const int t = idx / ncl, col = col0 + (idx - t * ncl);
            const int v = col / p.C, c = col - v * p.C;
            const TIN* row = xp + (size_t)t * VC + c;
            double acc = __dmul_rn((double)row[v * p.C], p.w[0]);
            for (int jj = p.radius; jj >= 1; --jj) {
                const double a = (double)row[pf_reflect(v - jj, p.V) * p.C];
                const double b = (double)row[pf_reflect(v + jj, p.V) * p.C];
                acc = __dadd_rn(acc, __dmul_rn(__dadd_rn(a, b), p.w[jj]));
            }
            ys[t * nc + (col - col0)] = (double)(TIN)acc;
        }
        if (tid == 0) {
            double c = 0.0;
            for (int i = 2; i <= T - 3; ++i) { c = 1.0 / (4.0 - c); cp[i] = c; }
        }
        __syncthreads();

        // (2) not-a-knot cubic spline in time (same elimination, same order of operations as vr_pad_frames_kernel).  The
        // right-hand sides do not depend on the recurrence: all threads compute them first (into Msh), so that the one thread
        // per column that runs the two sequential sweeps has a single load per step in front of its DADD -> DMUL chain
        // and the loads of the next steps are already in flight (the mocap files have 2751 / 8192 frames per column).
        for (int idx = tid; idx < (T - 2) * ncl; idx += blockDim.x) {
            const int i = 1 + idx / ncl, c = idx - (i - 1) * ncl;
            Msh[i * nc + c] = 6.0 * ((ys[(i - 1) * nc + c] - 2.0 * ys[i * nc + c]) + ys[(i + 1) * nc + c]);
        }
        __syncthreads();
        if (tid < ncl) {
            const int c = tid;
            const double M1 = Msh[1 * nc + c] / 6.0, Mn = Msh[(T - 2) * nc + c] / 6.0;
            __syncwarp(__activemask());
            Msh[1 * nc + c] = M1;
            Msh[(T - 2) * nc + c] = Mn;
            double d = 0.0;
            int i = 2;
            for (; i + 3 <= T - 4; i += 4) {                      // interior steps, four loads ahead of the chain
                double r0 = Msh[i * nc + c], r1 = Msh[(i + 1) * nc + c], r2 = Msh[(i + 2) * nc + c], r3 = Msh[(i + 3) * nc + c];
                const double c0 = cp[i], c1 = cp[i + 1], c2 = cp[i + 2], c3 = cp[i + 3];
                if (i == 2) r0 -= M1;
                d = (r0 - d) * c0; Msh[i * nc + c] = d;
                d = (r1 - d) * c1; Msh[(i + 1) * nc + c] = d;
                d = (r2 - d) * c2; Msh[(i + 2) * nc + c] = d;
                d = (r3 - d) * c3; Msh[(i + 3) * nc + c] = d;
            }
            for (; i <= T - 3; ++i) {
                double r = Msh[i * nc + c];
                if (i == 2) r -= M1;
                if (i == T - 3) r -= Mn;
                d = (r - d) * cp[i];
                Msh[i * nc + c] = d;
            }
            double next = 0.0;
            i = T - 3;
            if (i >= 2) { next = Msh[i * nc + c]; --i; }           // M_{T-3} = d'_{T-3}
            for (; i - 3 >= 2; i -= 4) {
                const double d0 = Msh[i * nc + c], d1 = Msh[(i - 1) * nc + c], d2 = Msh[(i - 2) * nc + c], d3 = Msh[(i - 3) * nc + c];
                const double c0 = cp[i], c1 = cp[i - 1], c2 = cp[i - 2], c3 = cp[i - 3];
                next = d0 - c0 * next; Msh[i * nc + c] = next;
                next = d1 - c1 * next; Msh[(i - 1) * nc + c] = next;
                next = d2 - c2 * next; Msh[(i - 2) * nc + c] = next;
                next = d3 - c3 * next; Msh[(i - 3) * nc + c] = next;
            }
            for (; i >= 2; --i) {
                next = Msh[i * nc + c] - cp[i] * next;
                Msh[i * nc + c] = next;
            }
            Msh[0 * nc + c] = 2.0 * Msh[1 * nc + c] - Msh[2 * nc + c];
            Msh[(T - 1) * nc + c] = 2.0 * Msh[(T - 2) * nc + c] - Msh[(T - 3) * nc + c];
        }
        __syncthreads();

        // (3) evaluate k*T frames in float64, cast to float32 (torch.Tensor(...) in the notebook)
        const int rows_per_step = (int)blockDim.x / ncl;
        const int cl = tid % ncl, col = col0 + cl;
        const int v = col / p.C, c = col - v * p.C;
        float* op = p.planar ? p.out + ((n * p.C + c) * KT) * p.V + v            // (N, C, k*T, V)
                             : p.out + n * KT * VC + col;                         // (N, k*T, V, C)
        const long long ostride = p.planar ? p.V : VC;
        int jc = -1;
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
        for (long long i = row_lo + tid / ncl; i < row_hi && tid < rows_per_step * ncl; i += rows_per_step) {
            int j;
            double tt;
            pf_locate(i, p.ratio, T, j, tt);
            if (j != jc) {
                pf_cubic(ys[j * nc + cl], ys[(j + 1) * nc + cl], Msh[j * nc + cl], Msh[(j + 1) * nc + cl], a0, a1, a2, a3);
                jc = j;
            }
            op[i * ostride] = pf_eval(tt, a0, a1, a2, a3);
        }
    }
}
#endif  // __CUDACC__

}  // namespace vr
