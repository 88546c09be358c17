// vr_stft_gemm.cuh -- the STFT against GENERAL (trained / trainable) kernels, on the 5th-generation tensor cores.
//
// Reference: `train_stft_kernel=True` (layers/virtual_radar.py:42,75) makes nnAudio's Fourier kernels `stft.wsin`,
// `stft.wcos` (n_fft x 1 x n_fft each) parameters; the forward is then two conv1d per signal against whatever those
// tensors hold (layers/virtual_radar.py:124-129; nnAudio STFT.forward, SURVEY Appendix B), so no FFT applies.  Written as
// one real GEMM per batch:
//
//     C[m, :] = A[m, :] . Bt^T,   m = (sequence, frame),  A[m] = [ I frame (n_fft) | Q frame (n_fft) ]   (K = 2 n_fft)
//     Bt rows: re_bin = [ wcos[bin] |  wsin[bin] ],  im_bin = [ -wsin[bin] | wcos[bin] ]                   (N = 2 n_fft)
//
// so that Re X = conv(I, wcos) + conv(Q, wsin), Im X = conv(Q, wcos) - conv(I, wsin) -- the combination of
// layers/virtual_radar.py:126-129 with nnAudio's imag = -conv(., wsin) -- come out of the same accumulator row.
//
// Kernel (`vr_gemm_tf32x3_kernel`): tcgen05.mma kind::tf32, M = 128 x N = 128 x K = 8 per instruction, accumulators in
// tensor memory, issued by one thread; operands in shared memory in the K-major 128-byte-swizzled layout, three
// stages, handed over on mbarriers (full: the warps' arrivals + the bulk copy's bytes; free: tcgen05.commit).  A -- the
// frames, read as views of the padded signal, never materialised -- is staged by the CTA's 1024 threads (global ->
// registers -> TF32 split -> shared); B -- the kernel matrix -- is split and tiled once per call and bulk-copied.
// float32 accuracy from 10-bit TF32 mantissas by the error-compensated split a = hi + lo (hi = a rounded to TF32,
// nearest / ties away, lo = a - hi, exact): A.B = Ahi.Bhi + Alo.Bhi + Ahi.Blo -- three MMAs per K step; the dropped lo.lo term is
// 2^-22 relative.  The tensor core ACCUMULATES with truncation, one truncation per instruction: with all 3 x K/8 = 192
// instructions adding into one accumulator the first version was biased by ~4e-6 relative (measured, profiles/r02h).
// Hence FOUR accumulators in the 512 tensor-memory columns: the hi.hi products rotate over three of them (21
// truncations each) and the two small cross terms, 2^-11 of the result, go to the fourth, where truncation is
// harmless; the epilogue adds the four in float32.  Epilogue from tensor memory (tcgen05.ld 32x32b, one row per thread):
// either a plain store, or |X| -> ln(|X| + 1e-6) -> fftshift roll (layers/virtual_radar.py:131-133) written straight
// into the (N, n_fft, F) output, optionally saving Re/Im for the backward pass.
// The same kernel does the backward GEMMs (operands are addressed through element strides, the frame view or the tiled
// image, so transposes cost nothing): dA = dC . Bt (gradient of the frames) and dBt = dC^T . A (gradient of the kernels).
// The kernel gradient's reduction runs over every frame of the batch and is split over gridDim.z; each slice stores its
// partial dBt with plain stores into its own K x K plane of a static pool, and vr_stft_dw_kernel adds the planes in slice
// order: no float atomics, no CTA waiting on another, the same bits on every run.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace vr {

// A/B switches of the operand loads (tools/ab.py build + tools/ab_stft.py, profiles/r02z7_ab_stft.log): PTX-predicated
// loads pay for the frame-column view (backward 1.271 -> 1.119 ms at 4096 sequences) and cost the strided loader
// (forward 0.474 -> 0.529 ms), so each loader keeps the form that measured faster.
#ifndef VR_GEMM_ASM_STRIDED
#define VR_GEMM_ASM_STRIDED 0
#endif
#ifndef VR_GEMM_ASM_COLS
#define VR_GEMM_ASM_COLS 1
#endif
constexpr int GM = 128, GN = 128, GK = 32;          // CTA tile, K block per stage
constexpr int G_THREADS = 1024;                     // every thread stages one 16-byte chunk of A and one of B per K block;
constexpr int G_WARPS = G_THREADS / 32;             // warp w reads accumulator lanes 32 (w % 4) and the (w / 4)-th part of
constexpr int G_PARTS = G_THREADS / 128;            // the columns in the epilogue
constexpr int G_ACC = 4;                            // accumulators in tensor memory (G_ACC * GN = 512 columns)
constexpr int G_STAGES = 3;
#ifndef VR_GEMM_AHEAD
#define VR_GEMM_AHEAD 2
#endif
constexpr int G_AHEAD = VR_GEMM_AHEAD;               // K blocks whose global loads are in flight in registers
constexpr int G_STAGE_BYTES = 2 * (GM + GN) * GK * 4;    // hi + lo of the A and B blocks: 64 KB
constexpr int G_SMEM_BYTES = G_STAGES * G_STAGE_BYTES + 1024;
static_assert(GM * (GK / 4) == G_THREADS && GN * (GK / 4) == G_THREADS, "one chunk of each operand per thread");
static_assert(GK * 4 == 128, "a K block is one 128-byte swizzle line per row");
static_assert(GK / 8 >= G_ACC - 1, "every K block touches all accumulators");

struct GemmParams {
    const float* A; long long sAm, sAk;             // A(m, k) = A[m * sAm + k * sAk]
    const float* B; long long sBn, sBk;             // B(n, k) = B[n * sBn + k * sBk]    (C = A . B^T)
    int M, N, K;
    int kb_per_split;                               // K blocks per gridDim.z slice
    float* C; long long ldc;                        // EPI 0: C[z * c_split + m * ldc + n], z = blockIdx.z (one plane per slice)
    long long c_split;
    float* out; float* csave;                       // EPI 1: (sequences, n_fft, F) log-magnitude; optional raw C, column-major (N x ldc)
    int F, n_fft, nb;                               // frames per sequence; bins per column tile (re block | im block)
    // the frame matrix as a VIEW of the padded signal (operand modes 1 and 2): frame row m = (sequence s, frame f),
    // column k = (component c = k / n_fft, sample j = k % n_fft)  ->  P[(s * 2 + c) * Lp + f * hop + j]
    const float* P; long long Lp; int hop;
    // operand mode G_TILED (B only): B already split into hi / lo and laid out as the shared-memory image of every
    // (column tile, K block): img[(tile_n * KB_all + kb) * G_BIMG_FLOATS ...] = [hi 16 KB | lo 16 KB], swizzled
    const float* Bimg;
};
enum { G_STRIDED = 0, G_FRAME_ROWS = 1, G_FRAME_COLS = 2, G_TILED = 3 };
constexpr int G_BIMG_FLOATS = 2 * GN * GK;          // floats per (column tile, K block) image

#ifdef __CUDACC__
__device__ __forceinline__ uint64_t umma_desc_kmajor_sw128(uint32_t saddr) {
    // cute::UMMA::SmemDescriptor: start address [0,14), leading byte offset [16,30), stride byte offset [32,46) (all >> 4),
    // version [46,48) = 1 on Blackwell, layout type [61,64) = 2 (SWIZZLE_128B).  K-major, 128-byte swizzle: a row is one
    // 128-byte line whose 16-byte chunks are XOR-ed with (row % 8) -- the hardware applies it to address bits [4,7) ^
    // [7,10), so the block must be 1024-byte aligned; SBO = 1024 = distance between 8-row groups; LBO is not used (the
    // K = 8 of one instruction lies inside the line); a K step advances the start address by 32 bytes.
    return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"((uint32_t)__cvta_generic_to_shared(bar)) : "memory");
}
// tensor memory -> registers, 32 lanes x W columns (W = 8 or 16); the caller waits once for all its loads
template <int W>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, float (&v)[W]);
template <>
__device__ __forceinline__ void tmem_ld<16>(uint32_t taddr, float (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]),
                   "=f"(v[8]), "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
                 : "r"(taddr) : "memory");
}
template <>
__device__ __forceinline__ void tmem_ld<8>(uint32_t taddr, float (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// one row's W columns summed over the four accumulators: the four loads are in flight together
template <int W>
__device__ __forceinline__ void tmem_ld_sum(uint32_t taddr, float (&v)[W]) {
    float a1[W], a2[W], a3[W];
    tmem_ld<W>(taddr, v);
    tmem_ld<W>(taddr + GN, a1);
    tmem_ld<W>(taddr + 2 * GN, a2);
    tmem_ld<W>(taddr + 3 * GN, a3);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < W; ++i) v[i] = ((v[i] + a1[i]) + a2[i]) + a3[i];
}
__device__ __forceinline__ void g_mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void g_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"((uint32_t)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ void g_mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
    } while (!ok);
}

// a = hi + lo with hi = a rounded to TF32 (10-bit mantissa), nearest with ties away from zero -- what cvt.rna.tf32.f32
// gives for every finite a that does not round up to infinity -- and lo = a - hi, exact.  Two integer instructions (the
// cvt is emulated with four on this target).  Ties away keeps the lo parts sign-symmetric.
__device__ __forceinline__ void tf32_split(float a, float& hi, float& lo) {
    hi = __uint_as_float((__float_as_uint(a) + 0x1000u) & 0xffffe000u);
    lo = a - hi;
}

// float index of element (n, k) of B inside the tiled image, for the hi part (the lo part is GN * GK floats further)
__host__ __device__ inline long long g_bimg_index(int n, int k, int KB_all) {
    const int tile_n = n / GN, r = n % GN, kb = k / GK, kk = k % GK, kc = kk >> 2;
    return ((long long)tile_n * KB_all + kb) * G_BIMG_FLOATS + r * (GK) + ((kc ^ (r & 7)) << 2) + (kk & 3);
}
// which 16-byte chunk (row r, K chunk kc) of a block thread c moves.  Shared memory holds a block K-major in the 128-byte
// swizzle the tensor core reads natively (UMMA layout type SWIZZLE_128B): row r is one 128-byte line (GK = 32 floats), its
// chunk kc at r * 128 + ((kc ^ (r % 8)) * 16); eight-row groups are 1024 bytes apart.
//  - K contiguous in memory (row-major operand): a quarter warp = the 8 chunks of one row: one whole 128-byte line from
//    global memory (a 16-byte load is processed a quarter warp at a time: the earlier layouts -- 32 rows x 1 chunk, then
//    8 rows x 4 chunks per warp -- cost 32 data-pipe wavefronts per load instruction either way, and the L1 data pipe
//    at 67-81 % of its peak bounded the loop, ncu profiles/r02t, r02w), and one whole line of shared memory, conflict-free.
//  - rows contiguous in memory (the transposed operands of the backward GEMMs): a warp = 32 rows x 1 chunk: its four
//    scalar loads are one line each, and the swizzle spreads a quarter warp's eight rows over all banks.
// (The first version had consecutive threads on consecutive chunks of a row in the unswizzled layout: 87 % of its
// shared-memory wavefronts were bank conflicts, ncu profiles/r02h.)
template <int ROWS>
__device__ __forceinline__ void g_chunk(int c, bool k_contig, int& r, int& kc) {
    if (k_contig) {
        r = c >> 3;
        kc = c & 7;
    } else {
        r = c % ROWS;
        kc = c / ROWS;
    }
}
// one thread's view of an operand: where its chunk of the next K block is, set up once per CTA.
//   G_STRIDED     X(row, k) = src[row * s_row + k * s_k]
//   G_FRAME_ROWS  X(m, k)   = frame m, column k of the padded signal (the forward's A): nothing is materialised, the 16-fold
//                 overlap of the frames is read from L2 instead of being written to and read back from HBM
//   G_FRAME_COLS  X(k, m)   = the same matrix transposed (B of the kernel-gradient GEMM: its K index runs over the frames)
// Predicated loads, written as PTX so that the value has ONE definition: with `v = 0; if (ok) v = load` the compiler may copy
// the loaded registers into the merged variable right behind the load, i.e. wait for it there -- in the kernel-gradient
// GEMM the loads meant to be in flight over two K blocks were not (22 % of the stall samples sat on those copies, ncu
// profiles/r02z4).  Used where it measured faster (see VR_GEMM_ASM_*).
__device__ __forceinline__ float4 ldg_v4_if(const float* q, bool ok) {
    float4 v;
    asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %5, 0;\n mov.f32 %0, 0f00000000;\n mov.f32 %1, 0f00000000;\n mov.f32 %2, 0f00000000;\n"
                 " mov.f32 %3, 0f00000000;\n @p ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];\n}"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(q), "r"((int)ok));
    return v;
}
__device__ __forceinline__ void ldg_into_if(float& v, const float* q, bool ok) {      // v keeps its value when !ok
    asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %2, 0;\n @p ld.global.nc.f32 %0, [%1];\n}" : "+f"(v) : "l"(q), "r"((int)ok));
}
__device__ __forceinline__ void tf32_store_split(unsigned char* hi, unsigned char* lo, uint32_t off, const float4 v) {
    float4 h, l;
    tf32_split(v.x, h.x, l.x);
    tf32_split(v.y, h.y, l.y);
    tf32_split(v.z, h.z, l.z);
    tf32_split(v.w, h.w, l.w);
    *reinterpret_cast<float4*>(hi + off) = h;
    *reinterpret_cast<float4*>(lo + off) = l;
}
template <int MODE>
struct GLoader;
template <>
struct GLoader<G_STRIDED> {
    const float* p;                                   // element (row, k) of the next block's chunk
    long long s_k, step;                              // element stride along K; advance per K block
    int k;                                            // its K index (bounds only matter in a ragged last block)
    uint32_t off;                                     // byte offset of the chunk inside a staged block
    bool row_ok, vec;                                 // row inside the matrix; one aligned 16-byte load per chunk
    template <int ROWS>
    __device__ __forceinline__ void init(const GemmParams&, const float* src, long long s_row, long long sk, int row0, int nrows, int k0, int tid) {
        int r, kc;
        g_chunk<ROWS>(tid, sk == 1, r, kc);
        const int row = row0 + r;
        row_ok = row < nrows;
        k = k0 + 4 * kc;
        s_k = sk;
        step = (long long)GK * sk;
        p = src + (long long)(row_ok ? row : 0) * s_row + (long long)k * sk;
        vec = sk == 1 && (reinterpret_cast<uintptr_t>(p) & 15) == 0;       // a K block is 128 bytes: alignment holds for all
        off = (uint32_t)(r * 128 + ((kc ^ (r & 7)) << 4));
    }
    __device__ __forceinline__ float4 load(const GemmParams&, int K) {
#if VR_GEMM_ASM_STRIDED
        const bool whole = row_ok && vec && k + 3 < K, parts = row_ok && !whole;
        float4 v = ldg_v4_if(p, whole);
        ldg_into_if(v.x, p, parts && k < K);
        ldg_into_if(v.y, p + s_k, parts && k + 1 < K);
        ldg_into_if(v.z, p + 2 * s_k, parts && k + 2 < K);
        ldg_into_if(v.w, p + 3 * s_k, parts && k + 3 < K);
#else
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row_ok) {
            if (vec && k + 3 < K) v = __ldg(reinterpret_cast<const float4*>(p));
            else {
                if (k < K) v.x = __ldg(p);
                if (k + 1 < K) v.y = __ldg(p + s_k);
                if (k + 2 < K) v.z = __ldg(p + 2 * s_k);
                if (k + 3 < K) v.w = __ldg(p + 3 * s_k);
            }
        }
#endif
        p += step;
        k += GK;
        return v;
    }
};
template <>
struct GLoader<G_FRAME_ROWS> {
    const float* base;                                // P + s * 2 Lp + f * hop: sample 0 of the I frame
    int k;
    uint32_t off;
    bool row_ok, vec;
    template <int ROWS>
    __device__ __forceinline__ void init(const GemmParams& g, const float*, long long, long long, int row0, int nrows, int k0, int tid) {
        int r, kc;
        g_chunk<ROWS>(tid, true, r, kc);
        const int row = row0 + r;
        row_ok = row < nrows;
        k = k0 + 4 * kc;
        const int m = row_ok ? row : 0, sq = m / g.F, f = m - sq * g.F;
        base = g.P + (long long)sq * 2 * g.Lp + (long long)f * g.hop;
        vec = (g.hop & 3) == 0 && (g.Lp & 3) == 0 && (reinterpret_cast<uintptr_t>(g.P) & 15) == 0;      // k, n_fft are multiples of 4
        off = (uint32_t)(r * 128 + ((kc ^ (r & 7)) << 4));
    }
    __device__ __forceinline__ float4 load(const GemmParams& g, int K) {                // K = 2 n_fft, a multiple of 4
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);                                    // (plain loads: the PTX form was slower here, r02z5)
        if (row_ok && k < K) {
            const float* q = base + (k >= g.n_fft ? g.Lp - g.n_fft : 0ll) + k;           // the Q frame lives in the next plane
            if (vec) v = __ldg(reinterpret_cast<const float4*>(q));
            else v = make_float4(__ldg(q), __ldg(q + 1), __ldg(q + 2), __ldg(q + 3));
        }
        k += GK;
        return v;
    }
};
template <>
struct GLoader<G_FRAME_COLS> {
    const float* q;                                   // this row's sample in frame m
    int m, f;                                         // frame index of the chunk's first element, and its frame number in its sequence
    uint32_t off;
    bool row_ok;
    template <int ROWS>
    __device__ __forceinline__ void init(const GemmParams& g, const float*, long long, long long, int row0, int nrows, int k0, int tid) {
        int r, kc;
        g_chunk<ROWS>(tid, false, r, kc);
        const int row = row0 + r;
        row_ok = row < nrows;
        const int col = row_ok ? row : 0, c = col >= g.n_fft ? 1 : 0;
        m = k0 + 4 * kc;
        const int sq = m / g.F;
        f = m - sq * g.F;
        q = g.P + (long long)c * g.Lp + (col - c * g.n_fft) + (long long)sq * 2 * g.Lp + (long long)f * g.hop;
        off = (uint32_t)(r * 128 + ((kc ^ (r & 7)) << 4));
    }
    // the next frame is hop samples further, or -- after a sequence's last frame -- at the start of the next sequence's
    // planes: a running pointer, no division and no 64-bit multiply per element
    __device__ __forceinline__ float4 load(const GemmParams& g, int K) {                // K = number of frames
        const long long wrap = 2 * g.Lp - (long long)g.F * g.hop;                       // uniform: next sequence's frame 0 - (frame F)
        float e[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#if VR_GEMM_ASM_COLS
            ldg_into_if(e[j], q, row_ok && m + j < K);
#else
            if (row_ok && m + j < K) e[j] = __ldg(q);
#endif
            q += g.hop;
            if (++f == g.F) { f = 0; q += wrap; }
        }
        constexpr int REST = GK - 4;                  // to the chunk of the next K block: REST = (REST / F) F + REST % F frames
        m += GK;
        f += REST % g.F;
        q += (long long)(REST / g.F) * 2 * g.Lp + (long long)(REST % g.F) * g.hop;
        if (f >= g.F) { f -= g.F; q += wrap; }
        return make_float4(e[0], e[1], e[2], e[3]);
    }
};

// Pipeline.  No CTA-wide barrier inside the K loop (the first versions had one per K block, and the slowest of the 32
// warps' global loads paced every block: 27 % of the stall samples at the barrier, 16 % at the loads, ncu profiles/r02w):
//   every warp:  wait free[s] (the MMAs that read stage s are complete) -> split its chunks of block kb into stage s ->
//                issue the loads of block kb + G_AHEAD into registers -> fence.proxy.async -> lane 0 arrives on full[s]
//   B of the forward and of the frame-gradient GEMM (the kernel matrix) is not staged by the warps at all: it is split and
//   tiled once per call (vr_stft_bt_kernel) and one thread bulk-copies the 32 KB image of a block (cp.async.bulk ->
//   complete_tx on full[s]) as soon as the stage is free.
//   warp 0 then: lane 0 waits full[s] (all 32 warps have arrived), issues the block's 12 MMAs and commits them to free[s].
// Warps other than 0 run up to G_STAGES blocks ahead of the tensor core.
template <int EPI, int AMODE, int BMODE>
__global__ void __launch_bounds__(G_THREADS, 1) vr_gemm_tf32x3_kernel(const __grid_constant__ GemmParams p) {
    extern __shared__ __align__(1024) unsigned char gsm[];
    __shared__ uint64_t bar_full[G_STAGES], bar_free[G_STAGES], bar_done;
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ntn = (p.N + GN - 1) / GN;                         // column tiles fastest: the CTAs that share an A tile run together
    const int tile_n = blockIdx.x % ntn, tile_m = blockIdx.x / ntn;    // (A once from HBM; it was read once per column tile, ncu r02s)
    const int m0 = tile_m * GM, n0 = tile_n * GN;

    if (tid == 0) {
        for (int i = 0; i < G_STAGES; ++i) {
            g_mbar_init(&bar_full[i], G_WARPS + (BMODE == G_TILED ? 1 : 0));     // + the bulk copy's expect_tx arrival
            g_mbar_init(&bar_free[i], 1);
        }
        g_mbar_init(&bar_done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {                                              // one warp allocates (and later frees) the accumulators' 512 columns
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"((uint32_t)__cvta_generic_to_shared(&tmem_base_s)), "r"((uint32_t)(G_ACC * GN)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // this thread's chunks, and the first two blocks' loads, before the set-up barrier
    const int KB_all = (p.K + GK - 1) / GK;
    const int kb_first = blockIdx.z * p.kb_per_split;
    const int KB = (KB_all - kb_first < p.kb_per_split) ? (KB_all - kb_first) : p.kb_per_split;     // this slice's K blocks (>= 1)
    constexpr bool B_TILED = BMODE == G_TILED;                    // B arrives by bulk copy: no registers, no split, no stores
    GLoader<AMODE> la;
    GLoader<B_TILED ? G_STRIDED : BMODE> lb;
    la.template init<GM>(p, p.A, p.sAm, p.sAk, m0, p.M, kb_first * GK, tid);
    // register prefetch: G_AHEAD K blocks in flight (one fragment per stage; the loop is unrolled over the stages)
    float4 fa0 = la.load(p, p.K), fb0 = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 fa1 = fb0, fb1 = fb0, fa2 = fb0, fb2 = fb0;
    if (KB > 1) fa1 = la.load(p, p.K);
    if (KB > 2 && G_AHEAD > 2) fa2 = la.load(p, p.K);
    if (!B_TILED) {
        lb.template init<GN>(p, p.B, p.sBn, p.sBk, n0, p.N, kb_first * GK, tid);
        fb0 = lb.load(p, p.K);
        if (KB > 1) fb1 = lb.load(p, p.K);
        if (KB > 2 && G_AHEAD > 2) fb2 = lb.load(p, p.K);
    }
    const float* bimg = B_TILED ? p.Bimg + ((long long)tile_n * KB_all + kb_first) * G_BIMG_FLOATS : nullptr;

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;

    // instruction descriptor (cute::UMMA::InstrDescriptor): D = F32 [4,6), A = B = TF32 [7,10) [10,13), both K-major,
    // N >> 3 at [17,23), M >> 4 at [24,29)
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(GN >> 3) << 17) | ((uint32_t)(GM >> 4) << 24);
    uint32_t use = 0;                                             // how often the stages have been used before
    auto k_block = [&](const int kb, const int s, float4& ra, float4& rb) {
        unsigned char* st = gsm + s * G_STAGE_BYTES;
        unsigned char* a_hi = st, *a_lo = st + GM * GK * 4, *b_hi = st + 2 * GM * GK * 4, *b_lo = b_hi + GN * GK * 4;
        if (use > 0) g_mbar_wait(&bar_free[s], (use - 1) & 1);    // the MMAs that read this stage have completed
        if (B_TILED) {
            if (tid == 32) {                                      // one thread of warp 1 (warp 0 issues the MMAs): 32 KB, hi | lo
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                             ::"r"((uint32_t)__cvta_generic_to_shared(&bar_full[s])), "r"((uint32_t)(G_BIMG_FLOATS * 4)) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"((uint32_t)__cvta_generic_to_shared(b_hi)), "l"(bimg + (long long)kb * G_BIMG_FLOATS),
                               "r"((uint32_t)(G_BIMG_FLOATS * 4)), "r"((uint32_t)__cvta_generic_to_shared(&bar_full[s])) : "memory");
            }
            tf32_store_split(a_hi, a_lo, la.off, ra);
            if (kb + G_AHEAD < KB) ra = la.load(p, p.K);
        } else {
            tf32_store_split(a_hi, a_lo, la.off, ra);
            tf32_store_split(b_hi, b_lo, lb.off, rb);
            if (kb + G_AHEAD < KB) { ra = la.load(p, p.K); rb = lb.load(p, p.K); }
        }       // the block after next: in flight over two blocks
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> visible to the tensor core's reads
        __syncwarp();
        if (lane == 0) g_mbar_arrive(&bar_full[s]);
        if (warp == 0) {
            if (lane == 0) {
                g_mbar_wait(&bar_full[s], use & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t ah = (uint32_t)__cvta_generic_to_shared(a_hi), al = (uint32_t)__cvta_generic_to_shared(a_lo);
                const uint32_t bh = (uint32_t)__cvta_generic_to_shared(b_hi), bl = (uint32_t)__cvta_generic_to_shared(b_lo);
#pragma unroll
                for (int ks = 0; ks < GK / 8; ++ks) {             // K = 8 per instruction = 32 bytes of every row
                    const uint64_t dah = umma_desc_kmajor_sw128(ah + ks * 32), dal = umma_desc_kmajor_sw128(al + ks * 32);
                    const uint64_t dbh = umma_desc_kmajor_sw128(bh + ks * 32), dbl = umma_desc_kmajor_sw128(bl + ks * 32);
                    const int step = kb * (GK / 8) + ks, big = step % (G_ACC - 1);
                    umma_tf32(tmem + big * GN, dah, dbh, idesc, step >= G_ACC - 1 ? 1u : 0u);   // hi.hi: rotate over three accumulators
                    umma_tf32(tmem + (G_ACC - 1) * GN, dal, dbh, idesc, step > 0 ? 1u : 0u);    // the small cross terms: the fourth
                    umma_tf32(tmem + (G_ACC - 1) * GN, dah, dbl, idesc, 1u);
                }
                umma_commit(&bar_free[s]);                        // arrives when the MMAs issued so far have read shared memory
                if (kb == KB - 1) umma_commit(&bar_done);
            }
            __syncwarp();
        }
    };
    static_assert(G_STAGES == 3 && (G_AHEAD == 3 || G_AHEAD == 2), "the loop below is written out for three stages");
    if (G_AHEAD == 3) {
        for (int kb = 0; kb < KB; kb += 3, ++use) {               // fragment i <-> stage i
            k_block(kb, 0, fa0, fb0);
            if (kb + 1 < KB) k_block(kb + 1, 1, fa1, fb1);
            if (kb + 2 < KB) k_block(kb + 2, 2, fa2, fb2);
        }
    } else {
        for (int kb = 0; kb < KB; kb += 6, ++use) {               // two fragments, three stages: period six
            k_block(kb, 0, fa0, fb0);
            if (kb + 1 < KB) k_block(kb + 1, 1, fa1, fb1);
            if (kb + 2 < KB) k_block(kb + 2, 2, fa0, fb0);
            ++use;
            if (kb + 3 < KB) k_block(kb + 3, 0, fa1, fb1);
            if (kb + 4 < KB) k_block(kb + 4, 1, fa0, fb0);
            if (kb + 5 < KB) k_block(kb + 5, 2, fa1, fb1);
        }
    }
    if (KB > 0) g_mbar_wait(&bar_done, 0u);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- epilogue: thread = accumulator row (TMEM lane 32 * (warp % 4) + lane); the warps of each group of four take one
    // part of the columns (bins) ----
    const int m = m0 + (tid & 127);
    const int part = warp >> 2;
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    if (EPI == 0) {
        // the tile goes through shared memory (the stages are free: bar_done covers every MMA) so that global memory sees
        // whole rows: a thread owns one ROW of the accumulator, and its direct stores were 32 lines per instruction
        constexpr int W = GN / G_PARTS;                           // 16 columns per thread
        constexpr int LDT = GN + 4;                               // padded row: a quarter warp's 16-byte stores hit all banks
        static_assert(GM * LDT * 4 <= G_STAGES * G_STAGE_BYTES, "tile fits the stages");
        float* tile = reinterpret_cast<float*>(gsm);
        if (KB > 0) {
            float v[W];
            tmem_ld_sum<W>(trow + part * W, v);
#pragma unroll
            for (int j = 0; j < W; j += 4)
                *reinterpret_cast<float4*>(tile + (tid & 127) * LDT + part * W + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
        __syncthreads();
        float* const C = p.C + blockIdx.z * p.c_split;
        const bool vec = (p.ldc & 3) == 0 && (p.c_split & 3) == 0 && (reinterpret_cast<uintptr_t>(p.C) & 15) == 0;
        if (KB > 0) {
            for (int i = tid; i < GM * (GN / 4); i += G_THREADS) {
                const int r = i / (GN / 4), c = (i % (GN / 4)) * 4;
                const int gm = m0 + r, gn = n0 + c;
                if (gm >= p.M || gn >= p.N) continue;
                const float4 v = *reinterpret_cast<const float4*>(tile + r * LDT + c);
                float* dst = C + (long long)gm * p.ldc + gn;
                if (vec && gn + 3 < p.N) *reinterpret_cast<float4*>(dst) = v;
                else {
                    const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (gn + j < p.N) dst[j] = e[j];
                }
            }
        }
    } else {
        // column tile: [re of bins t*nb .. | im of the same bins]; out[(seq * n_fft + ((bin + n_fft/2) % n_fft)) * F + f]
        constexpr int W = 8;
        const int nb = p.nb;                                      // a power of two >= 16
        const int parts = nb / W < G_PARTS ? nb / W : G_PARTS;
        const int per = nb / parts;                               // bins per part: a multiple of 8
        const int seq = m / p.F, f = m - seq * p.F;
        if (part < parts) {
            for (int c0 = part * per; c0 < (part + 1) * per; c0 += W) {
                float re[W], im[W];
                tmem_ld_sum<W>(trow + c0, re);
                tmem_ld_sum<W>(trow + nb + c0, im);
                if (m < p.M) {
                    float* o = p.out + (long long)seq * p.n_fft * p.F + f;
#pragma unroll
                    for (int j = 0; j < W; ++j) {
                        const int bin = tile_n * nb + c0 + j;
                        if (bin < p.n_fft) {
                            const float mag = sqrtf(fmaf(re[j], re[j], im[j] * im[j]));
                            int row = bin + (p.n_fft >> 1);
                            row = row >= p.n_fft ? row - p.n_fft : row;
                            o[(long long)row * p.F] = logf(mag + 1e-6f);
                            if (p.csave) {
                                p.csave[(long long)(n0 + c0 + j) * p.ldc + m] = re[j];          // column-major: lanes = rows, coalesced
                                p.csave[(long long)(n0 + nb + c0 + j) * p.ldc + m] = im[j];
                            }
                        }
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)(G_ACC * GN)) : "memory");
}

// ---- small kernels around the GEMM -------------------------------------------------------------------------------
// nnAudio center=True, pad_mode='reflect': padded position j (0 <= j < T + n_fft) holds sample stft_reflect(j)
__device__ __forceinline__ int stft_reflect(int j, int T, int n_fft) {
    int t = j - n_fft / 2;
    t = t < 0 ? -t : t;
    return t >= T ? 2 * (T - 1) - t : t;
}
// the padded, planar signal the frame views read: iq (S, T, 2) -> P (S, 2, Lp), P[s][c][j] = iq[s][reflect(j - n_fft/2)][c]
// for j < T + n_fft (nnAudio center=True, pad_mode='reflect'), 0 beyond.  Frame f of sequence s is P[s][c][f * hop ...].
__global__ void vr_stft_pad_kernel(const float* __restrict__ iq, float* __restrict__ P, long long S, int T, long long Lp, int n_fft) {
    const long long total = S * Lp;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long sq = i / Lp;
        const int j = (int)(i - sq * Lp);
        float2 z = make_float2(0.f, 0.f);
        if (j < T + n_fft) z = __ldg(reinterpret_cast<const float2*>(iq) + sq * T + stft_reflect(j, T, n_fft));
        P[sq * 2 * Lp + j] = z.x;
        P[(sq * 2 + 1) * Lp + j] = z.y;
    }
}
// kept frames only: the frames listed in `frames` (Fk strictly increasing indices, the same for every sequence) copied end to
// end into a compact planar buffer, P'[(s * 2 + c) * Fk n_fft + i n_fft + j] = padded[s][c][frames[i] hop + j], so that the
// GEMMs read it as a frame view with hop' = n_fft and F' = Fk.
__global__ void vr_stft_gather_kernel(const float* __restrict__ iq, const int* __restrict__ frames, float* __restrict__ P,
                                      long long S, int T, int Fk, int n_fft, int hop) {
    const long long Lp = (long long)Fk * n_fft, total = S * Lp;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long sq = i / Lp;
        const int r = (int)(i - sq * Lp), fi = r / n_fft, j = r - fi * n_fft;
        const int t = stft_reflect(__ldg(frames + fi) * hop + j, T, n_fft);
        const float2 z = __ldg(reinterpret_cast<const float2*>(iq) + sq * T + t);
        P[sq * 2 * Lp + r] = z.x;
        P[(sq * 2 + 1) * Lp + r] = z.y;
    }
}
// row of Bt that holds Re / Im of `bin` under the column-tile layout [re block | im block] of nb bins
__host__ __device__ inline int stft_row_re(int bin, int nb) { return (bin / nb) * 2 * nb + bin % nb; }
__host__ __device__ inline int stft_row_im(int bin, int nb) { return (bin / nb) * 2 * nb + nb + bin % nb; }
// Bt (2 n_fft, 2 n_fft) from stft.wsin / stft.wcos (n_fft, 1, n_fft), never stored as a matrix: written split into TF32
// hi / lo parts as the tiled shared-memory images the GEMMs bulk-copy -- `fwd` for C = A . Bt^T (B(n, k) = Bt[n][k]) and
// `bwd` for dA = dC . Bt (B'(k, n) = Bt[n][k]).  K = 2 n_fft; rows beyond K of a 128-row tile stay zero (the host clears).
__device__ __forceinline__ void stft_bimg_put(float* fwd, float* bwd, int n, int k, float v, int KB_all) {
    float hi, lo;
    tf32_split(v, hi, lo);
    const long long f = g_bimg_index(n, k, KB_all), t = g_bimg_index(k, n, KB_all);
    fwd[f] = hi; fwd[f + GN * GK] = lo;
    bwd[t] = hi; bwd[t + GN * GK] = lo;
}
__global__ void vr_stft_bt_kernel(const float* __restrict__ wsin, const float* __restrict__ wcos, float* __restrict__ fwd,
                                  float* __restrict__ bwd, int n_fft, int nb, int KB_all) {
    const int total = n_fft * n_fft;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int bin = i / n_fft, s = i - bin * n_fft;
        const float c = __ldg(wcos + i), sn = __ldg(wsin + i);
        const int re = stft_row_re(bin, nb), im = stft_row_im(bin, nb);
        stft_bimg_put(fwd, bwd, re, s, c, KB_all);
        stft_bimg_put(fwd, bwd, re, n_fft + s, sn, KB_all);
        stft_bimg_put(fwd, bwd, im, s, -sn, KB_all);
        stft_bimg_put(fwd, bwd, im, n_fft + s, c, KB_all);
    }
}
// backward of ln(|X| + 1e-6) and the roll: dC from grad_out and the saved Re / Im.  C and dC are column-major (2 n_fft
// columns of ldm floats, ldm a multiple of 4): blockIdx.y = bin, a thread takes four consecutive rows of its Re and Im
// columns as 16-byte accesses.
__global__ void vr_stft_dc_kernel(const float* __restrict__ gout, const float* __restrict__ csave, float* __restrict__ dC,
                                  int M, long long ldm, int F, int n_fft, int nb) {
    const int bin = blockIdx.y;
    const int cr = stft_row_re(bin, nb), ci = stft_row_im(bin, nb);
    const int row = (bin + n_fft / 2) % n_fft;
    const float4* re4 = reinterpret_cast<const float4*>(csave + cr * ldm);
    const float4* im4 = reinterpret_cast<const float4*>(csave + ci * ldm);
    float4* dre4 = reinterpret_cast<float4*>(dC + cr * ldm);
    float4* dim4 = reinterpret_cast<float4*>(dC + ci * ldm);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; 4 * i < M; i += gridDim.x * blockDim.x) {
        const float4 r4 = re4[i], i4 = im4[i];                    // rows >= M of the last group are padding: zero gradient
        const float re[4] = {r4.x, r4.y, r4.z, r4.w}, im[4] = {i4.x, i4.y, i4.z, i4.w};
        float dr[4], di[4];
        int seq = (4 * i) / F, f = 4 * i - seq * F;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            dr[j] = 0.f;
            di[j] = 0.f;
            if (4 * i + j < M) {
                const float g = __ldg(gout + ((long long)seq * n_fft + row) * F + f);
                const float mag = sqrtf(fmaf(re[j], re[j], im[j] * im[j]));
                const float w = mag > 0.f ? g / ((mag + 1e-6f) * mag) : 0.f;
                dr[j] = w * re[j];
                di[j] = w * im[j];
            }
            if (++f == F) { f = 0; ++seq; }
        }
        dre4[i] = make_float4(dr[0], dr[1], dr[2], dr[3]);
        dim4[i] = make_float4(di[0], di[1], di[2], di[3]);
    }
}
// overlap-add of the frame gradients through the reflect padding: dA (S*F, 2 n_fft) -> grad_iq (S, T, 2).  Gather form, one
// thread per output sample and component: padded position u receives dA[frame f][u - f hop] from every frame that covers
// it, and sample t is the image of u = t + n_fft/2 and of its mirror positions in the two reflected margins.  No atomics,
// no zero fill; consecutive threads read consecutive columns of the same frame rows.
__device__ __forceinline__ float stft_fold_at(const float* __restrict__ dA, long long seq, int c, int u, int F, int n_fft, int hop) {
    // frames f with f hop <= u < f hop + n_fft
    int f1 = u / hop;
    f1 = f1 < F - 1 ? f1 : F - 1;
    int f0 = u - n_fft + 1 <= 0 ? 0 : (u - n_fft + hop) / hop;
    float acc = 0.f;
    for (int f = f0; f <= f1; ++f) acc += __ldg(dA + ((seq * F + f) * 2 + c) * (long long)n_fft + (u - f * hop));
    return acc;
}
__global__ void vr_stft_fold_kernel(const float* __restrict__ dA, float* __restrict__ giq, long long S, int T, int F, int n_fft, int hop) {
    const long long total = S * T;
    const int h = n_fft / 2, U = T + n_fft;                        // padded length
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long seq = i / T;
        const int t = (int)(i - seq * T);
        float2 g = make_float2(0.f, 0.f);
#pragma unroll
        for (int side = 0; side < 3; ++side) {
            // padded positions that hold sample t: the direct one, the left mirror (u = h - t, 1 <= t <= h) and the right
            // mirror (u = h + 2 (T - 1) - t, T - 1 - h <= t <= T - 2)
            const int u = side == 0 ? t + h : (side == 1 ? h - t : h + 2 * (T - 1) - t);
            const bool on = side == 0 || (side == 1 ? (t >= 1 && t <= h) : (t <= T - 2 && t >= T - 1 - h));
            if (on && u >= 0 && u < U) {
                g.x += stft_fold_at(dA, seq, 0, u, F, n_fft, hop);
                g.y += stft_fold_at(dA, seq, 1, u, F, n_fft, hop);
            }
        }
        reinterpret_cast<float2*>(giq)[i] = g;
    }
}
// the same fold when dA holds only the kept frames (dA (S*Fk, 2 n_fft), row i = frame frames[i]): the kept frames covering
// position u are a contiguous run of the sorted table, found by binary search; summed in increasing frame order like
// stft_fold_at, so the result equals the full fold fed zero gradients for the frames that were not kept.  A sample that no
// kept frame covers gets 0.
__device__ __forceinline__ float stft_fold_kept_at(const float* __restrict__ dA, const int* __restrict__ frames, long long seq,
                                                   int c, int u, int Fk, int n_fft, int hop) {
    const int fmin = u - n_fft + 1 <= 0 ? 0 : (u - n_fft + hop) / hop;      // frames f with f hop <= u < f hop + n_fft
    int a = 0, b = Fk;                                                      // first table entry >= fmin
    while (a < b) {
        const int mid = (a + b) >> 1;
        if (__ldg(frames + mid) < fmin) a = mid + 1; else b = mid;
    }
    float acc = 0.f;
    for (int i = a; i < Fk; ++i) {
        const int f = __ldg(frames + i);
        if (f * hop > u) break;
        acc += __ldg(dA + ((seq * Fk + i) * 2 + c) * (long long)n_fft + (u - f * hop));
    }
    return acc;
}
__global__ void vr_stft_fold_kept_kernel(const float* __restrict__ dA, const int* __restrict__ frames, float* __restrict__ giq,
                                         long long S, int T, int Fk, int n_fft, int hop) {
    const long long total = S * T;
    const int h = n_fft / 2, U = T + n_fft;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long seq = i / T;
        const int t = (int)(i - seq * T);
        float2 g = make_float2(0.f, 0.f);
#pragma unroll
        for (int side = 0; side < 3; ++side) {          // the direct position and the two mirrors, as vr_stft_fold_kernel
            const int u = side == 0 ? t + h : (side == 1 ? h - t : h + 2 * (T - 1) - t);
            const bool on = side == 0 || (side == 1 ? (t >= 1 && t <= h) : (t <= T - 2 && t >= T - 1 - h));
            if (on && u >= 0 && u < U) {
                g.x += stft_fold_kept_at(dA, frames, seq, 0, u, Fk, n_fft, hop);
                g.y += stft_fold_kept_at(dA, frames, seq, 1, u, Fk, n_fft, hop);
            }
        }
        reinterpret_cast<float2*>(giq)[i] = g;
    }
}
// The split-K partials of the kernel gradient: at most G_SPLIT_PLANES_MAX tiles' worth of K x K planes per launch (the host
// caps splits * tiles, which one wave already bounds by the SM count), G_SPLIT_SLOTS slots handed out round-robin per launch
// so that launches in flight on other streams do not share one.  10 MB per slot, 40 MB in all.
constexpr int G_SPLIT_CTAS_MAX = 160;
constexpr int G_SPLIT_SLOTS = 4;
constexpr long long G_SPLIT_SLOT_FLOATS = (long long)G_SPLIT_CTAS_MAX * GM * GN;
__device__ float g_splitk_pool[G_SPLIT_SLOTS * G_SPLIT_SLOT_FLOATS];

// dBt (2 n_fft, 2 n_fft), as `splits` partial planes `stride` floats apart added in slice order -> grad wsin / wcos
__device__ __forceinline__ float stft_split_sum(const float* __restrict__ q, int splits, long long stride) {
    float v = __ldg(q);
    for (int z = 1; z < splits; ++z) v += __ldg(q + z * stride);
    return v;
}
__global__ void vr_stft_dw_kernel(const float* __restrict__ dBt, int splits, long long stride, float* __restrict__ gsin,
                                  float* __restrict__ gcos, int n_fft, int nb) {
    const int total = n_fft * n_fft;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int bin = i / n_fft, s = i - bin * n_fft;
        const float* re = dBt + (long long)stft_row_re(bin, nb) * 2 * n_fft;
        const float* im = dBt + (long long)stft_row_im(bin, nb) * 2 * n_fft;
        gcos[i] = stft_split_sum(re + s, splits, stride) + stft_split_sum(im + n_fft + s, splits, stride);
        gsin[i] = stft_split_sum(re + n_fft + s, splits, stride) - stft_split_sum(im + s, splits, stride);
    }
}
#endif  // __CUDACC__

}  // namespace vr
