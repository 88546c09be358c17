// vr_cabi.cu -- C ABI (include/virtual_radar_b200.h) over the fused sm_100a kernel.
// Host logic only: argument checks mirroring the reference's failure modes, bone partitioning,
// launch planning, and the pipelined host-buffer entry point.  No torch, no ATen.
#include "../../include/virtual_radar_b200.h"
#include "vr_kernels.cuh"
#include "vr_pad_frames.cuh"
#include "vr_backward.cuh"
#include "vr_stft_gemm.cuh"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <mutex>
#include <vector>

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t e_ = (expr);                                                                \
        if (e_ != cudaSuccess) return fail(VR_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

struct Tuning { int warps = 0, ctas_per_sm = 0, stages = 0; };
Tuning g_tuning;                                  // vr_set_tuning (benchmark knob)
unsigned long long* g_timeline = nullptr;         // vr_set_timeline_buffer (profiling aid)
// A/B builds for measurements are made with compile-time macros (tools/ab.py builds the variants); the shipped library
// has no environment switches.
#ifdef VR_AB_STATIC_JOBS
constexpr bool g_dynamic = false;                 // round-robin jobs instead of the ticket counter
#else
constexpr bool g_dynamic = true;                  // dynamic job scheduling for batches larger than the grid
#endif
#ifdef VR_AB_NO_PDL
constexpr bool g_pdl = false;
#else
constexpr bool g_pdl = true;                      // programmatic dependent launch
#endif
int g_schedule = -1;                              // vr_set_schedule: -1 automatic, 0 cooperative kernel only, 1 team-job kernel whenever it applies

// ---- bone partition -----------------------------------------------------------------------------
// Bones are grouped by source joint (the range phase of a joint is shared by all bones that start
// there, layers/virtual_radar.py:93,99), and the source joints are spread over the 4 lane groups
// by longest-processing-time-first on an instruction-cost estimate.
struct Partition {
    int group_of_edge[vr::NG * vr::MAX_EG * 4];
    std::vector<int> src_of[vr::NG];                  // source joints per group (sorted by out-degree desc)
    std::vector<std::vector<int>> edges_of[vr::NG];   // per source: list of edge ids
    int ne[vr::NG], ns[vr::NG];
};

int partition_edges(const int32_t* src, const int32_t* dst, int E, int V, Partition& P) {
    if (!src || !dst) return fail(VR_ERR_ARG, "edge arrays must not be null");
    if (E <= 0) return fail(VR_ERR_SHAPE, "need at least one edge, got E=%d", E);
    if (E > vr::NG * vr::MAX_EG) return fail(VR_ERR_UNSUPPORTED, "E=%d exceeds the supported %d bones", E, vr::NG * vr::MAX_EG);
    for (int e = 0; e < E; ++e)
        if (src[e] < 0 || src[e] >= V || dst[e] < 0 || dst[e] >= V)
            return fail(VR_ERR_SHAPE, "edge %d = (%d,%d) indexes a joint outside [0,%d) (IndexError in the reference, layers/virtual_radar.py:93-94)", e, src[e], dst[e], V);
    std::vector<int> joints;                            // distinct sources, first-appearance order
    std::vector<std::vector<int>> out;                  // edges per source
    for (int e = 0; e < E; ++e) {
        size_t i = 0;
        for (; i < joints.size(); ++i) if (joints[i] == src[e]) break;
        if (i == joints.size()) { joints.push_back(src[e]); out.emplace_back(); }
        out[i].push_back(e);
    }
    std::vector<int> order(joints.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = (int)i;
    const int COST_J = 55, COST_E = 61;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return out[a].size() > out[b].size(); });
    long load[vr::NG] = {0, 0, 0, 0};
    for (int g = 0; g < vr::NG; ++g) { P.src_of[g].clear(); P.edges_of[g].clear(); P.ne[g] = P.ns[g] = 0; }
    for (int i : order) {
        int best = 0;
        for (int g = 1; g < vr::NG; ++g) if (load[g] < load[best]) best = g;
        load[best] += COST_J + COST_E * (long)out[i].size();
        P.src_of[best].push_back(joints[i]);
        P.edges_of[best].push_back(out[i]);
        P.ne[best] += (int)out[i].size();
        P.ns[best] += 1;
        for (int e : out[i]) P.group_of_edge[e] = best;
    }
    for (int g = 0; g < vr::NG; ++g)
        if (P.ne[g] > vr::MAX_EG || P.ns[g] > vr::MAX_SG)
            return fail(VR_ERR_UNSUPPORTED, "bone group %d too large (%d bones, %d source joints; max %d/%d)", g, P.ne[g], P.ns[g], vr::MAX_EG, vr::MAX_SG);
    return VR_OK;
}

// ---- launch plan --------------------------------------------------------------------------------
int round_up(int v, int a) { return (v + a - 1) / a * a; }

int make_plan_z(int64_t N, int64_t T, int V, int M, const int32_t* src, const int32_t* dst, int E,
                int n_fft, int hop, int img, bool ups, bool iq_only, int sm_count, bool x_aligned, int ZCAP_MAX, bool park,
                vr::Params& p, int& grid, int& ctas_per_sm) {
    // iq_only: synthesis only; n_fft, hop and img are ignored (no frames, no output tile)
    if (img < 0 || img > 4096) return fail(VR_ERR_SHAPE, "image_size must be in [1, 4096], got %d", img);
    if (N <= 0 || T <= 0 || V <= 0 || M <= 0) return fail(VR_ERR_SHAPE, "N, T, V, M must be positive (got %lld, %lld, %d, %d)", (long long)N, (long long)T, V, M);
    if (iq_only) { n_fft = vr::NFFT; hop = 1; img = 0; }
    if (hop <= 0) return fail(VR_ERR_SHAPE, "hop_length must be positive, got %d", hop);
    if (n_fft != vr::NFFT) return fail(VR_ERR_UNSUPPORTED, "this ABI version implements n_fft=256 only (got %d)", n_fft);
    if (!iq_only && T <= n_fft / 2)
        return fail(VR_ERR_SHAPE, "T=%lld must exceed n_fft/2=%d: reflect padding needs it (the reference raises 'Padding size should be less than the corresponding input dimension')", (long long)T, n_fft / 2);
    if (T > (1ll << 30)) return fail(VR_ERR_UNSUPPORTED, "T=%lld too long", (long long)T);
    if ((int64_t)V * M * 4 > 65535) return fail(VR_ERR_UNSUPPORTED, "V*M=%lld too large", (long long)V * M);
    Partition P;
    int rc = partition_edges(src, dst, E, V, P);
    if (rc) return rc;

    memset(&p, 0, sizeof(p));
    p.N = N; p.T = T; p.V = V; p.M = M; p.E = E; p.hop = hop; p.VM = V * M;
    p.F = iq_only ? 0 : (int)(T / hop) + 1;
    p.iq_only = iq_only ? 1 : 0;
    p.inv_E = 1.0f / (float)E;
    p.negzero = -0.0f;
    p.plane_floats = vr::TL * p.VM;
    p.stage_bytes = round_up(3 * p.plane_floats * 4, 128);
    p.tma_in = (x_aligned && ((T * p.VM) % 4 == 0)) ? 1 : 0;

    // tables (warp-uniform in the kernel: one bone group per warp of a team); within a group the
    // source joints with exactly one bone are listed first (the kernel runs them two at a time)
    p.eg_max = p.sg_max = 0;
    for (int g = 0; g < vr::NG; ++g) {
        p.ne[g] = P.ne[g]; p.ns[g] = P.ns[g]; p.ns1[g] = 0;
        p.eg_max = std::max(p.eg_max, P.ne[g]);
        p.sg_max = std::max(p.sg_max, P.ns[g]);
        int ei = 0, si = 0;
        for (int pass = 0; pass < 2; ++pass)
            for (size_t s = 0; s < P.src_of[g].size(); ++s) {
                const bool single = P.edges_of[g][s].size() == 1;
                if (single != (pass == 0)) continue;
                const int eb = ei;
                for (int e : P.edges_of[g][s]) {
                    p.etab[g * vr::MAX_EG + ei] = (uint32_t)(src[e] * M * 4) | ((uint32_t)(dst[e] * M * 4) << 16);
                    ++ei;
                }
                p.stab[g * vr::MAX_SG + si] = (uint32_t)(P.src_of[g][s] * M * 4) | ((uint32_t)eb << 16) | ((uint32_t)ei << 24);
                ++si;
                if (single) p.ns1[g]++;
            }
    }

    // output columns: the frames themselves, or the image columns of the fused nearest resize
    p.img = img;
    p.ncols = img ? img : p.F;
    p.cscale = img ? (float)p.F / (float)img : 1.f;          // ATen compute_scales_value<float>: float(in) / out
    p.rscale = img ? (float)n_fft / (float)img : 1.f;
    p.sparse = (img && p.F > img) ? 1 : 0;

    // jobs: columns per job bounded by the z buffer
    auto span_of = [&](int CJ, int& zspan, int& cmax, int& slots) {
        const int jps = (p.ncols + CJ - 1) / CJ;
        zspan = cmax = slots = 0;
        for (int j = 0; j < jps; ++j) {
            vr::JobGeom g = vr::job_geom(j, jps, CJ, p.ncols, p.img, p.cscale, p.F, hop, (int)T);
            zspan = std::max(zspan, g.hi - g.lo + 1);
            cmax = std::max(cmax, g.nchunks);
            slots = std::max(slots, p.sparse ? g.nc : g.nf);
        }
    };
    int fj_max = (ZCAP_MAX - vr::NFFT - 2 * vr::TL - 2) / hop + 1;     // frames whose span fits the z buffer
    if (fj_max < 1) return fail(VR_ERR_UNSUPPORTED, "hop_length=%d too large", hop);
    int zspan = 0, cmax = 0, slots = 0;
    if (iq_only) {
        // samples per job: whole chunks, as many as the z buffer holds, evened out over the jobs of a sequence
        const int cap = ZCAP_MAX / vr::TL * vr::TL;
        const long long jps = (T + cap - 1) / cap;
        p.FJ = round_up((int)((T + jps - 1) / jps), vr::TL);
        p.jobs_per_seq = (int)((T + p.FJ - 1) / p.FJ);
    } else if (!img) {
        p.jobs_per_seq = (p.F + fj_max - 1) / fj_max;
        p.FJ = (p.F + p.jobs_per_seq - 1) / p.jobs_per_seq;
    } else {
        // columns per job: start from the estimate frames/scale, shrink until the exact span fits
        double est = (double)fj_max / std::max((double)p.cscale, 1e-6);
        int CJ = (int)std::min<double>(std::max(est, 1.0), (double)p.ncols);
        for (;;) {
            int jps = (p.ncols + CJ - 1) / CJ;
            CJ = (p.ncols + jps - 1) / jps;                               // even out the jobs (never grows CJ)
            if (CJ >= 8 && jps > 1) CJ = CJ / 4 * 4;                      // keep job boundaries float4-aligned
            span_of(CJ, zspan, cmax, slots);
            if (zspan <= ZCAP_MAX || CJ == 1) break;
            CJ = std::max(1, std::min(CJ - 1, CJ * ZCAP_MAX / zspan));
        }
        if (zspan > ZCAP_MAX) return fail(VR_ERR_UNSUPPORTED, "no job split fits the z buffer (T=%lld, hop=%d, image_size=%d)", (long long)T, hop, img);
        p.FJ = CJ;
    }
    if (!iq_only) p.jobs_per_seq = (p.ncols + p.FJ - 1) / p.FJ;
    p.n_jobs = N * (long long)p.jobs_per_seq;
    if (p.n_jobs >= (1ll << 31) / 2) return fail(VR_ERR_UNSUPPORTED, "N*jobs_per_seq=%lld too large for one launch; split the batch", p.n_jobs);
    if (iq_only) { zspan = p.FJ; cmax = p.FJ / vr::TL; }
    else span_of(p.FJ, zspan, cmax, slots);
    p.zcap = round_up(zspan, 16);
    p.cmax = cmax;

    // output tile
    const int FB_BULK_MAX = 20;
    if (iq_only) { p.FB = 0; p.ostride = 0; p.bulk_out = 0; }        // no output tile in shared memory
    else if (!img && p.jobs_per_seq == 1 && p.F <= FB_BULK_MAX) { p.FB = p.F; p.ostride = p.F; p.bulk_out = 1; }
    else if (img && slots <= FB_BULK_MAX) { p.FB = slots; p.ostride = slots | 1; p.bulk_out = 0; }
    else { p.FB = 16; p.ostride = 17; p.bulk_out = 0; }

    // consumer warps (teams of NG) / CTAs per SM / ring depth
    int W = g_tuning.warps > 0 ? g_tuning.warps : 8;
    W = std::min(W, std::min(vr::MAX_WARPS, VR_LB_THREADS / 32 - 1));
    W = std::max(vr::NG, W / vr::NG * vr::NG);
    p.W = W;
    const int NB = (M % 2 == 0) ? 2 : 1;
    p.scr_bytes = round_up(std::max(vr::XCH_BYTES, p.eg_max * 128 * NB), 128);
    p.xg_bytes = round_up(2 * vr::NG * 32 * NB * 4, 128);        // double-buffered
    int off = 0;
    off += round_up(vr::MAX_STAGES * (8 + 8 + 4) + 10 * 4, 128);          // full[] / empty[] mbarriers, issued sequence numbers, job queue
    p.off_tw = off;  off += (7 * 32 + 7 * 4) * 16 + vr::NFFT * 4;        // pass-1 / pass-2 twiddles, Hann window
    p.zpark = park ? 1 : 0;
    p.off_z = off;   off += round_up((park ? 1 : vr::NG) * p.zcap * 8, 128);   // the job's complex baseband samples (per bone group if !park)
    p.off_zp = off;  if (park) off += (W / vr::NG) * 2 * vr::NG * 32 * 8;     // per team: two parking buffers of 4 x 32 partial sums
    p.off_o = off;   off += round_up(vr::NFFT * p.ostride * 4, 128);
    p.off_scr = off; off += W * p.scr_bytes;
    p.off_xg = off;  off += (W / vr::NG) * p.xg_bytes;
    p.off_tab = off; if (ups) off += (W / vr::NG) * (int)sizeof(vr::UpsTab);   // per-team (offset, interval) of the chunk's steps
    p.off_ring = off;
    const int SMEM_SM = 233472, SMEM_CTA_MAX = 232448;
    const int teams = W / vr::NG;
    ctas_per_sm = g_tuning.ctas_per_sm > 0 ? g_tuning.ctas_per_sm : 2;
    int S = 0;
    for (; ctas_per_sm >= 1; --ctas_per_sm) {
        int budget = std::min(SMEM_SM / ctas_per_sm - 1024, SMEM_CTA_MAX);
        S = (budget - off) / p.stage_bytes;
        S = std::min(S, std::min(vr::MAX_STAGES, 3 * teams));
        if (g_tuning.stages > 0) S = std::min(S, g_tuning.stages);
        if (ups) { if (S >= teams) { S = teams; break; } continue; }    // fused up-sampling: one stage per team, no ring
        if (S >= teams + 1 || (ctas_per_sm == 1 && S >= 2)) break;
    }
    if (ctas_per_sm < 1 || S < 2)
        return fail(VR_ERR_UNSUPPORTED, "V*M=%d needs %d-byte chunks; no room for a load ring in shared memory", p.VM, p.stage_bytes);
    p.S = S;
    p.smem_bytes = off + S * p.stage_bytes;
    grid = (int)std::min<long long>(p.n_jobs, (long long)sm_count * ctas_per_sm);
    return VR_OK;
}

// Short sequences (one job each) keep one z plane per bone group and sum them once per job.  Long
// sequences are cut into jobs whose samples fit the z buffer; there a single plane is kept and the four
// partial sums of a chunk are parked and folded one chunk later.  A larger buffer means less halo
// (n_fft + 2 chunks of samples are synthesised twice at every cut) but can cost the second resident CTA
// per SM; two CTAs matter more (the kernel is latency-bound with one), so take the largest buffer that
// still leaves room for two.
int make_plan(int64_t N, int64_t T, int V, int M, const int32_t* src, const int32_t* dst, int E,
              int n_fft, int hop, int img, bool ups, int sm_count, bool x_aligned, vr::Params& p, int& grid, int& ctas_per_sm,
              bool iq_only = false) {
    const int want = g_tuning.ctas_per_sm > 0 ? g_tuning.ctas_per_sm : 2;
    const int caps[] = {2304, 1920, 1664, 1408, 1152};
    int rc = make_plan_z(N, T, V, M, src, dst, E, n_fft, hop, img, ups, iq_only, sm_count, x_aligned, caps[0], ups, p, grid, ctas_per_sm);
    if (rc || (!ups && ctas_per_sm >= want && p.jobs_per_seq == 1)) return rc;
    for (int zc : caps) {
        vr::Params q;
        int g2, c2;
        if (make_plan_z(N, T, V, M, src, dst, E, n_fft, hop, img, ups, iq_only, sm_count, x_aligned, zc, true, q, g2, c2) == VR_OK && c2 >= want) {
            p = q; grid = g2; ctas_per_sm = c2;
            return VR_OK;
        }
    }
    g_err[0] = 0;
    return make_plan_z(N, T, V, M, src, dst, E, n_fft, hop, img, ups, iq_only, sm_count, x_aligned, caps[0], true, p, grid, ctas_per_sm);
}

// ---- team-job schedule (vr_team_kernel) -----------------------------------------------------------
// Applies to batches of short sequences (one job per sequence, plain (N, n_fft, F) output in one bulk store, every
// chunk loadable by TMA).  Every team of 4 warps owns a whole sequence: private 2-stage ring, single z plane with
// parked partial sums, output tile built in the stage of the job's last chunk.  `p` comes from make_plan (bone
// tables, shapes); this re-lays the shared memory.  Returns false when the shape does not qualify.
bool make_team_plan(vr::Params& p, int sm_count, int& grid) {
    if (p.jobs_per_seq != 1 || p.img || !p.bulk_out || !p.tma_in) return false;
    const int T = (int)p.T;
    const int last = T - (T - 1) / vr::TL * vr::TL;                      // time steps of the last chunk
    if ((last * p.VM) % 4 != 0) return false;                            // its planes must be 16-byte multiples for TMA
    const int NB = (p.M % 2 == 0) ? 2 : 1;
    const int W = vr::TJ_TEAMS * vr::NG;
    p.W = W;
    p.zpark = 1;
    p.team_jobs = 1;
    p.zcap = round_up(T, 16);
    p.z_stride = round_up(p.zcap * 8, 128);
    p.stage_bytes = round_up(std::max(3 * p.plane_floats * 4, vr::NFFT * p.F * 4), 128);
    p.scr_bytes = round_up(std::max(vr::XCH_BYTES, p.eg_max * 128 * NB), 128);
    p.xg_bytes = round_up(2 * vr::NG * 32 * NB * 4, 128);
    int off = 128;                                                       // mbarriers + stage metadata
    p.off_tw = off;  off += round_up((7 * 32 + 7 * 4) * 16 + vr::NFFT * 4, 128);
    p.off_z = off;   off += vr::TJ_TEAMS * p.z_stride;
    p.off_zp = off;  off += vr::TJ_TEAMS * 2 * vr::NG * 32 * 8;
    p.off_scr = off; off += W * p.scr_bytes;
    p.off_xg = off;  off += vr::TJ_TEAMS * p.xg_bytes;
    p.off_ring = off; off += vr::TJ_TEAMS * vr::TJ_RS * p.stage_bytes;
    p.S = vr::TJ_RS;
    p.smem_bytes = off;
    const int SMEM_SM = 233472;
    if (p.smem_bytes > SMEM_SM / 2 - 1024) return false;                 // two CTAs per SM or not at all
    grid = (int)std::min<long long>((p.n_jobs + vr::TJ_TEAMS - 1) / vr::TJ_TEAMS, (long long)sm_count * 2);
    return true;
}

typedef void (*KernelFn)(const vr::Params);
// ps: per-sequence placements (VR_FLAG_PER_SEQUENCE); the scalar instantiations are the kernels without them
struct TeamVariant { bool fma; int vm; int nb; bool ps; KernelFn fn; };
#define VR_TEAM_VARIANT(VM, NB, PS) {false, VM, NB, PS, vr::vr_team_kernel<false, VM, NB, PS>}, \
                                    {true, VM, NB, PS, vr::vr_team_kernel<true, VM, NB, PS>}
const TeamVariant kTeamVariants[] = { VR_TEAM_VARIANT(0, 1, false), VR_TEAM_VARIANT(0, 2, false), VR_TEAM_VARIANT(50, 2, false),
                                      VR_TEAM_VARIANT(0, 1, true), VR_TEAM_VARIANT(0, 2, true), VR_TEAM_VARIANT(50, 2, true) };
const int kNumTeamVariants = sizeof(kTeamVariants) / sizeof(kTeamVariants[0]);
// vmc (optional): the compile-time V*M of the instantiation picked, 0 for the generic one
KernelFn pick_team_kernel(bool fma, int vm, int m, bool ps, int* vmc = nullptr) {
    const int nb = (m % 2 == 0) ? 2 : 1;
    KernelFn generic = nullptr;
    if (vmc) *vmc = 0;
    for (int i = 0; i < kNumTeamVariants; ++i) {
        if (kTeamVariants[i].fma != fma || kTeamVariants[i].nb != nb || kTeamVariants[i].ps != ps) continue;
        if (kTeamVariants[i].vm == vm) { if (vmc) *vmc = vm; return kTeamVariants[i].fn; }
        if (kTeamVariants[i].vm == 0) generic = kTeamVariants[i].fn;
    }
    return generic;
}

// kernel variants: range rounding mode x compile-time V*M (plane stride as an immediate); VM=0 is generic
struct Variant { bool fma; int vm; int nb; bool ups; bool park; bool ps; KernelFn fn; };
#define VR_VARIANT(VM, NB, UPS, PARK, PS) {false, VM, NB, UPS, PARK, PS, vr::vr_fused_kernel<false, VM, NB, UPS, PARK, PS>}, \
                                          {true, VM, NB, UPS, PARK, PS, vr::vr_fused_kernel<true, VM, NB, UPS, PARK, PS>}
#define VR_VARIANTS(PS) \
    /* short sequences (one job each, a z plane per bone group): generic V*M, one / two bodies at a time; NTU */ \
    VR_VARIANT(0, 1, false, false, PS), VR_VARIANT(0, 2, false, false, PS), VR_VARIANT(50, 2, false, false, PS), \
    /* long sequences (several jobs, parked partial sums) */ \
    VR_VARIANT(0, 1, false, true, PS), VR_VARIANT(0, 2, false, true, PS), VR_VARIANT(50, 2, false, true, PS), \
    /* fused temporal up-sampling (always long) */ \
    VR_VARIANT(0, 1, true, true, PS), VR_VARIANT(0, 2, true, true, PS), VR_VARIANT(50, 2, true, true, PS)
const Variant kVariants[] = { VR_VARIANTS(false), VR_VARIANTS(true) };
const int kNumVariants = sizeof(kVariants) / sizeof(kVariants[0]);
KernelFn pick_kernel(bool fma, int vm, int m, bool ups, bool park, bool ps, int* vmc = nullptr) {
    const int nb = (m % 2 == 0) ? 2 : 1;
    KernelFn generic = nullptr;
    if (vmc) *vmc = 0;
    for (int i = 0; i < kNumVariants; ++i) {
        if (kVariants[i].fma != fma || kVariants[i].nb != nb || kVariants[i].ups != ups || kVariants[i].park != park ||
            kVariants[i].ps != ps) continue;
        if (kVariants[i].vm == vm) { if (vmc) *vmc = vm; return kVariants[i].fn; }
        if (kVariants[i].vm == 0) generic = kVariants[i].fn;
    }
    return generic;
}

constexpr int TEAM_AUTO_WAVES = 3;      // automatic schedule: team-job kernel from this many jobs per team slot

struct DeviceInfo {
    int sm_count = 0; bool attr_set = false; int* tickets = nullptr; unsigned next_slot = 0;
    double* param_partials = nullptr; unsigned* param_count = nullptr; unsigned next_param_slot = 0;
    float* splitk_pool = nullptr; unsigned next_splitk_slot = 0;
};
std::mutex g_mu;
DeviceInfo g_dev[64];

// VR_FLAG_VIEWS: R radars per x sequence (R = 1 without the field).  Valid only with VR_FLAG_PER_SEQUENCE (every view has
// its own placement), and N -- the outputs -- must be a multiple of R.  Host-side, before anything touches the device.
int views_of(uint32_t flags, int64_t N, int& R) {
    R = (int)((flags & VR_FLAG_VIEWS_MASK) >> VR_FLAG_VIEWS_SHIFT);
    if (R == 0) { R = 1; return VR_OK; }
    if (!(flags & VR_FLAG_PER_SEQUENCE))
        return fail(VR_ERR_ARG, "VR_FLAG_VIEWS(%d) needs VR_FLAG_PER_SEQUENCE: each view has its own placement", R);
    if (N % R != 0) return fail(VR_ERR_SHAPE, "N=%lld outputs is not a multiple of the %d views per sequence", (long long)N, R);
    return VR_OK;
}

// vr_set_noise's pending setting, consumed by the next entry call of the thread that carries VR_FLAG_NOISE
struct NoiseSlot {
    const float* std = nullptr;
    const uint64_t* seed = nullptr;
};
thread_local NoiseSlot t_noise;

// The noise of an entry call: consumes the thread's pending setting when the flags ask for noise (the slot is cleared
// whether the call then succeeds or fails), nothing otherwise.  Host-side, before anything is enqueued.
int take_noise(uint32_t flags, vr::NoiseParams& q) {
    q.std = nullptr; q.seed = nullptr;
    if (!(flags & VR_FLAG_NOISE)) return VR_OK;
    const NoiseSlot s = t_noise;
    t_noise = NoiseSlot{};
    if (!(flags & VR_FLAG_PER_SEQUENCE))
        return fail(VR_ERR_ARG, "VR_FLAG_NOISE needs VR_FLAG_PER_SEQUENCE: the noise level is one per output");
    if (!s.std) return fail(VR_ERR_ARG, "VR_FLAG_NOISE without a pending vr_set_noise on this thread");
    q.std = s.std; q.seed = reinterpret_cast<const unsigned long long*>(s.seed);
    return VR_OK;
}

// The entries that do not take VR_FLAG_NOISE (the host entry, the backward entries) still consume a pending setting when
// a call carries the flag, before rejecting it, so that a stale setting never reaches a later launch
void drop_noise(uint32_t flags) {
    if (flags & VR_FLAG_NOISE) t_noise = NoiseSlot{};
}

int device_setup(int& dev, int& sm_count) {
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return fail(VR_ERR_CUDA, "device index %d out of range", dev);
    std::lock_guard<std::mutex> lk(g_mu);
    DeviceInfo& d = g_dev[dev];
    if (!d.attr_set) {
        cudaDeviceProp prop;
        CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
        if (prop.major < 10)
            return fail(VR_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", dev, prop.major, prop.minor);
        d.sm_count = prop.multiProcessorCount;
        for (int i = 0; i < kNumVariants; ++i)
            CUDA_TRY(cudaFuncSetAttribute(kVariants[i].fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
        for (int i = 0; i < kNumTeamVariants; ++i)
            CUDA_TRY(cudaFuncSetAttribute(kTeamVariants[i].fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
        CUDA_TRY(cudaGetSymbolAddress((void**)&d.tickets, vr::g_ticket_pool));
        CUDA_TRY(cudaFuncSetAttribute(vr::vr_stft_adjoint_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, vr::ADJ_SEG_MAX * 8));
        CUDA_TRY(cudaGetSymbolAddress((void**)&d.param_partials, vr::g_param_partials));
        CUDA_TRY(cudaGetSymbolAddress((void**)&d.param_count, vr::g_param_count));
        CUDA_TRY(cudaGetSymbolAddress((void**)&d.splitk_pool, vr::g_splitk_pool));
        d.attr_set = true;
    }
    sm_count = d.sm_count;
    return VR_OK;
}

// a counter pair for one launch with more jobs than CTAs (dynamic job scheduling)
int* next_ticket_slot(int dev) {
    std::lock_guard<std::mutex> lk(g_mu);
    DeviceInfo& d = g_dev[dev];
    return d.tickets + 2 * (d.next_slot++ % vr::TICKET_SLOTS);
}

// a slot of the parameter-gradient partials for one synthesis-adjoint launch
void next_param_slot(int dev, vr::BwdParams& p) {
    std::lock_guard<std::mutex> lk(g_mu);
    DeviceInfo& d = g_dev[dev];
    const unsigned s = d.next_param_slot++ % vr::PARAM_SLOTS;
    p.part = d.param_partials + (size_t)s * vr::PARAM_MAX_BLOCKS * 4;
    p.count = d.param_count + s;
}

// a slot of the kernel gradient's split-K partials for one launch
float* next_splitk_slot(int dev) {
    std::lock_guard<std::mutex> lk(g_mu);
    DeviceInfo& d = g_dev[dev];
    return d.splitk_pool + (size_t)(d.next_splitk_slot++ % vr::G_SPLIT_SLOTS) * vr::G_SPLIT_SLOT_FLOATS;
}

// Plans depend only on shapes and the bone list; the last one is kept per host thread so that a
// training loop calling forward() with the same shapes pays for partitioning and planning once.
struct PlanCache {
    bool valid = false;
    int64_t N = 0, T = 0;
    int V = 0, M = 0, E = 0, n_fft = 0, hop = 0, img = 0, sm_count = 0, grid = 0, cps = 0;
    bool aligned = false, ups = false, iq_only = false;
    Tuning tuning;
    std::vector<int32_t> src, dst;
    vr::Params p;
};
thread_local PlanCache t_plan;

int cached_plan(int64_t N, int64_t T, int V, int M, const int32_t* src, const int32_t* dst, int E,
                int n_fft, int hop, int img, bool ups, bool iq_only, int sm_count, bool aligned, vr::Params& p, int& grid, int& cps) {
    PlanCache& c = t_plan;
    if (c.valid && c.N == N && c.T == T && c.V == V && c.M == M && c.E == E && c.n_fft == n_fft && c.hop == hop && c.img == img && c.ups == ups &&
        c.iq_only == iq_only &&
        c.sm_count == sm_count && c.aligned == aligned && src && dst &&
        c.tuning.warps == g_tuning.warps && c.tuning.ctas_per_sm == g_tuning.ctas_per_sm && c.tuning.stages == g_tuning.stages &&
        memcmp(c.src.data(), src, sizeof(int32_t) * E) == 0 && memcmp(c.dst.data(), dst, sizeof(int32_t) * E) == 0) {
        p = c.p; grid = c.grid; cps = c.cps;
        return VR_OK;
    }
    c.valid = false;
    int rc = make_plan(N, T, V, M, src, dst, E, n_fft, hop, img, ups, sm_count, aligned, p, grid, cps, iq_only);
    if (rc) return rc;
    c.N = N; c.T = T; c.V = V; c.M = M; c.E = E; c.n_fft = n_fft; c.hop = hop; c.img = img; c.ups = ups; c.iq_only = iq_only;
    c.sm_count = sm_count; c.aligned = aligned;
    c.tuning = g_tuning;
    c.src.assign(src, src + E); c.dst.assign(dst, dst + E);
    c.p = p; c.grid = grid; c.cps = cps; c.valid = true;
    return VR_OK;
}

// Samples of a sequence that no job of a spectrogram plan synthesises.  A job covers the samples its frames' windows reach
// (job_geom), so with hop > n_fft / 2 the samples between two frames' windows and after the last window belong to no job:
// the spectrogram never reads them, but a debug launch must still write them to iq (launch fills them in).
bool iq_gaps(const vr::Params& p) {
    if (p.iq_only) return false;
    int next = 0;
    for (int j = 0; j < p.jobs_per_seq; ++j) {
        const vr::JobGeom g = vr::job_geom(j, p.jobs_per_seq, p.FJ, p.ncols, p.img, p.cscale, p.F, p.hop, (int)p.T);
        if (g.lo > next) return true;
        next = std::max(next, g.hi + 1);
    }
    return next < (int)p.T;
}

// The configuration of one fused launch: the plan, the schedule and the kernel instantiation.  launch() runs exactly
// this; vr_plan_launch reports it without a GPU.  debug: iq is written as well as out (never the team-job kernel);
// schedule: vr_set_schedule's mode.
struct LaunchPlan {
    vr::Params p;
    int grid = 0, cps = 0, vmc = 0;
    bool team = false, ticket = false;
    KernelFn fn = nullptr;
};
int plan_launch(int64_t N, int64_t T, int V, int M, const int32_t* src, const int32_t* dst, int E, int n_fft, int hop, int img,
                bool ups, bool iq_only, bool debug, uint32_t flags, bool aligned, int schedule, int sm_count, bool cached,
                LaunchPlan& L) {
    int rc = cached ? cached_plan(N, T, V, M, src, dst, E, n_fft, hop, img, ups, iq_only, sm_count, aligned, L.p, L.grid, L.cps)
                    : make_plan(N, T, V, M, src, dst, E, n_fft, hop, img, ups, sm_count, aligned, L.p, L.grid, L.cps, iq_only);
    if (rc) return rc;
    // schedule: batches with several sequences per team slot take the team-job kernel (no CTA-wide barriers, a double
    // buffer per team); small batches keep the cooperative kernel, whose latency per sequence is half
    L.team = false;
    if (!ups && !iq_only && !debug && !g_timeline && schedule != 0) {
        vr::Params q = L.p;
        int tg = 0;
        // automatic: from TEAM_AUTO_WAVES jobs per team slot in plain stream order (below that the cooperative kernel's
        // shorter latency per sequence wins: N = 1024 66 vs 74 us, N = 4096 248 vs 228 us); always when the caller has
        // declared the batches independent -- consecutive launches then overlap and only throughput counts
        // (N = 256: 14.8 vs 16.3 us per launch)
        const bool overlapped = g_pdl && (flags & VR_FLAG_INPUTS_READY);
        if (make_team_plan(q, sm_count, tg) &&
            (schedule == 1 || overlapped || q.n_jobs >= (long long)TEAM_AUTO_WAVES * sm_count * 2 * vr::TJ_TEAMS)) {
            L.p = q; L.grid = tg; L.team = true;
        }
    }
    const int job_slots = L.team ? L.grid * vr::TJ_TEAMS : L.grid;
    L.ticket = g_dynamic && L.p.n_jobs > job_slots;
    const bool fma = (flags & VR_FLAG_RANGE_FMA) != 0, per_seq = (flags & VR_FLAG_PER_SEQUENCE) != 0;
    L.fn = L.team ? pick_team_kernel(fma, L.p.VM, L.p.M, per_seq, &L.vmc)
                  : pick_kernel(fma, L.p.VM, L.p.M, ups, L.p.zpark != 0, per_seq, &L.vmc);
    return VR_OK;
}

int launch(const float* x, int64_t N, int64_t T, int V, int M, const int32_t* src, const int32_t* dst, int E,
           const float* lam_dev, const float* loc_dev, float lam_val, const float* loc_val,
           int n_fft, int hop, uint32_t flags, int img, float* out, float* iq, cudaStream_t stream,
           const double* coef = nullptr, int ups_T = 0, int ups_K = 0, const vr::NoiseParams& noise = vr::NoiseParams{}) {
    // coef != nullptr: fused temporal up-sampling; T is then the UP-SAMPLED length ups_K * ups_T and x is only
    // used for its alignment (the kernel reads the spline coefficients instead).  out == nullptr: synthesis only (iq).
    // noise: from take_noise (VR_FLAG_NOISE), read by the PS kernels only
    const bool iq_only = out == nullptr;
    if (!x || (!out && !iq)) return fail(VR_ERR_ARG, "x and out (or iq) must not be null");
    if ((lam_dev == nullptr) != (loc_dev == nullptr)) return fail(VR_ERR_ARG, "wavelength and radar_location must both be device pointers or both be null");
    if (flags & ~(VR_FLAG_RANGE_FMA | VR_FLAG_INPUTS_READY | VR_FLAG_PER_SEQUENCE | VR_FLAG_VIEWS_MASK | VR_FLAG_NOISE))
        return fail(VR_ERR_ARG, "unknown flags 0x%x", flags);
    if (((flags & VR_FLAG_NOISE) != 0) != (noise.std != nullptr))
        return fail(VR_ERR_ARG, "VR_FLAG_NOISE needs a noise setting (vr_set_noise) and a noise setting needs the flag");
    int views;
    int rc = views_of(flags, N, views);
    if (rc) return rc;
    int dev, sm_count;
    rc = device_setup(dev, sm_count);
    if (rc) return rc;
    LaunchPlan L;
    rc = plan_launch(N, T, V, M, src, dst, E, n_fft, hop, img, coef != nullptr, iq_only, iq != nullptr, flags,
                     ((uintptr_t)x & 15) == 0, g_schedule, sm_count, true, L);
    if (rc) return rc;
    vr::Params& p = L.p;
    p.x = x; p.out = out; p.iq = iq; p.tl = g_timeline;
    p.views = views;
    p.noise = noise;
    p.ticket = L.ticket ? next_ticket_slot(dev) : nullptr;
    p.early_reads = (g_pdl && !coef && (flags & VR_FLAG_INPUTS_READY)) ? 1 : 0;   // coef is written by the launch just before
    p.coef = coef; p.ups_T = ups_T; p.ups_K = ups_K;
    p.ups_ratio = coef ? (double)(ups_T - 1) / (double)((long long)ups_K * ups_T - 1) : 0.0;
    p.lam_ptr = lam_dev; p.loc_ptr = loc_dev;
    p.lam_val = lam_val;
    if (loc_val) { p.loc_val[0] = loc_val[0]; p.loc_val[1] = loc_val[1]; p.loc_val[2] = loc_val[2]; }
    // Programmatic dependent launch: the kernel's prologue (barrier init, twiddle table) may overlap
    // the tail of the previous kernel in the stream; the kernel executes griddepcontrol.wait before
    // its first global-memory access, so stream order is preserved.
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)L.grid); cfg.blockDim = dim3(L.team ? (unsigned)vr::TJ_THREADS : (unsigned)(p.W + 1) * 32);
    cfg.dynamicSmemBytes = (size_t)p.smem_bytes; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = g_pdl ? 1 : 0;
    cfg.attrs = attr; cfg.numAttrs = 1;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, L.fn, p));
    // A debug launch writes every sample of iq: where its plan leaves samples to no job (hop > n_fft / 2), the
    // synthesis-only launch follows on the stream and writes all of iq again -- the same bits where both write (the two
    // launches fold each chunk's partial sums in the same fixed order, and the noise is keyed by (seed, n, t)).  Its
    // stores wait for this launch to complete (griddepcontrol.wait), so the order of the two writes is the stream's.
    if (iq && out && iq_gaps(p))
        return launch(x, N, T, V, M, src, dst, E, lam_dev, loc_dev, lam_val, loc_val, n_fft, hop, flags, img, nullptr, iq,
                      stream, coef, ups_T, ups_K, noise);
    return VR_OK;
}

// ---- host staging for vr_forward_host_f32 ---------------------------------------------------------
struct Staging {
    float* x[2] = {nullptr, nullptr};
    float* o[2] = {nullptr, nullptr};
    size_t xcap = 0, ocap = 0;
    cudaStream_t st[2] = {nullptr, nullptr};
};
Staging g_stage[64];
std::mutex g_stage_mu[64];                        // one per device: host-pipelined calls on different devices do not serialise

}  // namespace

extern "C" {

int vr_abi_version(void) { return VR_ABI_VERSION; }
const char* vr_last_error(void) { return g_err; }

int vr_set_tuning(int warps, int ctas_per_sm, int stages) {
    if (warps < 0 || warps > vr::MAX_WARPS || ctas_per_sm < 0 || ctas_per_sm > 4 || stages < 0)
        return fail(VR_ERR_ARG, "bad tuning (%d,%d,%d)", warps, ctas_per_sm, stages);
    g_tuning.warps = warps; g_tuning.ctas_per_sm = ctas_per_sm; g_tuning.stages = stages;
    return VR_OK;
}

int vr_set_schedule(int mode) {
    if (mode < -1 || mode > 1) return fail(VR_ERR_ARG, "schedule must be -1 (automatic), 0 (cooperative) or 1 (team jobs), got %d", mode);
    g_schedule = mode;
    return VR_OK;
}

int vr_set_noise(const float* noise_std_dev, const uint64_t* seed_dev) {
    t_noise = NoiseSlot{};
    if (!noise_std_dev || !seed_dev) return fail(VR_ERR_ARG, "noise_std_dev and seed_dev must not be null");
    if (((uintptr_t)noise_std_dev & 3) != 0 || ((uintptr_t)seed_dev & 7) != 0)
        return fail(VR_ERR_ARG, "noise_std_dev must be 4-byte and seed_dev 8-byte aligned");
    t_noise.std = noise_std_dev; t_noise.seed = seed_dev;
    return VR_OK;
}

int vr_forward_f32(const float* x_dev, int64_t N, int64_t T, int32_t V, int32_t M,
                   const int32_t* src_host, const int32_t* dst_host, int32_t E,
                   const float* wavelength_dev, const float* radar_loc_dev,
                   int32_t n_fft, int32_t hop, uint32_t flags, float* out_dev, void* stream) {
    vr::NoiseParams nz;
    if (int rc = take_noise(flags, nz)) return rc;
    if (!wavelength_dev || !radar_loc_dev) return fail(VR_ERR_ARG, "wavelength_dev and radar_loc_dev must not be null");
    return launch(x_dev, N, T, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev, 0.f, nullptr,
                  n_fft, hop, flags, 0, out_dev, nullptr, (cudaStream_t)stream, nullptr, 0, 0, nz);
}

int vr_forward_debug_f32(const float* x_dev, int64_t N, int64_t T, int32_t V, int32_t M,
                         const int32_t* src_host, const int32_t* dst_host, int32_t E,
                         const float* wavelength_dev, const float* radar_loc_dev,
                         int32_t n_fft, int32_t hop, uint32_t flags, float* out_dev, float* iq_dev, void* stream) {
    vr::NoiseParams nz;
    if (int rc = take_noise(flags, nz)) return rc;
    if (!wavelength_dev || !radar_loc_dev) return fail(VR_ERR_ARG, "wavelength_dev and radar_loc_dev must not be null");
    if (!iq_dev) return fail(VR_ERR_ARG, "iq_dev must not be null");
    return launch(x_dev, N, T, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev, 0.f, nullptr,
                  n_fft, hop, flags, 0, out_dev, iq_dev, (cudaStream_t)stream, nullptr, 0, 0, nz);
}

int vr_synth_f32(const float* x_dev, int64_t N, int64_t T, int32_t V, int32_t M,
                 const int32_t* src_host, const int32_t* dst_host, int32_t E,
                 const float* wavelength_dev, const float* radar_loc_dev, uint32_t flags, float* iq_dev, void* stream) {
    vr::NoiseParams nz;
    if (int rc = take_noise(flags, nz)) return rc;
    if (!wavelength_dev || !radar_loc_dev) return fail(VR_ERR_ARG, "wavelength_dev and radar_loc_dev must not be null");
    if (!iq_dev) return fail(VR_ERR_ARG, "iq_dev must not be null");
    return launch(x_dev, N, T, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev, 0.f, nullptr,
                  vr::NFFT, 1, flags, 0, nullptr, iq_dev, (cudaStream_t)stream, nullptr, 0, 0, nz);
}

int vr_forward_image_f32(const float* x_dev, int64_t N, int64_t T, int32_t V, int32_t M,
                         const int32_t* src_host, const int32_t* dst_host, int32_t E,
                         const float* wavelength_dev, const float* radar_loc_dev,
                         int32_t n_fft, int32_t hop, uint32_t flags, int32_t image_size,
                         float* out_dev, void* stream) {
    vr::NoiseParams nz;
    if (int rc = take_noise(flags, nz)) return rc;
    if (!wavelength_dev || !radar_loc_dev) return fail(VR_ERR_ARG, "wavelength_dev and radar_loc_dev must not be null");
    if (image_size < 1) return fail(VR_ERR_SHAPE, "image_size must be positive, got %d", image_size);
    return launch(x_dev, N, T, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev, 0.f, nullptr,
                  n_fft, hop, flags, image_size, out_dev, nullptr, (cudaStream_t)stream, nullptr, 0, 0, nz);
}

int vr_job_geometry(int64_t N, int64_t T, int32_t V, int32_t M, const int32_t* src_host, const int32_t* dst_host,
                    int32_t E, int32_t n_fft, int32_t hop, int32_t image_size, int64_t job, int64_t geom[8]) {
    if (!geom) return fail(VR_ERR_ARG, "geom must not be null");
    vr::Params p;
    int grid, cps;
    int rc = make_plan(N, T, V, M, src_host, dst_host, E, n_fft, hop, image_size, false, 148, true, p, grid, cps);
    if (rc) return rc;
    if (job < 0 || job >= p.n_jobs) return fail(VR_ERR_ARG, "job %lld outside [0, %lld)", (long long)job, (long long)p.n_jobs);
    const vr::JobGeom g = vr::job_geom((int)job, p.jobs_per_seq, p.FJ, p.ncols, p.img, p.cscale, p.F, hop, (int)T);
    geom[0] = g.n; geom[1] = g.c0; geom[2] = g.nc; geom[3] = g.f0; geom[4] = g.nf; geom[5] = g.lo; geom[6] = g.hi; geom[7] = g.nchunks;
    return VR_OK;
}

int vr_plan_image(int64_t N, int64_t T, int32_t V, int32_t M, const int32_t* src_host, const int32_t* dst_host,
                  int32_t E, int32_t n_fft, int32_t hop, int32_t image_size, int32_t sm_count, int64_t plan[16]) {
    if (!plan) return fail(VR_ERR_ARG, "plan must not be null");
    vr::Params p;
    int grid, cps;
    int rc = make_plan(N, T, V, M, src_host, dst_host, E, n_fft, hop, image_size, false, sm_count > 0 ? sm_count : 148, true, p, grid, cps);
    if (rc) return rc;
    plan[0] = grid; plan[1] = (p.W + 1) * 32; plan[2] = p.smem_bytes; plan[3] = p.S; plan[4] = p.FJ;
    plan[5] = p.jobs_per_seq; plan[6] = p.FB; plan[7] = p.tma_in; plan[8] = p.bulk_out; plan[9] = p.cmax;
    plan[10] = p.sparse; plan[11] = p.ncols; plan[12] = p.zcap; plan[13] = cps; plan[14] = vr::TL; plan[15] = vr::NG;
    return VR_OK;
}

int vr_forward_host_f32(const float* x_host, int64_t N, int64_t T, int32_t V, int32_t M,
                        const int32_t* src_host, const int32_t* dst_host, int32_t E,
                        float wavelength, const float* radar_loc_host,
                        int32_t n_fft, int32_t hop, uint32_t flags, float* out_host, int64_t sub_batch) {
    drop_noise(flags);
    if (!x_host || !out_host || !radar_loc_host) return fail(VR_ERR_ARG, "host pointers must not be null");
    if (flags & (VR_FLAG_PER_SEQUENCE | VR_FLAG_VIEWS_MASK | VR_FLAG_NOISE))
        return fail(VR_ERR_ARG, "vr_forward_host_f32 takes one host placement for the batch; VR_FLAG_PER_SEQUENCE, "
                                "VR_FLAG_VIEWS and VR_FLAG_NOISE need a device-pointer entry point");
    if (N <= 0 || T <= 0 || V <= 0 || M <= 0 || hop <= 0) return fail(VR_ERR_SHAPE, "N, T, V, M, hop must be positive");
    int dev, sm_count;
    int rc = device_setup(dev, sm_count);
    if (rc) return rc;
    const size_t xseq = (size_t)3 * T * V * M, oseq = (size_t)n_fft * (T / hop + 1);
    if (sub_batch <= 0) {
        // ~16 MB of input per sub-batch keeps both copy engines and the SMs busy
        sub_batch = std::max<int64_t>(1, (int64_t)((16u << 20) / (xseq * 4)));
        sub_batch = std::min<int64_t>(sub_batch, (N + 3) / 4 > 0 ? (N + 3) / 4 : 1);
    }
    sub_batch = std::min<int64_t>(sub_batch, N);
    Staging& sg = g_stage[dev];
    std::lock_guard<std::mutex> lk(g_stage_mu[dev]);   // one host-pipelined call per device at a time (the staging buffers are per device)
    if (!sg.st[0]) {
        CUDA_TRY(cudaStreamCreateWithFlags(&sg.st[0], cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&sg.st[1], cudaStreamNonBlocking));
    }
    if (sg.xcap < sub_batch * xseq || sg.ocap < sub_batch * oseq) {
        for (int i = 0; i < 2; ++i) {
            if (sg.x[i]) cudaFree(sg.x[i]);
            if (sg.o[i]) cudaFree(sg.o[i]);
            sg.x[i] = sg.o[i] = nullptr;
        }
        sg.xcap = sg.ocap = 0;
        for (int i = 0; i < 2; ++i) {
            CUDA_TRY(cudaMalloc(&sg.x[i], sub_batch * xseq * 4));
            CUDA_TRY(cudaMalloc(&sg.o[i], sub_batch * oseq * 4));
        }
        sg.xcap = sub_batch * xseq; sg.ocap = sub_batch * oseq;
    }
    int b = 0;
    for (int64_t n0 = 0; n0 < N; n0 += sub_batch, b ^= 1) {
        const int64_t nb = std::min<int64_t>(sub_batch, N - n0);
        CUDA_TRY(cudaMemcpyAsync(sg.x[b], x_host + n0 * xseq, nb * xseq * 4, cudaMemcpyHostToDevice, sg.st[b]));
        rc = launch(sg.x[b], nb, T, V, M, src_host, dst_host, E, nullptr, nullptr, wavelength, radar_loc_host,
                    n_fft, hop, flags, 0, sg.o[b], nullptr, sg.st[b]);
        if (rc) { cudaStreamSynchronize(sg.st[0]); cudaStreamSynchronize(sg.st[1]); return rc; }
        CUDA_TRY(cudaMemcpyAsync(out_host + n0 * oseq, sg.o[b], nb * oseq * 4, cudaMemcpyDeviceToHost, sg.st[b]));
    }
    CUDA_TRY(cudaStreamSynchronize(sg.st[0]));
    CUDA_TRY(cudaStreamSynchronize(sg.st[1]));
    return VR_OK;
}

}  // extern "C"
namespace {
// scipy.ndimage._filters._gaussian_kernel1d(sigma, 0, radius), radius = int(4 * sigma + 0.5), float64; w[0] = centre
int gaussian_weights(float sigma, int& radius, double* w) {
    const double sd = (double)sigma;
    radius = (int)(4.0 * sd + 0.5);
    if (radius > vr::PF_MAX_RADIUS) return fail(VR_ERR_UNSUPPORTED, "sigma=%g needs a Gaussian radius of %d > %d", sd, radius, vr::PF_MAX_RADIUS);
    double phi[2 * vr::PF_MAX_RADIUS + 1], sum = 0.0;
    const double sigma2 = sd * sd;
    for (int i = -radius; i <= radius; ++i) phi[i + radius] = exp(-0.5 / sigma2 * (double)(i * i));
    for (int i = 0; i <= 2 * radius; ++i) sum += phi[i];
    for (int j = 0; j <= radius; ++j) w[j] = phi[radius + j] / sum;
    return VR_OK;
}

// the arguments vr_pad_frames_f32 and its backward pass accept
int pad_check(int64_t N, int64_t T, int32_t V, int32_t M, int32_t num_pad_frames, float sigma) {
    if (N <= 0 || V <= 0 || M <= 0) return fail(VR_ERR_SHAPE, "N, V, M must be positive (got %lld, %d, %d)", (long long)N, V, M);
    if (T < 4) return fail(VR_ERR_SHAPE, "T=%lld: cubic interpolation needs at least 4 frames (scipy interp1d raises ValueError)", (long long)T);
    if (num_pad_frames < 1) return fail(VR_ERR_SHAPE, "num_pad_frames must be >= 1, got %d", num_pad_frames);
    if (!(sigma > 0.f)) return fail(VR_ERR_SHAPE, "sigma must be positive, got %g", (double)sigma);
    if ((double)T * num_pad_frames > 2.0e9) return fail(VR_ERR_UNSUPPORTED, "T*num_pad_frames too large");
    return VR_OK;
}

// the arguments vr_pad_frames_joints accepts
int pad_joints_check(int64_t N, int64_t T, int32_t V, int32_t C, int32_t num_pad_frames, float sigma) {
    if (N <= 0 || V <= 0 || C <= 0) return fail(VR_ERR_SHAPE, "N, V, C must be positive (got %lld, %d, %d)", (long long)N, V, C);
    if (T < 4) return fail(VR_ERR_SHAPE, "T=%lld: cubic interpolation needs at least 4 frames (scipy interp1d raises ValueError)", (long long)T);
    if (num_pad_frames < 1) return fail(VR_ERR_SHAPE, "num_pad_frames must be >= 1, got %d", num_pad_frames);
    if (!(sigma > 0.f)) return fail(VR_ERR_SHAPE, "sigma must be positive, got %g", (double)sigma);
    if ((double)T * num_pad_frames > 2.0e9) return fail(VR_ERR_UNSUPPORTED, "T*num_pad_frames too large");
    return VR_OK;
}

// Launch configuration of the three up-sampling kernels (vr_plan_pad_frames): kind 0 vr_pad_frames_kernel, 1 its backward,
// 2 the notebook variant (MC = C, the coordinates per joint).  One CTA of 1024 threads owns nc adjacent columns of one
// (sequence, coordinate) plane -- of one sequence for kind 2 -- and, for kind 2, one of nrs slices of the output rows;
// the grid strides over the units.  w (optional): the Gaussian weights, w[0] = centre.
struct PadPlan { long long nc, ncb, units, grid, smem, nrs, rows_per_slice; int radius; };
int pad_plan(int kind, int64_t N, int64_t T, int32_t V, int32_t MC, int32_t num_pad_frames, float sigma, int sm_count,
             PadPlan& q, double* w) {
    if (kind < 0 || kind > 2) return fail(VR_ERR_ARG, "kind must be 0 (forward), 1 (backward) or 2 (notebook), got %d", kind);
    int rc = kind == 2 ? pad_joints_check(N, T, V, MC, num_pad_frames, sigma) : pad_check(N, T, V, MC, num_pad_frames, sigma);
    if (rc) return rc;
    double wbuf[vr::PF_MAX_RADIUS + 1];
    rc = gaussian_weights(sigma, q.radius, w ? w : wbuf);
    if (rc) return rc;
    const long long cols = (long long)V * MC, KT = (long long)num_pad_frames * T;
    long long nc;
    if (kind == 0) {                 // 12 bytes per (frame, column) + 8 bytes per frame of shared memory
        nc = (200 * 1024 - 8ll * T) / (12ll * T);
        if (nc < 1) return fail(VR_ERR_UNSUPPORTED, "T=%lld too long for the shared-memory spline solve (max %d frames)", (long long)T, 200 * 1024 / 20);
    } else if (kind == 1) {          // 16 bytes per (frame, column): dL/dys and dL/dM in float64
        if (T > 200 * 1024 / 20)     // the forward's limit (vr_pad_frames_f32)
            return fail(VR_ERR_UNSUPPORTED, "T=%lld too long for the shared-memory spline solve (max %d frames)", (long long)T, 200 * 1024 / 20);
        nc = (200 * 1024) / (16ll * T);
    } else {                         // 16 bytes per (frame, column) + 8 per frame
        nc = (200 * 1024 - 8ll * T) / (16ll * T);
        if (nc < 1) return fail(VR_ERR_UNSUPPORTED, "T=%lld too long for the shared-memory spline solve (max %d frames)", (long long)T, 200 * 1024 / 24);
    }
    nc = std::min<long long>(std::min<long long>(nc, cols), 1024);     // one thread per column solves its spline
    q.ncb = (cols + nc - 1) / nc;
    q.nc = (cols + q.ncb - 1) / q.ncb;                                   // even out the blocks
    q.smem = kind == 0 ? T * q.nc * 12 + T * 8 + 16 : kind == 1 ? T * q.nc * 16 : T * q.nc * 16 + T * 8 + 16;
    q.nrs = 1;
    if (kind == 2) {
        // row slices: only when the per-unit preamble (Gaussian + sequential spline solve, ~50 cycles per frame) is cheap next
        // to the evaluation (a latency-bound chain of conversions and FP64 operations: ~500 cycles per value and thread were
        // measured with one CTA per SM), and only up to one wave of CTAs
        const double solve_cost = 50.0 * (double)T, eval_cost = 500.0 * (double)KT * q.nc / 1024.0;
        long long nrs = std::min<long long>(std::max<long long>(1, sm_count / std::max<long long>(1, N * q.ncb)),
                                            std::max<long long>(1, (long long)(eval_cost / (2.0 * solve_cost))));
        q.nrs = std::min<long long>(nrs, std::max<long long>(1, KT / 1024));
    }
    q.rows_per_slice = (KT + q.nrs - 1) / q.nrs;
    q.units = (kind == 2 ? N : N * 3) * q.ncb * q.nrs;
    q.grid = std::min<long long>(q.units, (long long)sm_count * 4);
    return VR_OK;
}

// Dataset.pad_frames on the device.  out_dev: the up-sampled batch, and/or coef_dev: only the spline
// (per-interval cubics) for the fused radar kernel.
int pad_launch(const float* x_dev, int64_t N, int64_t T, int32_t V, int32_t M, int32_t num_pad_frames,
               float sigma, float* out_dev, double* coef_dev, void* stream) {
    if (!x_dev || (!out_dev && !coef_dev)) return fail(VR_ERR_ARG, "x_dev and out_dev must not be null");
    int rc = pad_check(N, T, V, M, num_pad_frames, sigma);
    if (rc) return rc;
    int dev, sm_count;
    rc = device_setup(dev, sm_count);
    if (rc) return rc;
    vr::PadParams p;
    memset(&p, 0, sizeof(p));
    PadPlan q;
    rc = pad_plan(0, N, T, V, M, num_pad_frames, sigma, sm_count, q, p.w);
    if (rc) return rc;
    p.radius = q.radius;
    p.x = x_dev; p.out = out_dev; p.coef = coef_dev;
    p.planes = N * 3; p.T = (int)T; p.VM = V * M; p.K = num_pad_frames;
    p.ratio = (double)(T - 1) / (double)((long long)num_pad_frames * T - 1);
    p.nc = (int)q.nc; p.ncb = (int)q.ncb;
    static std::mutex mu;
    static bool attr_done[64] = {false};
    {
        std::lock_guard<std::mutex> lk(mu);
        if (!attr_done[dev]) {
            CUDA_TRY(cudaFuncSetAttribute(vr::vr_pad_frames_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            attr_done[dev] = true;
        }
    }
    const size_t smem = (size_t)q.smem;
    const int grid = (int)q.grid;
    vr::vr_pad_frames_kernel<<<grid, 1024, smem, (cudaStream_t)stream>>>(p);
    CUDA_TRY(cudaGetLastError());
    return VR_OK;
}
}  // namespace
extern "C" {

int vr_pad_frames_f32(const float* x_dev, int64_t N, int64_t T, int32_t V, int32_t M, int32_t num_pad_frames,
                      float sigma, float* out_dev, void* stream) {
    if (!out_dev) return fail(VR_ERR_ARG, "x_dev and out_dev must not be null");
    return pad_launch(x_dev, N, T, V, M, num_pad_frames, sigma, out_dev, nullptr, stream);
}

int vr_pad_frames_backward_f32(const float* grad_out_dev, int64_t N, int64_t T, int32_t V, int32_t M, int32_t num_pad_frames,
                               float sigma, float* grad_x_dev, void* stream) {
    if (!grad_out_dev || !grad_x_dev) return fail(VR_ERR_ARG, "grad_out_dev and grad_x_dev must not be null");
    int rc = pad_check(N, T, V, M, num_pad_frames, sigma);
    if (rc) return rc;
    int dev, sm_count;
    rc = device_setup(dev, sm_count);
    if (rc) return rc;
    vr::PadBwdParams p;
    memset(&p, 0, sizeof(p));
    PadPlan q;
    rc = pad_plan(1, N, T, V, M, num_pad_frames, sigma, sm_count, q, p.w);
    if (rc) return rc;
    p.radius = q.radius;
    {
        double c = 0.0;                                          // the forward's Thomas recurrence, bit for bit
        for (int i = 2; i < vr::PF_CP_N; ++i) { c = 1.0 / (4.0 - c); p.cp[i] = c; }
        if (1.0 / (4.0 - c) != c) return fail(VR_ERR_UNSUPPORTED, "Thomas coefficients did not reach their fixed point");
    }
    p.g = grad_out_dev; p.gx = grad_x_dev;
    p.planes = N * 3; p.T = (int)T; p.VM = V * M; p.K = num_pad_frames;
    p.ratio = (double)(T - 1) / (double)((long long)num_pad_frames * T - 1);
    p.nc = (int)q.nc; p.ncb = (int)q.ncb;
    static std::mutex mu;
    static bool attr_done[64] = {false};
    {
        std::lock_guard<std::mutex> lk(mu);
        if (!attr_done[dev]) {
            CUDA_TRY(cudaFuncSetAttribute(vr::vr_pad_frames_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            attr_done[dev] = true;
        }
    }
    const size_t smem = (size_t)q.smem;
    const int grid = (int)q.grid;
    vr::vr_pad_frames_backward_kernel<<<grid, 1024, smem, (cudaStream_t)stream>>>(p);
    CUDA_TRY(cudaGetLastError());
    return VR_OK;
}

int vr_pad_frames_joints(const void* x_dev, int32_t x_is_f64, int64_t N, int64_t T, int32_t V, int32_t C,
                         int32_t num_pad_frames, float sigma, int32_t planar_out, float* out_dev, void* stream) {
    if (!x_dev || !out_dev) return fail(VR_ERR_ARG, "x_dev and out_dev must not be null");
    int rc = pad_joints_check(N, T, V, C, num_pad_frames, sigma);
    if (rc) return rc;
    int dev, sm_count;
    rc = device_setup(dev, sm_count);
    if (rc) return rc;
    vr::PadNbParams p;
    memset(&p, 0, sizeof(p));
    PadPlan q;
    rc = pad_plan(2, N, T, V, C, num_pad_frames, sigma, sm_count, q, p.w);
    if (rc) return rc;
    p.radius = q.radius;
    p.x = x_dev; p.out = out_dev; p.N = N; p.T = (int)T; p.V = V; p.C = C; p.K = num_pad_frames; p.planar = planar_out ? 1 : 0;
    p.ratio = (double)(T - 1) / (double)((long long)num_pad_frames * T - 1);
    p.nc = (int)q.nc; p.ncb = (int)q.ncb; p.nrs = (int)q.nrs; p.rows_per_slice = q.rows_per_slice;
    static std::mutex mu;
    static bool attr_done[64] = {false};
    {
        std::lock_guard<std::mutex> lk(mu);
        if (!attr_done[dev]) {
            CUDA_TRY(cudaFuncSetAttribute(vr::vr_pad_frames_nb_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            CUDA_TRY(cudaFuncSetAttribute(vr::vr_pad_frames_nb_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            attr_done[dev] = true;
        }
    }
    const size_t smem = (size_t)q.smem;
    const int grid = (int)q.grid;
    if (x_is_f64) vr::vr_pad_frames_nb_kernel<double><<<grid, 1024, smem, (cudaStream_t)stream>>>(p);
    else vr::vr_pad_frames_nb_kernel<float><<<grid, 1024, smem, (cudaStream_t)stream>>>(p);
    CUDA_TRY(cudaGetLastError());
    return VR_OK;
}

int64_t vr_upsampled_workspace_bytes(int64_t N, int64_t T, int32_t V, int32_t M) {
    if (N <= 0 || T < 2 || V <= 0 || M <= 0) return 0;
    return N * (T - 1) * 4 * 3 * (int64_t)V * M * (int64_t)sizeof(double);
}

}  // extern "C"
namespace {
int upsampled_impl(const float* x_dev, int64_t N, int64_t T, int32_t V, int32_t M,
                   const int32_t* src_host, const int32_t* dst_host, int32_t E,
                   const float* wavelength_dev, const float* radar_loc_dev,
                   int32_t n_fft, int32_t hop, uint32_t flags,
                   int32_t num_pad_frames, float sigma, int32_t image_size,
                   void* workspace_dev, int64_t workspace_bytes, float* out_dev, float* iq_dev, void* stream,
                   const vr::NoiseParams& noise) {
    if (!wavelength_dev || !radar_loc_dev) return fail(VR_ERR_ARG, "wavelength_dev and radar_loc_dev must not be null");
    if (!x_dev || (!out_dev && !iq_dev) || !workspace_dev) return fail(VR_ERR_ARG, "x_dev, out_dev and workspace_dev must not be null");
    if (image_size < 0) return fail(VR_ERR_SHAPE, "image_size must be >= 0, got %d", image_size);
    if (N <= 0 || V <= 0 || M <= 0) return fail(VR_ERR_SHAPE, "N, V, M must be positive (got %lld, %d, %d)", (long long)N, V, M);
    if (T < 4) return fail(VR_ERR_SHAPE, "T=%lld: cubic interpolation needs at least 4 frames (scipy interp1d raises ValueError)", (long long)T);
    if (num_pad_frames < 1) return fail(VR_ERR_SHAPE, "num_pad_frames must be >= 1, got %d", num_pad_frames);
    if ((double)T * num_pad_frames > (double)(1ll << 30)) return fail(VR_ERR_UNSUPPORTED, "T*num_pad_frames too large");
    int views;                                            // VR_FLAG_VIEWS: the spline of the N / R raw sequences, once
    int rc = views_of(flags, N, views);
    if (rc) return rc;
    const int64_t Nx = N / views;
    if (workspace_bytes < vr_upsampled_workspace_bytes(Nx, T, V, M))
        return fail(VR_ERR_ARG, "workspace of %lld bytes is smaller than vr_upsampled_workspace_bytes = %lld",
                    (long long)workspace_bytes, (long long)vr_upsampled_workspace_bytes(Nx, T, V, M));
    if (((uintptr_t)workspace_dev & 7) != 0) return fail(VR_ERR_ARG, "workspace_dev must be 8-byte aligned");
    double* coef = static_cast<double*>(workspace_dev);
    rc = pad_launch(x_dev, Nx, T, V, M, num_pad_frames, sigma, nullptr, coef, stream);
    if (rc) return rc;
    return launch(x_dev, N, T * num_pad_frames, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev, 0.f, nullptr,
                  n_fft, hop, flags, image_size, out_dev, iq_dev, (cudaStream_t)stream, coef, (int)T, num_pad_frames, noise);
}
}  // namespace
extern "C" {

int vr_forward_upsampled_f32(const float* x_dev, int64_t N, int64_t T, int32_t V, int32_t M,
                             const int32_t* src_host, const int32_t* dst_host, int32_t E,
                             const float* wavelength_dev, const float* radar_loc_dev,
                             int32_t n_fft, int32_t hop, uint32_t flags,
                             int32_t num_pad_frames, float sigma, int32_t image_size,
                             void* workspace_dev, int64_t workspace_bytes, float* out_dev, void* stream) {
    vr::NoiseParams nz;
    if (int rc = take_noise(flags, nz)) return rc;
    return upsampled_impl(x_dev, N, T, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev, n_fft, hop, flags,
                          num_pad_frames, sigma, image_size, workspace_dev, workspace_bytes, out_dev, nullptr, stream, nz);
}

int vr_forward_upsampled_debug_f32(const float* x_dev, int64_t N, int64_t T, int32_t V, int32_t M,
                                   const int32_t* src_host, const int32_t* dst_host, int32_t E,
                                   const float* wavelength_dev, const float* radar_loc_dev,
                                   int32_t n_fft, int32_t hop, uint32_t flags, int32_t num_pad_frames, float sigma,
                                   void* workspace_dev, int64_t workspace_bytes, float* out_dev, float* iq_dev, void* stream) {
    vr::NoiseParams nz;
    if (int rc = take_noise(flags, nz)) return rc;
    if (!iq_dev) return fail(VR_ERR_ARG, "iq_dev must not be null");
    return upsampled_impl(x_dev, N, T, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev, n_fft, hop, flags,
                          num_pad_frames, sigma, 0, workspace_dev, workspace_bytes, out_dev, iq_dev, stream, nz);
}

int vr_synth_upsampled_f32(const float* x_dev, int64_t N, int64_t T, int32_t V, int32_t M,
                           const int32_t* src_host, const int32_t* dst_host, int32_t E,
                           const float* wavelength_dev, const float* radar_loc_dev, uint32_t flags,
                           int32_t num_pad_frames, float sigma, void* workspace_dev, int64_t workspace_bytes,
                           float* iq_dev, void* stream) {
    vr::NoiseParams nz;
    if (int rc = take_noise(flags, nz)) return rc;
    if (!iq_dev) return fail(VR_ERR_ARG, "iq_dev must not be null");
    return upsampled_impl(x_dev, N, T, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev, vr::NFFT, 1, flags,
                          num_pad_frames, sigma, 0, workspace_dev, workspace_bytes, nullptr, iq_dev, stream, nz);
}

int vr_backward_params_f32(const float* x_dev, const float* iq_dev, const float* grad_out_dev,
                           int64_t N, int64_t T, int32_t V, int32_t M,
                           const int32_t* src_host, const int32_t* dst_host, int32_t E,
                           const float* wavelength_dev, const float* radar_loc_dev,
                           int32_t n_fft, int32_t hop, uint32_t flags,
                           float* gz_work_dev, double* grad_params_dev, void* stream) {
    return vr_backward_f32(x_dev, iq_dev, grad_out_dev, N, T, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev,
                           n_fft, hop, flags, gz_work_dev, grad_params_dev, nullptr, stream);
}

}  // extern "C"
namespace {
// The backward entries' checks of everything but the device pointers, before the device is touched.  T: the steps the
// adjoint runs over (up-sampled length for the _upsampled entries).
int backward_args(int64_t N, int64_t T, int V, int M, const int32_t* src_host, const int32_t* dst_host, int E, int n_fft,
                  int hop, uint32_t flags, bool synth_only) {
    if (flags & ~(VR_FLAG_RANGE_FMA | VR_FLAG_PER_SEQUENCE | VR_FLAG_VIEWS_MASK)) return fail(VR_ERR_ARG, "unknown flags 0x%x", flags);
    int views;
    int rc = views_of(flags, N, views);
    if (rc) return rc;
    if (N <= 0 || T <= 0 || V <= 0 || M <= 0 || hop <= 0) return fail(VR_ERR_SHAPE, "N, T, V, M, hop must be positive");
    if (n_fft != vr::NFFT) return fail(VR_ERR_UNSUPPORTED, "this ABI version implements n_fft=256 only (got %d)", n_fft);
    if (!synth_only && T <= n_fft / 2) return fail(VR_ERR_SHAPE, "T=%lld must exceed n_fft/2=%d", (long long)T, n_fft / 2);
    if (T > (1ll << 30)) return fail(VR_ERR_UNSUPPORTED, "T=%lld too long", (long long)T);
    if (!src_host || !dst_host) return fail(VR_ERR_ARG, "edge arrays must not be null");
    if (E <= 0 || E > vr::NG * vr::MAX_EG) return fail(VR_ERR_UNSUPPORTED, "E=%d outside [1, %d]", E, vr::NG * vr::MAX_EG);
    if (V > 65535) return fail(VR_ERR_UNSUPPORTED, "V=%d too large", V);
    for (int e = 0; e < E; ++e)
        if (src_host[e] < 0 || src_host[e] >= V || dst_host[e] < 0 || dst_host[e] >= V)
            return fail(VR_ERR_SHAPE, "edge %d = (%d,%d) indexes a joint outside [0,%d)", e, src_host[e], dst_host[e], V);
    return VR_OK;
}

// the _upsampled backward entries' checks of the raw length and the factor
int backward_ups_args(int64_t T, int num_pad_frames) {
    if (T < 4) return fail(VR_ERR_SHAPE, "T=%lld: cubic interpolation needs at least 4 frames", (long long)T);
    if (num_pad_frames < 1) return fail(VR_ERR_SHAPE, "num_pad_frames must be >= 1, got %d", num_pad_frames);
    if ((double)T * num_pad_frames > (double)(1ll << 30)) return fail(VR_ERR_UNSUPPORTED, "T*num_pad_frames too large");
    return VR_OK;
}

// The configuration of one backward call: the adjoint STFT (unless the entry is synthesis only), then the synthesis
// adjoint -- the scalar kernels with a slot of the static partials (g_param_partials), or the per-sequence kernel
// vr_synth_adjoint_ps_kernel<ups, views_mode> with the scratch tail of the caller's gradient buffer and the fold.
// backward_impl launches exactly this; vr_plan_backward reports it without a GPU.
constexpr int BWD_SYNTH_SCALAR = 0, BWD_SYNTH_SCALAR_UPS = 1, BWD_SYNTH_PS = 2;
struct BackwardPlan {
    bool stft = false;
    int seg_len = 0, segs = 0, stft_grid = 0;
    long long stft_smem = 0;
    int synth = BWD_SYNTH_SCALAR, views_mode = vr::VIEWS_NONE, views = 1, grid = 0, fold_grid = 0;
    bool ups = false;
    long long units = 0, ps_segs = 0;   // per-sequence: warp units and segments per sequence; scalar: units = steps
    long long gx_floats = 0;            // extent of the dL/dx zero fill (0: not wanted)
};
int plan_backward(int64_t N, int64_t T, int V, int M, const int32_t* src_host, const int32_t* dst_host, int E, int n_fft,
                  int hop, uint32_t flags, bool synth_only, bool ups, bool want_gx, int sm_count, BackwardPlan& B) {
    int rc = backward_args(N, T, V, M, src_host, dst_host, E, n_fft, hop, flags, synth_only);
    if (rc) return rc;
    if (ups && want_gx) return fail(VR_ERR_ARG, "the _upsampled backward entries take no dL/dx");
    B = BackwardPlan{};
    views_of(flags, N, B.views);
    B.ups = ups;
    B.gx_floats = want_gx ? (N / B.views) * 3 * T * V * M : 0;
    B.stft = !synth_only;
    if (B.stft) {
        vr::adjoint_plan(N, T, sm_count, B.seg_len, B.segs);
        B.stft_grid = (int)std::min<long long>(N * B.segs, (long long)sm_count * 8);
        B.stft_smem = (long long)B.seg_len * 8;
    }
    if (flags & VR_FLAG_PER_SEQUENCE) {
        // views: with dL/dx one warp runs a row's views in order (one owner per dL/dx row); without it the units are per
        // output, as without views, for R times the parallelism.  R = 1: the plain per-sequence kernel
        B.synth = BWD_SYNTH_PS;
        B.views_mode = B.views == 1 ? vr::VIEWS_NONE : want_gx ? vr::VIEWS_ROWS : vr::VIEWS_OUTPUTS;
        B.ps_segs = vr::ps_segments(T);
        B.units = (B.views_mode == vr::VIEWS_ROWS ? N / B.views : N) * B.ps_segs;
        B.grid = (int)std::min<long long>((B.units + 3) / 4, (long long)sm_count * 16);   // 4 warps per block
        B.fold_grid = (int)((4 * N + 127) / 128);
        return VR_OK;
    }
    B.synth = ups ? BWD_SYNTH_SCALAR_UPS : BWD_SYNTH_SCALAR;
    B.units = N * T;
    B.grid = (int)std::min<long long>(std::min<long long>((B.units + 127) / 128, (long long)sm_count * 16), vr::PARAM_MAX_BLOCKS);
    return VR_OK;
}

int backward_impl(const float* x_dev, const float* iq_dev, const float* grad_out_dev,
                  int64_t N, int64_t T, int32_t V, int32_t M,
                  const int32_t* src_host, const int32_t* dst_host, int32_t E,
                  const float* wavelength_dev, const float* radar_loc_dev,
                  int32_t n_fft, int32_t hop, uint32_t flags, bool synth_only,
                  float* gz_work_dev, double* grad_params_dev, float* grad_x_dev, void* stream,
                  const double* coef = nullptr, int ups_T = 0, int ups_K = 0);
// backward_impl with the joint positions of the up-sampling spline whose cubics vr_forward_upsampled_debug_f32 /
// vr_synth_upsampled_f32 left in workspace_dev; T is the RAW length
int backward_ups_impl(const void* workspace_dev, const float* iq_dev, const float* grad_out_dev,
                      int64_t N, int64_t T, int32_t V, int32_t M, const int32_t* src_host, const int32_t* dst_host, int32_t E,
                      const float* wavelength_dev, const float* radar_loc_dev, int32_t n_fft, int32_t hop, uint32_t flags,
                      int32_t num_pad_frames, bool synth_only, float* gz_work_dev, double* grad_params_dev, void* stream) {
    drop_noise(flags);
    if (!workspace_dev) return fail(VR_ERR_ARG, "workspace_dev must not be null");
    if (((uintptr_t)workspace_dev & 7) != 0) return fail(VR_ERR_ARG, "workspace_dev must be 8-byte aligned");
    if (int rc = backward_ups_args(T, num_pad_frames)) return rc;
    return backward_impl(nullptr, iq_dev, grad_out_dev, N, T * num_pad_frames, V, M, src_host, dst_host, E, wavelength_dev,
                         radar_loc_dev, n_fft, hop, flags, synth_only, gz_work_dev, grad_params_dev, nullptr, stream,
                         static_cast<const double*>(workspace_dev), (int)T, num_pad_frames);
}
}  // namespace
extern "C" {

int vr_synth_adjoint_f32(const float* x_dev, const float* grad_iq_dev, int64_t N, int64_t T, int32_t V, int32_t M,
                         const int32_t* src_host, const int32_t* dst_host, int32_t E,
                         const float* wavelength_dev, const float* radar_loc_dev, uint32_t flags,
                         double* grad_params_dev, float* grad_x_dev, void* stream) {
    // the second stage of vr_backward_f32 alone: dL/d(iq) comes from the caller (a general STFT differentiated by autograd)
    return backward_impl(x_dev, nullptr, nullptr, N, T, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev,
                         vr::NFFT, 16, flags, true, const_cast<float*>(grad_iq_dev), grad_params_dev, grad_x_dev, stream);
}

int vr_backward_f32(const float* x_dev, const float* iq_dev, const float* grad_out_dev,
                    int64_t N, int64_t T, int32_t V, int32_t M,
                    const int32_t* src_host, const int32_t* dst_host, int32_t E,
                    const float* wavelength_dev, const float* radar_loc_dev,
                    int32_t n_fft, int32_t hop, uint32_t flags,
                    float* gz_work_dev, double* grad_params_dev, float* grad_x_dev, void* stream) {
    return backward_impl(x_dev, iq_dev, grad_out_dev, N, T, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev,
                         n_fft, hop, flags, false, gz_work_dev, grad_params_dev, grad_x_dev, stream);
}

int vr_backward_upsampled_params_f32(const void* workspace_dev, const float* iq_dev, const float* grad_out_dev,
                                     int64_t N, int64_t T, int32_t V, int32_t M,
                                     const int32_t* src_host, const int32_t* dst_host, int32_t E,
                                     const float* wavelength_dev, const float* radar_loc_dev,
                                     int32_t n_fft, int32_t hop, uint32_t flags, int32_t num_pad_frames,
                                     float* gz_work_dev, double* grad_params_dev, void* stream) {
    return backward_ups_impl(workspace_dev, iq_dev, grad_out_dev, N, T, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev,
                             n_fft, hop, flags, num_pad_frames, false, gz_work_dev, grad_params_dev, stream);
}

}  // extern "C"
namespace {
int backward_impl(const float* x_dev, const float* iq_dev, const float* grad_out_dev,
                  int64_t N, int64_t T, int32_t V, int32_t M,
                  const int32_t* src_host, const int32_t* dst_host, int32_t E,
                  const float* wavelength_dev, const float* radar_loc_dev,
                  int32_t n_fft, int32_t hop, uint32_t flags, bool synth_only,
                  float* gz_work_dev, double* grad_params_dev, float* grad_x_dev, void* stream,
                  const double* coef, int ups_T, int ups_K) {
    drop_noise(flags);                                   // VR_FLAG_NOISE is rejected below as an unknown flag
    // synth_only: gz_work_dev already holds dL/d(iq); the adjoint STFT is skipped.  coef != nullptr: the joint positions are
    // the up-sampling spline's (T = ups_K * ups_T steps, x_dev unused), parameter gradients only
    if ((!x_dev && !coef) || !gz_work_dev || !grad_params_dev || !wavelength_dev || !radar_loc_dev || (!synth_only && (!iq_dev || !grad_out_dev)))
        return fail(VR_ERR_ARG, "device pointers must not be null");
    int rc = backward_args(N, T, V, M, src_host, dst_host, E, n_fft, hop, flags, synth_only);
    if (rc) return rc;
    if ((flags & VR_FLAG_PER_SEQUENCE) && ((uintptr_t)grad_params_dev & 7) != 0)
        return fail(VR_ERR_ARG, "grad_params_dev must be 8-byte aligned (float64 per-sequence gradients)");
    int dev, sm_count;
    rc = device_setup(dev, sm_count);
    if (rc) return rc;
    BackwardPlan B;
    rc = plan_backward(N, T, V, M, src_host, dst_host, E, n_fft, hop, flags, synth_only, coef != nullptr, grad_x_dev != nullptr,
                       sm_count, B);
    if (rc) return rc;
    vr::BwdParams p;
    memset(&p, 0, sizeof(p));
    for (int e = 0; e < E; ++e) { p.src[e] = (uint16_t)src_host[e]; p.dst[e] = (uint16_t)dst_host[e]; }
    p.x = x_dev; p.iq = iq_dev; p.gout = grad_out_dev; p.gz = gz_work_dev; p.gparams = grad_params_dev; p.gx = grad_x_dev;
    p.lam_ptr = wavelength_dev; p.loc_ptr = radar_loc_dev;
    p.N = N; p.T = T; p.V = V; p.M = M; p.E = E; p.hop = hop; p.VM = V * M;
    p.F = (int)(T / hop) + 1;
    p.fma_range = (flags & VR_FLAG_RANGE_FMA) ? 1 : 0;
    p.inv_E = 1.0f / (float)E;
    p.coef = coef; p.ups_T = ups_T;
    p.ups_ratio = coef ? (double)(ups_T - 1) / (double)((long long)ups_K * ups_T - 1) : 0.0;
    p.views = B.views;
    p.seg_len = B.seg_len; p.segs = B.segs;
    cudaStream_t st = (cudaStream_t)stream;
    if (grad_x_dev) CUDA_TRY(cudaMemsetAsync(grad_x_dev, 0, (size_t)B.gx_floats * sizeof(float), st));
    if (B.stft) {                                       // writes every sample of gz: no zero fill
        vr::vr_stft_adjoint_kernel<<<B.stft_grid, vr::BWD_WARPS * 32, (size_t)B.stft_smem, st>>>(p);
        CUDA_TRY(cudaGetLastError());
    }
    if (B.synth == BWD_SYNTH_PS) {
        // per-sequence gradients: (x sequence, segment) units, each running its views, reduced warp by warp into the scratch
        // tail of grad_params_dev (vr_per_sequence_grad_doubles), then folded per output in segment order
        p.ps_segs = B.ps_segs;
        p.part = grad_params_dev + 4 * N;
        if (B.views_mode == vr::VIEWS_ROWS) {
            if (coef) vr::vr_synth_adjoint_ps_kernel<true, vr::VIEWS_ROWS><<<B.grid, 128, 0, st>>>(p);
            else vr::vr_synth_adjoint_ps_kernel<false, vr::VIEWS_ROWS><<<B.grid, 128, 0, st>>>(p);
        } else if (B.views_mode == vr::VIEWS_OUTPUTS) {
            if (coef) vr::vr_synth_adjoint_ps_kernel<true, vr::VIEWS_OUTPUTS><<<B.grid, 128, 0, st>>>(p);
            else vr::vr_synth_adjoint_ps_kernel<false, vr::VIEWS_OUTPUTS><<<B.grid, 128, 0, st>>>(p);
        } else {
            if (coef) vr::vr_synth_adjoint_ps_kernel<true, vr::VIEWS_NONE><<<B.grid, 128, 0, st>>>(p);
            else vr::vr_synth_adjoint_ps_kernel<false, vr::VIEWS_NONE><<<B.grid, 128, 0, st>>>(p);
        }
        CUDA_TRY(cudaGetLastError());
        vr::vr_param_fold_kernel<<<(unsigned)B.fold_grid, 128, 0, st>>>(p.part, grad_params_dev, N, p.ps_segs);
        CUDA_TRY(cudaGetLastError());
        return VR_OK;
    }
    next_param_slot(dev, p);
    if (B.synth == BWD_SYNTH_SCALAR_UPS) vr::vr_synth_adjoint_ups_kernel<<<B.grid, 128, 0, st>>>(p);
    else vr::vr_synth_adjoint_kernel<<<B.grid, 128, 0, st>>>(p);
    CUDA_TRY(cudaGetLastError());
    return VR_OK;
}
}  // namespace
extern "C" {

int vr_synth_adjoint_upsampled_f32(const void* workspace_dev, const float* grad_iq_dev,
                                   int64_t N, int64_t T, int32_t V, int32_t M,
                                   const int32_t* src_host, const int32_t* dst_host, int32_t E,
                                   const float* wavelength_dev, const float* radar_loc_dev, uint32_t flags,
                                   int32_t num_pad_frames, double* grad_params_dev, void* stream) {
    // the second stage of vr_backward_upsampled_params_f32 alone: dL/d(iq) comes from the caller (a general STFT)
    return backward_ups_impl(workspace_dev, nullptr, nullptr, N, T, V, M, src_host, dst_host, E, wavelength_dev, radar_loc_dev,
                             vr::NFFT, 16, flags, num_pad_frames, true, const_cast<float*>(grad_iq_dev), grad_params_dev, stream);
}

int64_t vr_per_sequence_grad_doubles(int64_t N, int64_t T) {
    if (N <= 0 || T <= 0) return 0;
    return 4 * N + 4 * N * vr::ps_segments(T);
}

int vr_release_host_staging(void) {
    int cur = 0;
    cudaGetDevice(&cur);
    for (int d = 0; d < 64; ++d) {
        std::lock_guard<std::mutex> lk(g_stage_mu[d]);
        Staging& sg = g_stage[d];
        if (!sg.st[0] && !sg.x[0]) continue;
        cudaSetDevice(d);
        for (int i = 0; i < 2; ++i) {
            if (sg.x[i]) cudaFree(sg.x[i]);
            if (sg.o[i]) cudaFree(sg.o[i]);
            if (sg.st[i]) cudaStreamDestroy(sg.st[i]);
            sg.x[i] = sg.o[i] = nullptr; sg.st[i] = nullptr;
        }
        sg.xcap = sg.ocap = 0;
    }
    cudaSetDevice(cur);
    return VR_OK;
}

int vr_set_timeline_buffer(void* dev_u64_8_per_cta) {
    g_timeline = static_cast<unsigned long long*>(dev_u64_8_per_cta);
    return VR_OK;
}

int vr_plan(int64_t N, int64_t T, int32_t V, int32_t M, const int32_t* src_host, const int32_t* dst_host,
            int32_t E, int32_t n_fft, int32_t hop, int32_t sm_count, int64_t plan[16]) {
    if (!plan) return fail(VR_ERR_ARG, "plan must not be null");
    vr::Params p;
    int grid, cps;
    int rc = make_plan(N, T, V, M, src_host, dst_host, E, n_fft, hop, 0, false, sm_count > 0 ? sm_count : 148, true, p, grid, cps);
    if (rc) return rc;
    plan[0] = grid; plan[1] = (p.W + 1) * 32; plan[2] = p.smem_bytes; plan[3] = p.S; plan[4] = p.FJ;
    plan[5] = p.jobs_per_seq; plan[6] = p.FB; plan[7] = p.tma_in; plan[8] = p.bulk_out; plan[9] = p.cmax;
    plan[10] = p.eg_max; plan[11] = p.sg_max; plan[12] = p.zcap; plan[13] = cps; plan[14] = vr::TL; plan[15] = vr::NG;
    return VR_OK;
}

int vr_plan_team(int64_t N, int64_t T, int32_t V, int32_t M, const int32_t* src_host, const int32_t* dst_host,
                 int32_t E, int32_t n_fft, int32_t hop, int32_t sm_count, int64_t plan[8]) {
    if (!plan) return fail(VR_ERR_ARG, "plan must not be null");
    vr::Params p;
    int grid, cps;
    const int sms = sm_count > 0 ? sm_count : 148;
    int rc = make_plan(N, T, V, M, src_host, dst_host, E, n_fft, hop, 0, false, sms, true, p, grid, cps);
    if (rc) return rc;
    if (!make_team_plan(p, sms, grid))
        return fail(VR_ERR_UNSUPPORTED, "the team-job schedule does not apply to this shape (needs one job per sequence, a bulk-stored tile, TMA-loadable chunks and room for two CTAs per SM)");
    plan[0] = grid; plan[1] = vr::TJ_THREADS; plan[2] = p.smem_bytes; plan[3] = vr::TJ_RS; plan[4] = vr::TJ_TEAMS;
    plan[5] = p.stage_bytes; plan[6] = p.z_stride;
    plan[7] = (p.n_jobs >= (long long)TEAM_AUTO_WAVES * sms * 2 * vr::TJ_TEAMS) ? 1 : 0;
    return VR_OK;
}

int vr_plan_launch(int32_t mode, int64_t N, int64_t T, int32_t V, int32_t M, const int32_t* src_host, const int32_t* dst_host,
                   int32_t E, int32_t n_fft, int32_t hop, int32_t image_size, int32_t num_pad_frames, uint32_t flags,
                   int32_t x_aligned, int32_t schedule, int32_t sm_count, int64_t plan[24]) {
    if (!plan) return fail(VR_ERR_ARG, "plan must not be null");
    if (mode < 0 || mode > 2) return fail(VR_ERR_ARG, "mode must be 0 (spectrogram), 1 (debug: iq too) or 2 (synthesis only), got %d", mode);
    if (schedule < -1 || schedule > 1) return fail(VR_ERR_ARG, "schedule must be -1, 0 or 1, got %d", schedule);
    if (num_pad_frames < 0) return fail(VR_ERR_SHAPE, "num_pad_frames must be >= 0, got %d", num_pad_frames);
    if (mode != 0 && image_size != 0) return fail(VR_ERR_ARG, "the debug and synthesis-only entries take no image_size");
    const bool ups = num_pad_frames > 0;
    LaunchPlan L;
    int rc = plan_launch(N, ups ? T * num_pad_frames : T, V, M, src_host, dst_host, E, n_fft, hop, image_size, ups, mode == 2,
                         mode == 1, flags, x_aligned != 0, schedule, sm_count > 0 ? sm_count : 148, false, L);
    if (rc) return rc;
    const vr::Params& p = L.p;
    plan[0] = L.team; plan[1] = L.grid; plan[2] = L.team ? vr::TJ_THREADS : (p.W + 1) * 32; plan[3] = p.smem_bytes;
    plan[4] = p.S; plan[5] = p.FJ; plan[6] = p.jobs_per_seq; plan[7] = p.n_jobs; plan[8] = p.FB; plan[9] = p.ostride;
    plan[10] = p.tma_in; plan[11] = p.bulk_out; plan[12] = p.cmax; plan[13] = p.zcap; plan[14] = p.zpark; plan[15] = p.sparse;
    plan[16] = p.ncols; plan[17] = L.cps; plan[18] = L.ticket; plan[19] = (p.M % 2 == 0) ? 2 : 1; plan[20] = L.vmc;
    plan[21] = p.eg_max; plan[22] = p.sg_max; plan[23] = mode == 1 && iq_gaps(p);
    return VR_OK;
}

int vr_selftest_rounding(uint64_t n, float wavelength, uint64_t mismatches[3]) {
    if (!mismatches) return fail(VR_ERR_ARG, "mismatches must not be null");
    unsigned long long* d = nullptr;
    CUDA_TRY(cudaMalloc(&d, 3 * sizeof(unsigned long long)));
    CUDA_TRY(cudaMemset(d, 0, 3 * sizeof(unsigned long long)));
    vr::vr_selftest_kernel<<<1184, 256>>>(n, wavelength, d);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    unsigned long long h[3] = {0, 0, 0};
    if (e == cudaSuccess) e = cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(VR_ERR_CUDA, "selftest: %s", cudaGetErrorString(e));
    for (int i = 0; i < 3; ++i) mismatches[i] = h[i];
    return VR_OK;
}

int vr_plan_adjoint_stft(int64_t N, int64_t T, int32_t hop, int32_t sm_count, int64_t plan[4], int64_t* segments,
                         int64_t max_segments) {
    if (!plan) return fail(VR_ERR_ARG, "plan must not be null");
    if (N <= 0 || hop <= 0) return fail(VR_ERR_SHAPE, "N, hop must be positive");
    if (T <= vr::NFFT / 2) return fail(VR_ERR_SHAPE, "T=%lld must exceed n_fft/2=%d", (long long)T, vr::NFFT / 2);
    if (T > (1ll << 30)) return fail(VR_ERR_UNSUPPORTED, "T=%lld too long", (long long)T);
    const int sms = sm_count > 0 ? sm_count : 148;
    int seg_len, segs;
    vr::adjoint_plan(N, T, sms, seg_len, segs);
    plan[0] = seg_len; plan[1] = segs; plan[2] = std::min<long long>(N * segs, (long long)sms * 8); plan[3] = (int64_t)seg_len * 8;
    if (segments) {
        if (max_segments < segs) return fail(VR_ERR_ARG, "segments holds %lld rows, the plan has %d", (long long)max_segments, segs);
        const int F = (int)(T / hop) + 1;
        for (int k = 0; k < segs; ++k) {
            const long long s0 = (long long)k * seg_len, s1 = std::min<long long>(T, s0 + seg_len);
            int lo, hi;
            vr::adj_seg_frames(s0, s1, T, F, hop, lo, hi);
            int64_t* r = segments + 4 * k;
            r[0] = s0; r[1] = s1; r[2] = lo; r[3] = hi;
        }
    }
    return VR_OK;
}

int vr_plan_backward(int32_t entry, int64_t N, int64_t T, int32_t V, int32_t M, const int32_t* src_host,
                     const int32_t* dst_host, int32_t E, int32_t n_fft, int32_t hop, uint32_t flags, int32_t want_grad_x,
                     int32_t num_pad_frames, int32_t sm_count, int64_t plan[16]) {
    if (!plan) return fail(VR_ERR_ARG, "plan must not be null");
    if (entry < 0 || entry > 4)
        return fail(VR_ERR_ARG, "entry must be 0 (backward), 1 (backward_params), 2 (synth_adjoint), 3 (backward_upsampled_params) "
                                "or 4 (synth_adjoint_upsampled), got %d", entry);
    drop_noise(flags);
    const bool ups = entry >= 3, synth_only = entry == 2 || entry == 4;
    if (want_grad_x && entry != 0 && entry != 2) return fail(VR_ERR_ARG, "only vr_backward_f32 and vr_synth_adjoint_f32 take dL/dx");
    if (ups) {
        if (int rc = backward_ups_args(T, num_pad_frames)) return rc;
        T *= num_pad_frames;
    }
    if (synth_only) { n_fft = vr::NFFT; hop = 16; }        // what the synthesis-only entries pass: they run no STFT
    BackwardPlan B;
    int rc = plan_backward(N, T, V, M, src_host, dst_host, E, n_fft, hop, flags, synth_only, ups, want_grad_x != 0,
                           sm_count > 0 ? sm_count : 148, B);
    if (rc) return rc;
    const bool ps = B.synth == BWD_SYNTH_PS;
    plan[0] = B.stft; plan[1] = B.seg_len; plan[2] = B.segs; plan[3] = B.stft_grid; plan[4] = B.stft_smem; plan[5] = B.synth;
    plan[6] = B.ups; plan[7] = B.views_mode; plan[8] = B.views; plan[9] = B.grid; plan[10] = B.units; plan[11] = B.ps_segs;
    plan[12] = B.fold_grid; plan[13] = ps ? 1 : 0; plan[14] = B.gx_floats; plan[15] = ps ? 0 : vr::PARAM_MAX_BLOCKS;
    return VR_OK;
}

int vr_plan_pad_frames(int32_t kind, int64_t N, int64_t T, int32_t V, int32_t M_or_C, int32_t num_pad_frames, float sigma,
                       int32_t sm_count, int64_t plan[8]) {
    if (!plan) return fail(VR_ERR_ARG, "plan must not be null");
    PadPlan q;
    int rc = pad_plan(kind, N, T, V, M_or_C, num_pad_frames, sigma, sm_count > 0 ? sm_count : 148, q, nullptr);
    if (rc) return rc;
    plan[0] = q.nc; plan[1] = q.ncb; plan[2] = q.units; plan[3] = q.grid; plan[4] = q.smem; plan[5] = q.nrs;
    plan[6] = q.rows_per_slice; plan[7] = q.radius;
    return VR_OK;
}

int vr_partition_edges(const int32_t* src_host, const int32_t* dst_host, int32_t E, int32_t V, int32_t* group_of_edge) {
    if (!group_of_edge) return fail(VR_ERR_ARG, "group_of_edge must not be null");
    Partition P;
    int rc = partition_edges(src_host, dst_host, E, V, P);
    if (rc) return rc;
    for (int e = 0; e < E; ++e) group_of_edge[e] = P.group_of_edge[e];
    return VR_OK;
}

}  // extern "C"

// ---- the STFT against general kernels: tcgen05 GEMM (vr_stft_gemm.cuh) --------------------------------------------
namespace {
int gemm_setup(int dev) {
    static std::mutex mu;
    static bool done[64] = {false};
    std::lock_guard<std::mutex> lk(mu);
    if (!done[dev]) {
        CUDA_TRY(cudaFuncSetAttribute(vr::vr_gemm_tf32x3_kernel<1, vr::G_FRAME_ROWS, vr::G_TILED>, cudaFuncAttributeMaxDynamicSharedMemorySize, vr::G_SMEM_BYTES));
        CUDA_TRY(cudaFuncSetAttribute(vr::vr_gemm_tf32x3_kernel<0, vr::G_STRIDED, vr::G_TILED>, cudaFuncAttributeMaxDynamicSharedMemorySize, vr::G_SMEM_BYTES));
        CUDA_TRY(cudaFuncSetAttribute(vr::vr_gemm_tf32x3_kernel<0, vr::G_STRIDED, vr::G_FRAME_COLS>, cudaFuncAttributeMaxDynamicSharedMemorySize, vr::G_SMEM_BYTES));
        done[dev] = true;
    }
    return VR_OK;
}
bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }      // nullptr counts as aligned
int stft_nb(int n_fft) { return n_fft < vr::GN / 2 ? n_fft : vr::GN / 2; }    // bins per column tile: [re block | im block]
int stft_check(int64_t N, int64_t T, int n_fft, int hop) {
    if (N <= 0 || T <= 0 || hop <= 0) return fail(VR_ERR_SHAPE, "N, T, hop must be positive");
    if (n_fft < 16 || n_fft > 1024 || (n_fft & (n_fft - 1)) != 0) return fail(VR_ERR_UNSUPPORTED, "n_fft must be a power of two in [16, 1024], got %d", n_fft);
    if (T <= n_fft / 2) return fail(VR_ERR_SHAPE, "T=%lld must exceed n_fft/2=%d: reflect padding needs it", (long long)T, n_fft / 2);
    if (N * (T / hop + 1) >= (1ll << 31) / 2) return fail(VR_ERR_UNSUPPORTED, "too many frames for one launch; split the batch");
    return VR_OK;
}
}  // namespace

extern "C" {

static long long stft_ldm(long long M) { return (M + 3) & ~3ll; }
// floats of one tiled hi / lo image of the (2 n_fft)^2 kernel matrix (vr_stft_gemm.cuh, G_TILED)
static long long stft_bimg_floats(int n_fft) {
    const long long K = 2ll * n_fft;
    return ((K + vr::GN - 1) / vr::GN) * ((K + vr::GK - 1) / vr::GK) * (long long)vr::G_BIMG_FLOATS;
}
static long long stft_lp(long long T, int n_fft) { return (T + n_fft + 3) & ~3ll; }     // padded signal length, 16-byte rows

}  // extern "C"
namespace {
// The launch configuration of the general-kernel STFT's GEMMs (vr_plan_stft_general; the launches below take every number
// from it).  P (S, 2, Lp) is the planar signal the frame views read: the reflect-padded signal (hop, F = T / hop + 1) on the
// full route, the compact copy of the kept frames (hop' = n_fft, F = F_kept) on the kept-frames route.
struct StftPlan {
    int nb, F, K, hop_view;                          // bins per column tile; frames per sequence; K = 2 n_fft; hop of the view
    long long M, ldm, Lp;                            // GEMM rows (sequence, frame); leading dimension of C / dC; plane length
    int row_tiles, col_tiles, kblocks;               // forward and dA GEMMs: M x K output, K = 2 n_fft reduction
    int dbt_tiles, splits, kb_per_split, kb_last;    // kernel-gradient GEMM: K x K output, reduction over the M frames
};
int stft_plan(int64_t N, int64_t T, int n_fft, int hop, int64_t F_kept, int sm_count, StftPlan& q) {
    int rc = stft_check(N, T, n_fft, hop);
    if (rc) return rc;
    if (F_kept < 0 || F_kept > T / hop + 1) return fail(VR_ERR_SHAPE, "F_kept=%lld outside [0, T/hop+1 = %lld] (0: all frames)", (long long)F_kept, (long long)(T / hop + 1));
    q.nb = stft_nb(n_fft);
    q.K = 2 * n_fft;
    q.F = F_kept ? (int)F_kept : (int)(T / hop) + 1;
    q.hop_view = F_kept ? n_fft : hop;
    q.M = N * (long long)q.F;
    q.ldm = stft_ldm(q.M);
    q.Lp = F_kept ? F_kept * (long long)n_fft : stft_lp(T, n_fft);
    q.row_tiles = (int)((q.M + vr::GM - 1) / vr::GM);
    q.col_tiles = (q.K + vr::GN - 1) / vr::GN;
    q.kblocks = (q.K + vr::GK - 1) / vr::GK;
    // the kernel gradient's reduction runs over all frames of the batch: split it over gridDim.z so that the (2 n_fft / 128)^2
    // output tiles fill the machine.  One CTA per SM at a time (192 KB of stages): whole waves, i.e. splits * tiles <= a
    // multiple of sm_count; one wave unless that leaves a slice fewer than 8 K blocks; and no more planes than a pool slot holds
    q.dbt_tiles = ((q.K + vr::GM - 1) / vr::GM) * ((q.K + vr::GN - 1) / vr::GN);
    const int kb_all = (int)((q.M + vr::GK - 1) / vr::GK);
    const int splits = std::max(1, std::min(std::min(sm_count, vr::G_SPLIT_CTAS_MAX) / q.dbt_tiles, (kb_all + 7) / 8));
    q.kb_per_split = (kb_all + splits - 1) / splits;
    q.splits = (kb_all + q.kb_per_split - 1) / q.kb_per_split;
    q.kb_last = kb_all - (q.splits - 1) * q.kb_per_split;
    return VR_OK;
}

// The GEMM part of the forward, over the planar signal P of the plan.  Each output column is one GEMM row with the same K
// order and B tiles on both routes.
int stft_forward_gemm(const StftPlan& q, const float* P, int n_fft, const float* wsin_dev, const float* wcos_dev,
                      float* bt_work, float* c_save, float* out_dev, cudaStream_t st) {
    const int K = q.K;
    const long long img = stft_bimg_floats(n_fft);
    if (K % vr::GN) CUDA_TRY(cudaMemsetAsync(bt_work, 0, (size_t)(2 * img) * sizeof(float), st));      // rows past K of the one tile
    vr::vr_stft_bt_kernel<<<(n_fft * n_fft + 255) / 256, 256, 0, st>>>(wsin_dev, wcos_dev, bt_work, bt_work + img, n_fft, q.nb, q.kblocks);
    vr::GemmParams g;
    memset(&g, 0, sizeof(g));
    g.P = P; g.Lp = q.Lp; g.hop = q.hop_view;        // A = the frames, read as views of the padded signal
    g.Bimg = bt_work;                                // B = the kernel matrix, pre-split and pre-tiled: bulk copies
    g.M = (int)q.M; g.N = K; g.K = K; g.kb_per_split = q.kblocks;
    g.out = out_dev; g.csave = c_save; g.ldc = q.ldm; g.F = q.F; g.n_fft = n_fft; g.nb = q.nb;
    dim3 grid((unsigned)((long long)q.row_tiles * q.col_tiles));
    vr::vr_gemm_tf32x3_kernel<1, vr::G_FRAME_ROWS, vr::G_TILED><<<grid, vr::G_THREADS, vr::G_SMEM_BYTES, st>>>(g);
    CUDA_TRY(cudaGetLastError());
    return VR_OK;
}

// The GEMM part of the backward over the same plan: dC, then dA (frame gradients, folded by the caller) and dBt (kernel
// gradients, reduced over every frame of the batch)
int stft_backward_gemm(const StftPlan& q, const float* grad_out_dev, const float* P, int n_fft,
                       const float* bt_work, const float* c_save, float* dc_work, float* da_work, float* dbt_work,
                       float* grad_wsin_dev, float* grad_wcos_dev, int dev, int sm_count, cudaStream_t st) {
    const int K = q.K;
    const long long M = q.M, ldm = q.ldm;
    vr::vr_stft_dc_kernel<<<dim3((unsigned)std::min<long long>((M / 4 + 256) / 256, sm_count * 4ll), (unsigned)n_fft), 256, 0, st>>>(grad_out_dev, c_save, dc_work, (int)M, ldm, q.F, n_fft, q.nb);
    vr::GemmParams g;
    if (da_work) {                                   // dA[m, k] = sum_n dC[m, n] Bt[n, k]
        memset(&g, 0, sizeof(g));
        g.A = dc_work; g.sAm = 1; g.sAk = ldm;       // dC is column-major: dC(m, n) = dc[n * ldm + m]
        g.Bimg = bt_work + stft_bimg_floats(n_fft);  // B'(n' = k, k' = n) = Bt[n][k]: the transposed image
        g.M = (int)M; g.N = K; g.K = K; g.C = da_work; g.ldc = K; g.kb_per_split = q.kblocks;
        dim3 grid((unsigned)((long long)q.row_tiles * q.col_tiles));
        vr::vr_gemm_tf32x3_kernel<0, vr::G_STRIDED, vr::G_TILED><<<grid, vr::G_THREADS, vr::G_SMEM_BYTES, st>>>(g);
    }
    if (dbt_work) {                                  // dBt[n, k] = sum_m dC[m, n] A[m, k]
        memset(&g, 0, sizeof(g));
        g.A = dc_work; g.sAm = ldm; g.sAk = 1;       // A'(m' = n, k' = m) = dC(m, n) = dc[n * ldm + m]: rows of 16-byte aligned chunks
        g.P = P; g.Lp = q.Lp; g.hop = q.hop_view; g.F = q.F; g.n_fft = n_fft;     // B'(n' = k, k' = m) = A[m][k], a view
        g.M = K; g.N = K; g.K = (int)M; g.C = dbt_work; g.ldc = K;
        // each slice writes its own K x K plane of a split-K pool slot, added in slice order below
        g.kb_per_split = q.kb_per_split;
        if (q.splits > 1) { g.C = next_splitk_slot(dev); g.c_split = (long long)K * K; }
        dim3 grid((unsigned)q.dbt_tiles, 1u, (unsigned)q.splits);
        vr::vr_gemm_tf32x3_kernel<0, vr::G_STRIDED, vr::G_FRAME_COLS><<<grid, vr::G_THREADS, vr::G_SMEM_BYTES, st>>>(g);
        vr::vr_stft_dw_kernel<<<(n_fft * n_fft + 255) / 256, 256, 0, st>>>(g.C, q.splits, g.c_split, grad_wsin_dev, grad_wcos_dev, n_fft, q.nb);
    }
    CUDA_TRY(cudaGetLastError());
    return VR_OK;
}

// the argument checks of both forward entries (F: frames of the GEMM, T / hop + 1 or F_kept)
int stft_forward_args(const float* iq_dev, const float* wsin_dev, const float* wcos_dev, const float* frames_work,
                      const float* bt_work, const float* c_save, const float* out_dev, int64_t N, int64_t T, int n_fft, int hop,
                      int& dev, int& sm_count) {
    if (!iq_dev || !wsin_dev || !wcos_dev || !frames_work || !bt_work || !out_dev) return fail(VR_ERR_ARG, "device pointers must not be null");
    if (!aligned16(bt_work) || !aligned16(c_save) || (reinterpret_cast<uintptr_t>(iq_dev) & 7))     // bulk copies, 16-byte column accesses, float2 samples
        return fail(VR_ERR_ARG, "bt_work and c_save must be 16-byte aligned, iq_dev 8-byte aligned");
    int rc = stft_check(N, T, n_fft, hop);
    if (rc) return rc;
    rc = device_setup(dev, sm_count);
    if (rc) return rc;
    return gemm_setup(dev);
}

// the argument checks of both backward entries
int stft_backward_args(const float* grad_out_dev, const float* frames_work, const float* bt_work, const float* c_save,
                       const float* dc_work, const float* da_work, const float* dbt_work, const float* grad_iq_dev,
                       const float* grad_wsin_dev, const float* grad_wcos_dev, int64_t N, int64_t T, int n_fft, int hop,
                       int& dev, int& sm_count) {
    if (!grad_out_dev || !frames_work || !bt_work || !c_save || !dc_work) return fail(VR_ERR_ARG, "device pointers must not be null");
    if (!aligned16(bt_work) || !aligned16(c_save) || !aligned16(dc_work) || (reinterpret_cast<uintptr_t>(grad_iq_dev) & 7))
        return fail(VR_ERR_ARG, "bt_work, c_save and dc_work must be 16-byte aligned, grad_iq_dev 8-byte aligned");
    if ((da_work == nullptr) != (grad_iq_dev == nullptr)) return fail(VR_ERR_ARG, "da_work and grad_iq_dev go together");
    if ((dbt_work == nullptr) != (grad_wsin_dev == nullptr) || (dbt_work == nullptr) != (grad_wcos_dev == nullptr))
        return fail(VR_ERR_ARG, "dbt_work, grad_wsin_dev and grad_wcos_dev go together");
    int rc = stft_check(N, T, n_fft, hop);
    if (rc) return rc;
    rc = device_setup(dev, sm_count);
    if (rc) return rc;
    return gemm_setup(dev);
}

// the frame table of the kept-frames entries: F_kept in [1, T / hop + 1] (the table's contents stay on the device: strictly
// increasing indices in [0, T / hop + 1) are the caller's contract)
int stft_kept_check(const int32_t* frames_dev, int64_t N, int64_t T, int hop, int64_t F_kept) {
    if (!frames_dev) return fail(VR_ERR_ARG, "frames_dev must not be null");
    if (hop <= 0 || T <= 0) return fail(VR_ERR_SHAPE, "T, hop must be positive");
    if (F_kept < 1 || F_kept > T / hop + 1) return fail(VR_ERR_SHAPE, "F_kept=%lld outside [1, T/hop+1 = %lld]", (long long)F_kept, (long long)(T / hop + 1));
    if (N * F_kept >= (1ll << 31) / 2) return fail(VR_ERR_UNSUPPORTED, "too many frames for one launch; split the batch");
    return VR_OK;
}
}  // namespace
extern "C" {

int64_t vr_stft_general_workspace_floats(int64_t N, int64_t T, int32_t n_fft, int32_t hop, int64_t parts[3]) {
    if (N <= 0 || T <= 0 || hop <= 0 || n_fft <= 0) return 0;
    const int64_t M = N * (T / hop + 1), K = 2ll * n_fft;
    const int64_t a = 2 * N * stft_lp(T, n_fft), b = 2 * stft_bimg_floats(n_fft), c = K * stft_ldm(M);   // padded planar signal (the frames are views of it);       // C / dC: column-major, leading dimension a multiple of 4
    if (parts) { parts[0] = a; parts[1] = b; parts[2] = c; }
    return a + b + c;
}

int vr_stft_general_f32(const float* iq_dev, int64_t N, int64_t T, int32_t n_fft, int32_t hop,
                        const float* wsin_dev, const float* wcos_dev, float* frames_work, float* bt_work,
                        float* c_save /* may be NULL */, float* out_dev, void* stream) {
    int dev, sm_count;
    int rc = stft_forward_args(iq_dev, wsin_dev, wcos_dev, frames_work, bt_work, c_save, out_dev, N, T, n_fft, hop, dev, sm_count);
    if (rc) return rc;
    StftPlan q;
    rc = stft_plan(N, T, n_fft, hop, 0, sm_count, q);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    vr::vr_stft_pad_kernel<<<(unsigned)std::min<long long>((N * q.Lp + 255) / 256, sm_count * 16ll), 256, 0, st>>>(iq_dev, frames_work, N, (int)T, q.Lp, n_fft);
    return stft_forward_gemm(q, frames_work, n_fft, wsin_dev, wcos_dev, bt_work, c_save, out_dev, st);
}

int vr_stft_general_backward_f32(const float* grad_out_dev, const float* frames_work, const float* bt_work, const float* c_save,
                                 int64_t N, int64_t T, int32_t n_fft, int32_t hop,
                                 float* dc_work, float* da_work /* NULL: no grad_iq */, float* dbt_work /* NULL: no kernel grads */,
                                 float* grad_iq_dev, float* grad_wsin_dev, float* grad_wcos_dev, void* stream) {
    int dev, sm_count;
    int rc = stft_backward_args(grad_out_dev, frames_work, bt_work, c_save, dc_work, da_work, dbt_work, grad_iq_dev,
                                grad_wsin_dev, grad_wcos_dev, N, T, n_fft, hop, dev, sm_count);
    if (rc) return rc;
    StftPlan q;
    rc = stft_plan(N, T, n_fft, hop, 0, sm_count, q);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    rc = stft_backward_gemm(q, grad_out_dev, frames_work, n_fft, bt_work, c_save, dc_work, da_work,
                            dbt_work, grad_wsin_dev, grad_wcos_dev, dev, sm_count, st);
    if (rc || !da_work) return rc;
    vr::vr_stft_fold_kernel<<<(unsigned)std::min<long long>((N * T + 255) / 256, sm_count * 16ll), 256, 0, st>>>(da_work, grad_iq_dev, N, (int)T, q.F, n_fft, hop);
    CUDA_TRY(cudaGetLastError());
    return VR_OK;
}

int64_t vr_stft_general_frames_workspace_floats(int64_t N, int64_t F_kept, int32_t n_fft, int64_t parts[3]) {
    if (N <= 0 || F_kept <= 0 || n_fft <= 0) return 0;
    const int64_t M = N * F_kept, K = 2ll * n_fft;
    const int64_t a = 2 * N * F_kept * n_fft, b = 2 * stft_bimg_floats(n_fft), c = K * stft_ldm(M);    // compact kept frames; B images; C / dC
    if (parts) { parts[0] = a; parts[1] = b; parts[2] = c; }
    return a + b + c;
}

int vr_stft_general_frames_f32(const float* iq_dev, int64_t N, int64_t T, int32_t n_fft, int32_t hop,
                               const int32_t* frames_dev, int64_t F_kept,
                               const float* wsin_dev, const float* wcos_dev, float* frames_work, float* bt_work,
                               float* c_save /* may be NULL */, float* out_dev, void* stream) {
    int dev, sm_count;
    int rc = stft_forward_args(iq_dev, wsin_dev, wcos_dev, frames_work, bt_work, c_save, out_dev, N, T, n_fft, hop, dev, sm_count);
    if (rc) return rc;
    rc = stft_kept_check(frames_dev, N, T, hop, F_kept);
    if (rc) return rc;
    StftPlan q;
    rc = stft_plan(N, T, n_fft, hop, F_kept, sm_count, q);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    vr::vr_stft_gather_kernel<<<(unsigned)std::min<long long>((N * q.Lp + 255) / 256, sm_count * 16ll), 256, 0, st>>>(iq_dev, frames_dev, frames_work, N, (int)T, (int)F_kept, n_fft, hop);
    return stft_forward_gemm(q, frames_work, n_fft, wsin_dev, wcos_dev, bt_work, c_save, out_dev, st);
}

int vr_stft_general_frames_backward_f32(const float* grad_out_dev, const float* frames_work, const float* bt_work, const float* c_save,
                                        int64_t N, int64_t T, int32_t n_fft, int32_t hop, const int32_t* frames_dev, int64_t F_kept,
                                        float* dc_work, float* da_work, float* dbt_work,
                                        float* grad_iq_dev, float* grad_wsin_dev, float* grad_wcos_dev, void* stream) {
    int dev, sm_count;
    int rc = stft_backward_args(grad_out_dev, frames_work, bt_work, c_save, dc_work, da_work, dbt_work, grad_iq_dev,
                                grad_wsin_dev, grad_wcos_dev, N, T, n_fft, hop, dev, sm_count);
    if (rc) return rc;
    rc = stft_kept_check(frames_dev, N, T, hop, F_kept);
    if (rc) return rc;
    StftPlan q;
    rc = stft_plan(N, T, n_fft, hop, F_kept, sm_count, q);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    rc = stft_backward_gemm(q, grad_out_dev, frames_work, n_fft, bt_work, c_save,
                            dc_work, da_work, dbt_work, grad_wsin_dev, grad_wcos_dev, dev, sm_count, st);
    if (rc || !da_work) return rc;
    vr::vr_stft_fold_kept_kernel<<<(unsigned)std::min<long long>((N * T + 255) / 256, sm_count * 16ll), 256, 0, st>>>(da_work, frames_dev, grad_iq_dev, N, (int)T, (int)F_kept, n_fft, hop);
    CUDA_TRY(cudaGetLastError());
    return VR_OK;
}

int vr_plan_stft_general(int64_t N, int64_t T, int32_t n_fft, int32_t hop, int64_t F_kept, int32_t sm_count, int64_t plan[13]) {
    if (!plan) return fail(VR_ERR_ARG, "plan must not be null");
    StftPlan q;
    int rc = stft_plan(N, T, n_fft, hop, F_kept, sm_count > 0 ? sm_count : 148, q);
    if (rc) return rc;
    plan[0] = q.nb; plan[1] = q.F; plan[2] = q.M; plan[3] = q.ldm; plan[4] = q.Lp;
    plan[5] = q.row_tiles; plan[6] = q.col_tiles; plan[7] = q.kblocks;
    plan[8] = q.dbt_tiles; plan[9] = q.splits; plan[10] = q.kb_per_split; plan[11] = q.kb_last; plan[12] = q.hop_view;
    return VR_OK;
}

}  // extern "C"
