// mtfjsp_gemm.cu -- fused per-node linear layer of the GNN encoder on the 5th-gen tensor cores (sm_100a).
//
//   Z[r, :] = act(X[r, :] * in_scale + in_shift) @ W^T + bias          (act = ReLU or identity; affine optional)
//   stats  += (column sums of Z, column sums of Z^2)                   (FP64, for the BatchNorm that follows)
//
// Replaces, per layer of model/gcn_mlp.py:238-249 (Linear -> BatchNorm1d(batch stats) -> ReLU chain) and the outer
// BatchNorm of :154-157: the cuBLAS sgemm, the separate BatchNorm statistics pass and the separate normalise+ReLU pass.
// The normalisation of layer i is applied in the *prologue* of layer i+1 (scale/shift per input column), its
// statistics are accumulated in the *epilogue* of layer i, so every activation is written once and read once.
//
// Mechanics: one persistent CTA per SM, 128 threads.  W (128 x K, K-major = nn.Linear layout) is converted to TF32
// and parked in shared memory in the UMMA no-swizzle K-major core-matrix layout once; per 128-row tile the CTA
// stages X the same way (prologue math in registers), one elected thread issues K/8 `tcgen05.mma.kind::tf32`
// (M=128, N=128, K=8) accumulating in TMEM, `tcgen05.commit` arrives on an mbarrier, then each warp pulls its
// 32 TMEM lanes with `tcgen05.ld.32x32b.x32`, adds the bias, transposes through shared memory and writes 128-byte
// coalesced rows while accumulating the column statistics.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <type_traits>

#include "../../include/mtfjsp.h"

namespace {

constexpr int TILE_M = 128, TILE_N = 128;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!ok);
}
// shared-memory matrix descriptor, K-major, SWIZZLE_NONE: core matrix = 8 rows x 16 bytes, rows 16 B apart;
// LBO = byte distance between the two 16-byte K chunks of one MMA, SBO = byte distance between 8-row groups.
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)(lbo_bytes >> 4) << 16;
    d |= (uint64_t)(sbo_bytes >> 4) << 32;
    d |= 1ull << 46;  // descriptor version for sm_100
    return d;         // layout_type (bits 61-63) = 0: no swizzle
}
// instruction descriptor: D = F32, A = B = TF32, both K-major, N = 128, M = 128
constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((TILE_N >> 3) << 17) | ((TILE_M >> 4) << 24);

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(IDESC), "r"(accumulate));
}

#define TMEM_LD32(taddr, r)                                                                                          \
    asm volatile(                                                                                                    \
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                                    \
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,"  \
        "%29,%30,%31}, [%32];"                                                                                       \
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),  \
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),       \
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),      \
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])                    \
        : "r"(taddr))

// stage a [128 x KP] f32 block (row-major in global, leading dimension ld, `valid_rows` rows, `K` real columns) into
// the UMMA layout: element (r, k) at (r/8)*SBO + (k/4)*128 + (r%8)*16 + (k%4)*4.  A warp iteration covers
// 8 rows x 64 bytes: 2 full sectors per row in global, 512 contiguous bytes in shared memory.
template <bool AFFINE, int NWARPS>
__device__ __forceinline__ void stage_block(float* sdst, const float* __restrict__ g, long long row0, long long rows,
                                            int K, int KP, int ld, const float* s_scale, const float* s_shift,
                                            bool relu, int warp, int lane) {
    const int sbo = (KP / 4) * 128;
    const int r = lane & 7, c = lane >> 3;  // a quarter-warp covers 128 contiguous bytes of shared memory
    const int quads = KP / 16;
    const int total = 16 * quads;
    constexpr int U = 8;  // loads in flight per thread
    for (int it0 = warp; it0 < total; it0 += NWARPS * U) {
        float4 v[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const int it = it0 + u * NWARPS;
            const int grp = it / quads, q = it - grp * quads;
            const long long row = row0 + grp * 8 + r;
            const int k = q * 16 + c * 4;
            v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (it < total && row < rows && k < K) v[u] = __ldg(reinterpret_cast<const float4*>(g + row * ld + k));
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const int it = it0 + u * NWARPS;
            if (it >= total) break;
            const int grp = it / quads, q = it - grp * quads;
            const long long row = row0 + grp * 8 + r;
            const int k = q * 16 + c * 4;
            float4 x = v[u];
            if (AFFINE) {
                if (row < rows && k < K) {
                    x.x = x.x * s_scale[k] + s_shift[k]; x.y = x.y * s_scale[k + 1] + s_shift[k + 1];
                    x.z = x.z * s_scale[k + 2] + s_shift[k + 2]; x.w = x.w * s_scale[k + 3] + s_shift[k + 3];
                    if (relu) { x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f); }
                }
            }
            x.x = to_tf32(x.x); x.y = to_tf32(x.y); x.z = to_tf32(x.z); x.w = to_tf32(x.w);
            *reinterpret_cast<float4*>(reinterpret_cast<char*>(sdst) + grp * sbo + (q * 4 + c) * 128 + r * 16) = x;
        }
    }
}

constexpr int NPROD = 8;  // producer warps

// Producer-side staging of one A stage (128 rows x KS columns starting at column kbase), split in two: (1) every
// 16-byte piece goes global -> shared with cp.async (no register staging; several stages are in flight at once);
// (2) once landed, the issuing thread rounds its own pieces to TF32 in place and applies the folded BatchNorm
// (+ReLU) of the producing layer.
template <int KS>
__device__ __forceinline__ void tile_issue(float* sdst, const float* __restrict__ g, long long row0, long long rows, int K,
                                           int kbase, int pw, int lane) {
    constexpr int SBO = (KS / 4) * 128, QUADS = KS / 16, TOTAL = 16 * QUADS;
    const int r = lane & 7, c = lane >> 3;  // a quarter-warp covers 128 contiguous bytes of shared memory
    static_assert(NPROD % QUADS == 0, "a warp keeps one K chunk: its folded BatchNorm constants live in registers");
#pragma unroll
    for (int it = pw; it < TOTAL; it += NPROD) {
        const int grp = it / QUADS, q = it % QUADS;
        const long long row = row0 + grp * 8 + r;
        const int k = kbase + q * 16 + c * 4;
        const bool ok = row < rows && k < K;
        const float* src = ok ? g + row * K + k : g;
        const uint32_t dst = smem_u32(reinterpret_cast<char*>(sdst) + grp * SBO + (q * 4 + c) * 128 + r * 16);
        const int nbytes = ok ? 16 : 0;  // src-size 0: the 16 bytes are zero-filled
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
    }
}

template <int KS, bool AFFINE>
__device__ __forceinline__ void tile_transform(float* sdst, long long row0, long long rows, int K, int kbase,
                                               const float* s_scale, const float* s_shift, bool relu, int pw, int lane) {
    constexpr int SBO = (KS / 4) * 128, QUADS = KS / 16, TOTAL = 16 * QUADS;
    const int r = lane & 7, c = lane >> 3;
    const int q = pw % QUADS, k = kbase + q * 16 + c * 4;  // fixed per lane (NPROD % QUADS == 0)
    float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
    if (AFFINE) { sc = *reinterpret_cast<const float4*>(s_scale + k); sh = *reinterpret_cast<const float4*>(s_shift + k); }
    const bool kok = k < K;
    constexpr int PER = TOTAL / NPROD;  // pieces per lane
    static_assert(PER >= 1 && PER <= 8, "stage size");
    char* const colbase = reinterpret_cast<char*>(sdst) + (q * 4 + c) * 128 + r * 16;
    float4 x[PER];
#pragma unroll
    for (int u = 0; u < PER; u++) {  // all loads first: the in-place stores below would otherwise serialise them
        const int grp = (pw + u * NPROD) / QUADS;
        x[u] = *reinterpret_cast<const float4*>(colbase + grp * SBO);
    }
#pragma unroll
    for (int u = 0; u < PER; u++) {
        const int grp = (pw + u * NPROD) / QUADS;
        float4 v = x[u];
        if (AFFINE) {
            const long long row = row0 + grp * 8 + r;
            if (row < rows && kok) {
                v.x = v.x * sc.x + sh.x; v.y = v.y * sc.y + sh.y; v.z = v.z * sc.z + sh.z; v.w = v.w * sc.w + sh.w;
                if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
            }
        }
        v.x = to_tf32(v.x); v.y = to_tf32(v.y); v.z = to_tf32(v.z); v.w = to_tf32(v.w);
        *reinterpret_cast<float4*>(colbase + grp * SBO) = v;
    }
}

constexpr int NEPI = 8;          // epilogue warps: warp w drains TMEM lanes 32*(w%4).., columns 64*(w/4)..
constexpr int GEMM_WARPS = NEPI + NPROD;  // warps 0-7 epilogue, 8-15 operand staging (+ one MMA-issuing thread)
constexpr int STG_W = 32;       // per-warp 32 x 32 transpose tile, XOR-swizzled in 16-byte pieces

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// Grouped form (per-env BatchNorm statistics, mtfjsp.h "grouped encoder layers"): tiles are env-aligned.  With N <= 128
// rows per env a tile is rpt = (128 / N) * N rows of whole envs; with N > 128 an env is P = ceil(N / 128) tiles of
// 128 rows starting at its first row (the last piece owns N - 128 (P - 1) of them).
__device__ __forceinline__ long long gtile_row0(long long tile, int rpt, int nodes, int P) {
    return P == 1 ? tile * rpt : (tile / P) * nodes + (tile % P) * 128;
}
__device__ __forceinline__ int gtile_rows(long long tile, long long row0, long long rows, int rpt, int nodes, int P) {
    if (P > 1) return nodes - (int)(tile % P) * 128 < 128 ? nodes - (int)(tile % P) * 128 : 128;
    return rows - row0 < rpt ? (int)(rows - row0) : rpt;
}
// env_stats[env][piece][0|1][c] = column sums of Z and Z^2 over the env rows of one tile, read back from Z (L2) after the
// epilogue warps stored the tile (bar.sync 3 before the call).  One thread per (env, column) adds the rows in row order
// in FP64, so the sums depend only on the env's own rows, never on where the env sits in the tile or the batch.
__device__ __forceinline__ void env_stats_tile(const float* Z, double* __restrict__ env_stats, long long tile, long long row0,
                                               int nrows, int nodes, int P, int tid) {
    const int prow = P == 1 ? nodes : nrows;
    const int nenv = P == 1 ? nrows / nodes : 1;
    const long long env0 = P == 1 ? row0 / nodes : tile / P;
    const int piece = P == 1 ? 0 : (int)(tile % P);
    for (int item = tid; item < nenv * 128; item += NEPI * 32) {
        const int e = item >> 7, c = item & 127;
        const float* zp = Z + (row0 + (long long)e * nodes) * 128 + c;
        double s = 0.0, q = 0.0;
#pragma unroll 4
        for (int j = 0; j < prow; j++) {
            const double v = (double)__ldcg(zp + (long long)j * 128);
            s += v;
            q = fma(v, v, q);
        }
        double* dst = env_stats + ((env0 + e) * P + piece) * 256 + c;
        dst[0] = s;
        dst[128] = q;
    }
}

// Warp-specialised.  The A operand streams through a ring of NSTAGE shared-memory stages of 128 rows x KS columns
// (KS = min(K, 64): a K=128 tile is two stages), NSTAGE-1 of them in flight from HBM while one is transformed and
// multiplied; the accumulator is double-buffered in TMEM so the epilogue warps drain tile i while tile i+1 is formed.
//   sfree[s]      (count 1)  tcgen05.commit after the MMAs that read stage slot s: the slot may be refilled
//   full[b]       (count 1)  tcgen05.commit after the last MMA of a tile: TMEM[b] is ready
//   tmem_empty[b] (count 8)  the eight epilogue warps have pulled TMEM[b] into registers
constexpr int NSTAGE = 4;

// GROUPED: env-aligned tiles and per-env statistics (env_stats_tile) in `stats` instead of the batch-wide atomics; no
// input affine (the grouped K <= 16 first layer has none).
template <int KP, bool GROUPED>
__global__ void __launch_bounds__(GEMM_WARPS * 32, 1) linear_tf32_kernel(const float* __restrict__ X, long long rows, int K,
                                                                         const float* __restrict__ W,
                                                                         const float* __restrict__ bias,
                                                                         const float* __restrict__ in_scale,
                                                                         const float* __restrict__ in_shift, int in_relu,
                                                                         float* __restrict__ Z, double* __restrict__ stats,
                                                                         long long num_tiles, int g_rpt = 0,
                                                                         int g_nodes = 0, int g_P = 0) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr int KS = KP > 64 ? 64 : KP, SPT = KP / KS;  // stage width, stages per tile
    constexpr size_t WBYTES = (size_t)TILE_N * KP * 4, SBYTES = (size_t)TILE_M * KS * 4;
    float* sW = reinterpret_cast<float*>(smem);
    unsigned char* sRing = smem + WBYTES;
    float* sStg = reinterpret_cast<float*>(sRing + NSTAGE * SBYTES);
    float* s_bias = sStg + NEPI * 32 * STG_W;
    float* s_scale = s_bias + TILE_N;
    float* s_shift = s_scale + 128;
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_shift + 128);  // full[2], tmem_empty[2], sfree[NSTAGE]
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 4 + NSTAGE);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool affine = in_scale != nullptr;

    if (tid < TILE_N) s_bias[tid] = bias ? bias[tid] : 0.f;
    if (tid < 128) {
        s_scale[tid] = (affine && tid < K) ? in_scale[tid] : 1.f;
        s_shift[tid] = (affine && tid < K) ? in_shift[tid] : 0.f;
    }
    if (tid == 0) {
        mbar_init(smem_u32(s_bar + 0), 1);
        mbar_init(smem_u32(s_bar + 1), 1);
        mbar_init(smem_u32(s_bar + 2), NEPI);
        mbar_init(smem_u32(s_bar + 3), NEPI);
        for (int st = 0; st < NSTAGE; st++) mbar_init(smem_u32(s_bar + 4 + st), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {  // TMEM: 2 x 128 columns x 128 lanes of FP32 accumulators
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(256));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    // weights: [128 out, K in] row-major = K-major B operand, staged once per CTA
    stage_block<false, GEMM_WARPS>(sW, W, 0, TILE_N, K, KP, K, nullptr, nullptr, false, warp, lane);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *s_tmem;
    constexpr uint32_t SBO_W = (uint32_t)(KP / 4) * 128u, SBO_A = (uint32_t)(KS / 4) * 128u;
    const uint32_t bar_full = smem_u32(s_bar), bar_empty = smem_u32(s_bar + 2), bar_free = smem_u32(s_bar + 4);

    if (warp >= NEPI) {
        // ================= producers =================
        const int pw = warp - NEPI;
        const long long my_tiles = (num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x;
        const long long nst = my_tiles * SPT;  // stages this CTA streams, in order
        auto issue = [&](long long g) {        // every thread commits one group per stage, empty past the end
            if (g < nst) {
                const long long tile = blockIdx.x + (g / SPT) * (long long)gridDim.x;
                tile_issue<KS>(reinterpret_cast<float*>(sRing + (g % NSTAGE) * SBYTES), X,
                               GROUPED ? gtile_row0(tile, g_rpt, g_nodes, g_P) : tile * TILE_M, rows, K,
                               (int)(g % SPT) * KS, pw, lane);
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        for (int g = 0; g < NSTAGE - 1; g++) issue(g);
        for (long long g = 0; g < nst; g++) {
            const long long i = g / SPT, tile = blockIdx.x + i * (long long)gridDim.x;
            const int h = (int)(g % SPT), slot = (int)(g % NSTAGE), buf = (int)(i & 1);
            float* sA = reinterpret_cast<float*>(sRing + slot * SBYTES);
            asm volatile("cp.async.wait_group %0;" ::"n"(NSTAGE - 2) : "memory");  // stage g has landed (this thread's pieces)
            if (!GROUPED && affine) tile_transform<KS, true>(sA, tile * TILE_M, rows, K, h * KS, s_scale, s_shift, in_relu != 0, pw, lane);
            else tile_transform<KS, false>(sA, tile * TILE_M, rows, K, h * KS, nullptr, nullptr, false, pw, lane);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> visible to the MMA
            // refill the slot stage g-1 used: its MMAs ran while this stage was being transformed
            if (g >= 1 && g + NSTAGE - 1 < nst)
                mbar_wait(bar_free + (uint32_t)((g - 1) % NSTAGE) * 8, (uint32_t)(((g - 1) / NSTAGE) & 1));
            issue(g + NSTAGE - 1);
            asm volatile("bar.sync 1, %0;" ::"n"(NPROD * 32) : "memory");  // the producer warps
            if (tid == NEPI * 32) {
                if (h == 0 && i >= 2) mbar_wait(bar_empty + buf * 8, (uint32_t)(((i >> 1) - 1) & 1));  // TMEM[buf] drained
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t aA = smem_u32(sA), aW = smem_u32(sW) + (uint32_t)h * (KS / 8) * 256u;
#pragma unroll
                for (int k = 0; k < KS / 8; k++) {  // one MMA consumes 8 TF32 = two 16-byte chunks = 256 bytes of K
                    umma_tf32(tmem_base + buf * TILE_N, make_desc(aA + k * 256, 128, SBO_A), make_desc(aW + k * 256, 128, SBO_W),
                              (h > 0 || k > 0) ? 1u : 0u);
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_free + slot * 8)
                             : "memory");
                if (h == SPT - 1)
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_full + buf * 8)
                                 : "memory");
            }
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else {
        // ================= epilogue =================
        // Each warp drains a 32-row x 32-column chunk: TMEM gives lane = row with the 32 columns in registers; a
        // swizzled 4 KB shared-memory tile (16-byte piece j of row r at position j ^ (r & 7), conflict-free both
        // ways) turns that into lane = (row % 4, 4 columns) so that rows leave as full 128-byte lines (STG.128) and
        // the BatchNorm column statistics stay lane-local.
        float* stg = sStg + warp * 32 * STG_W;
        const int quad = warp & 3, half = warp >> 2;  // TMEM lanes 32*quad.., columns 64*half..
        const int sub = lane >> 3, c4 = lane & 7;     // lane owns columns 4*c4..4*c4+3 of rows == sub (mod 4)
        double csum[2][4] = {}, csq[2][4] = {};
        const float4 b0 = *reinterpret_cast<const float4*>(s_bias + half * 64 + c4 * 4);
        const float4 b1 = *reinterpret_cast<const float4*>(s_bias + half * 64 + 32 + c4 * 4);
        long long i = 0;
        for (long long tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, i++) {
            const int buf = (int)(i & 1);
            mbar_wait(bar_full + buf * 8, (uint32_t)((i >> 1) & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const long long trow0 = GROUPED ? gtile_row0(tile, g_rpt, g_nodes, g_P) : tile * TILE_M;
            const int tnrows = GROUPED ? gtile_rows(tile, trow0, rows, g_rpt, g_nodes, g_P) : 0;
            const long long rend = GROUPED ? trow0 + tnrows : rows;  // rows past rend belong to another tile (or none)
            const long long row0 = trow0 + quad * 32;
#pragma unroll
            for (int c2 = 0; c2 < 2; c2++) {
                const int cc = half * 2 + c2;
                uint32_t r[32];
                const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * TILE_N + cc * 32);
                TMEM_LD32(taddr, r);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (c2 == 1) {  // this warp no longer needs TMEM[buf]
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    if (lane == 0) mbar_arrive(bar_empty + buf * 8);
                }
#pragma unroll
                for (int j = 0; j < 8; j++)
                    *reinterpret_cast<uint4*>(stg + lane * STG_W + ((j ^ (lane & 7)) << 2)) =
                        make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                __syncwarp();
                const float4 bb = c2 == 0 ? b0 : b1;
                float* zp = Z + (row0 + sub) * TILE_N + cc * 32 + c4 * 4;
                float4 s = make_float4(0.f, 0.f, 0.f, 0.f), q = make_float4(0.f, 0.f, 0.f, 0.f);
                const bool full = row0 + 32 <= rend;
#pragma unroll
                for (int it = 0; it < 8; it++) {
                    const int rr = it * 4 + sub;
                    float4 v = *reinterpret_cast<const float4*>(stg + rr * STG_W + ((c4 ^ (rr & 7)) << 2));
                    v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
                    if (full || row0 + rr < rend) {
                        *reinterpret_cast<float4*>(zp + (size_t)it * 4 * TILE_N) = v;
                        if (!GROUPED) {
                            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
                            q.x = fmaf(v.x, v.x, q.x); q.y = fmaf(v.y, v.y, q.y); q.z = fmaf(v.z, v.z, q.z); q.w = fmaf(v.w, v.w, q.w);
                        }
                    }
                }
                if (!GROUPED) {
                    csum[c2][0] += (double)s.x; csum[c2][1] += (double)s.y; csum[c2][2] += (double)s.z; csum[c2][3] += (double)s.w;
                    csq[c2][0] += (double)q.x; csq[c2][1] += (double)q.y; csq[c2][2] += (double)q.z; csq[c2][3] += (double)q.w;
                }
                __syncwarp();
            }
            if (GROUPED) {
                asm volatile("bar.sync 3, %0;" ::"n"(NEPI * 32) : "memory");  // the tile's rows are stored
                env_stats_tile(Z, stats, tile, trow0, tnrows, g_nodes, g_P, tid);
            }
        }
        if (!GROUPED && stats) {  // fold the four row classes, then one atomic per column and warp
#pragma unroll
            for (int c2 = 0; c2 < 2; c2++)
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    double a = csum[c2][j], b = csq[c2][j];
                    a += __shfl_xor_sync(0xffffffffu, a, 8); a += __shfl_xor_sync(0xffffffffu, a, 16);
                    b += __shfl_xor_sync(0xffffffffu, b, 8); b += __shfl_xor_sync(0xffffffffu, b, 16);
                    if (sub == 0) {
                        atomicAdd(stats + half * 64 + c2 * 32 + c4 * 4 + j, a);
                        atomicAdd(stats + TILE_N + half * 64 + c2 * 32 + c4 * 4 + j, b);
                    }
                }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256));
}

// ---------------------------------------------------------------------------------------------------------------------
// K = 128 layers: the same kernel with the A operand brought in by the TMA unit.  `cp.async.bulk.tensor.2d` copies
// 128-row x 32-column boxes (128 bytes per row) of X into shared memory in the 128-byte-swizzled K-major layout that the
// MMA descriptor names (LayoutType SWIZZLE_128B: 16-byte piece c of row r sits at r * 128 + ((c ^ (r & 7)) << 4), 8-row
// groups 1,024 bytes apart), completion counted in bytes on the stage's mbarrier; rows past the end of X arrive as zeros.
// One thread issues two boxes per 64-column stage instead of 256 threads issuing eight 16-byte cp.async each -- ncu
// showed the cp.async form asking L2 for 2.9 GB of sectors for 1.2 GB of operand.  The staging warps still pass over the
// stage once in place (TF32 rounding + the folded BatchNorm / ReLU of the producing layer), each thread on fixed
// columns, conflict-free in the swizzled layout as well.
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;             // LBO: not used by swizzled K-major layouts
    d |= (uint64_t)(1024 >> 4) << 32;   // SBO: 8 rows x 128 bytes
    d |= 1ull << 46;                    // descriptor version for sm_100
    d |= 2ull << 61;                    // SWIZZLE_128B
    return d;
}
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_dst),
                 "l"(map), "r"(bar), "r"(c0), "r"(c1)
                 : "memory");
}

// GROUPED: the affine is per BatchNorm group, g_scale / g_shift [G,128] in global memory, group = (row / nodes) / epg
template <bool AFFINE, bool GROUPED = false>
__device__ __forceinline__ void tile_transform_sw(unsigned char* stage, long long row0, long long rows, int kbase,
                                                  const float* s_scale, const float* s_shift, bool relu, int pw, int lane,
                                                  const float* g_scale = nullptr, const float* g_shift = nullptr,
                                                  int nodes = 1, int epg = 1) {
    // stage = two boxes of 128 rows x 128 bytes; this thread owns logical 16-byte piece (q * 4 + c) of rows 8 * grp + r
    const int r = lane & 7, c = lane >> 3, q = pw & 3;
    const int piece = q * 4 + c, box = piece >> 3, pb = piece & 7;
    const int k = kbase + piece * 4;
    float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
    if (AFFINE) { sc = *reinterpret_cast<const float4*>(s_scale + k); sh = *reinterpret_cast<const float4*>(s_shift + k); }
    unsigned char* const base = stage + box * 16384 + r * 128 + ((pb ^ r) << 4);  // (8 grp + r) & 7 == r
    float4 x[8];
#pragma unroll
    for (int u = 0; u < 8; u++) x[u] = *reinterpret_cast<const float4*>(base + ((pw >> 2) + 2 * u) * 1024);
#pragma unroll
    for (int u = 0; u < 8; u++) {
        const int grp = (pw >> 2) + 2 * u;
        float4 v = x[u];
        if (AFFINE) {
            if (row0 + grp * 8 + r < rows) {
                if (GROUPED) {
                    const long long g = (row0 + grp * 8 + r) / nodes / epg;
                    sc = __ldg(reinterpret_cast<const float4*>(g_scale + g * 128 + k));
                    sh = __ldg(reinterpret_cast<const float4*>(g_shift + g * 128 + k));
                }
                v.x = v.x * sc.x + sh.x; v.y = v.y * sc.y + sh.y; v.z = v.z * sc.z + sh.z; v.w = v.w * sc.w + sh.w;
                if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
            }
        }
        v.x = to_tf32(v.x); v.y = to_tf32(v.y); v.z = to_tf32(v.z); v.w = to_tf32(v.w);
        *reinterpret_cast<float4*>(base + grp * 1024) = v;
    }
}

// AGG: the layer that follows a neighbourhood aggregation (model/gcn_mlp.py:125-149 then :238-249).  The aggregation is
// linear, so it commutes with the product: the rows go through the MMA one by one and the <= 3-term weighted mean over
// (self, job predecessor, machine predecessor) is formed from the PRODUCT rows in the epilogue, where the tile passes
// through shared memory anyway -- out[r] = (y[r] + w_job y[r-1] + w_mach y[src]) / n + bias, y = act(X) W^T.  Tiles hold
// whole envs (rpt = (128 / N) * N rows; the TMA box is rpt rows, the rest of the stage is ignored) so that every
// neighbour is in the tile; the separate aggregation pass (one read and one write of [rows,128]) disappears.
// GROUPED: env-aligned tiles (rpt rows of whole envs, or 128-row pieces of an env when nodes > 128: g_P pieces), the
// input affine per BatchNorm group ([G,128], envs_per_group = g_epg) and per-env statistics (env_stats_tile) in `stats`.
template <bool AGG, bool GROUPED>
__global__ void __launch_bounds__(GEMM_WARPS * 32, 1) linear_tf32_tma_kernel(const __grid_constant__ CUtensorMap tmapX, long long rows,
                                                                             const float* __restrict__ W,
                                                                             const float* __restrict__ bias,
                                                                             const float* __restrict__ in_scale,
                                                                             const float* __restrict__ in_shift, int in_relu,
                                                                             float* __restrict__ Z, double* __restrict__ stats,
                                                                             long long num_tiles, int rpt, int nodes,
                                                                             const float2* __restrict__ adj_w,
                                                                             const int16_t* __restrict__ adj_src, int g_P = 1,
                                                                             int g_epg = 1) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr int KP = 128, KS = 64, SPT = 2;
    constexpr int NST = AGG ? 3 : NSTAGE;  // the full-tile epilogue buffer of AGG takes one stage's room
    constexpr size_t WBYTES = (size_t)TILE_N * KP * 4, SBYTES = (size_t)TILE_M * KS * 4;
    constexpr size_t STG_FLOATS = AGG ? (size_t)TILE_M * TILE_N : (size_t)NEPI * 32 * STG_W;
    float* sW = reinterpret_cast<float*>(smem);
    unsigned char* sRing = smem + WBYTES;  // 1,024-byte aligned: WBYTES = 64 KB
    float* sStg = reinterpret_cast<float*>(sRing + NST * SBYTES);
    float* s_bias = sStg + STG_FLOATS;
    float* s_scale = s_bias + TILE_N;
    float* s_shift = s_scale + 128;
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_shift + 128);  // full[2], tmem_empty[2], sfree[NST], landed[NST]
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 4 + 2 * NST);
    float2* s_adjw = reinterpret_cast<float2*>(s_tmem + 4);        // AGG: [128] (w_job, w_mach) of the tile's rows
    int16_t* s_adjs = reinterpret_cast<int16_t*>(s_adjw + 128);    //      [128] tile row of the machine predecessor, -1 = none
    const int tile_rows = (AGG || GROUPED) ? rpt : TILE_M;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool affine = in_scale != nullptr;
    if (tid < TILE_N) s_bias[tid] = bias ? bias[tid] : 0.f;
    if (tid < 128) {
        s_scale[tid] = affine ? in_scale[tid] : 1.f;
        s_shift[tid] = affine ? in_shift[tid] : 0.f;
    }
    if (tid == 0) {
        mbar_init(smem_u32(s_bar + 0), 1);
        mbar_init(smem_u32(s_bar + 1), 1);
        mbar_init(smem_u32(s_bar + 2), NEPI);
        mbar_init(smem_u32(s_bar + 3), NEPI);
        for (int st = 0; st < 2 * NST; st++) mbar_init(smem_u32(s_bar + 4 + st), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmapX) : "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(256));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    stage_block<false, GEMM_WARPS>(sW, W, 0, TILE_N, KP, KP, KP, nullptr, nullptr, false, warp, lane);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *s_tmem;
    constexpr uint32_t SBO_W = (uint32_t)(KP / 4) * 128u;
    const uint32_t bar_full = smem_u32(s_bar), bar_empty = smem_u32(s_bar + 2), bar_free = smem_u32(s_bar + 4);
    const uint32_t bar_land = smem_u32(s_bar + 4 + NST);

    if (warp >= NEPI) {
        // ================= producers =================
        const int pw = warp - NEPI;
        const long long my_tiles = (num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x;
        const long long nst = my_tiles * SPT;  // stages this CTA streams, in order
        auto issue = [&](long long g) {        // one thread: two boxes of stage g into its ring slot
            if (g < nst) {
                const long long tile = blockIdx.x + (g / SPT) * (long long)gridDim.x;
                const int slot = (int)(g % NST);
                const uint32_t dst = smem_u32(sRing + slot * SBYTES), bar = bar_land + slot * 8;
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)(tile_rows * 256)) : "memory");
                const int col = (int)(g % SPT) * KS;
                const int row = (int)(GROUPED ? gtile_row0(tile, rpt, nodes, g_P) : tile * tile_rows);
                tma_load_2d(dst, &tmapX, col, row, bar);
                tma_load_2d(dst + 16384, &tmapX, col + 32, row, bar);
            }
        };
        const bool loader = tid == (NEPI + 1) * 32;  // first lane of the second staging warp
        if (loader)
            for (int g = 0; g < NST - 1; g++) issue(g);
        for (long long g = 0; g < nst; g++) {
            const long long i = g / SPT, tile = blockIdx.x + i * (long long)gridDim.x;
            const int h = (int)(g % SPT), slot = (int)(g % NST), buf = (int)(i & 1);
            unsigned char* sA = sRing + slot * SBYTES;
            mbar_wait(bar_land + slot * 8, (uint32_t)((g / NST) & 1));  // stage g has landed
            const long long arow0 = GROUPED ? gtile_row0(tile, rpt, nodes, g_P) : tile * tile_rows;
            if (affine) tile_transform_sw<true, GROUPED>(sA, arow0, rows, h * KS, s_scale, s_shift, in_relu != 0, pw, lane, in_scale,
                                                         in_shift, nodes, g_epg);
            else tile_transform_sw<false>(sA, arow0, rows, h * KS, nullptr, nullptr, false, pw, lane);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> visible to the MMA
            if (loader) {  // refill the slot stage g-1 used: its MMAs ran while this stage was being transformed
                if (g >= 1 && g + NST - 1 < nst)
                    mbar_wait(bar_free + (uint32_t)((g - 1) % NST) * 8, (uint32_t)(((g - 1) / NST) & 1));
                issue(g + NST - 1);
            }
            asm volatile("bar.sync 1, %0;" ::"n"(NPROD * 32) : "memory");  // the producer warps
            if (tid == NEPI * 32) {
                if (h == 0 && i >= 2) mbar_wait(bar_empty + buf * 8, (uint32_t)(((i >> 1) - 1) & 1));  // TMEM[buf] drained
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t aA = smem_u32(sA), aW = smem_u32(sW) + (uint32_t)h * (KS / 8) * 256u;
#pragma unroll
                for (int k = 0; k < KS / 8; k++) {  // 8 TF32 = 32 bytes of K inside the 128-byte swizzle row; 4 MMAs per box
                    umma_tf32(tmem_base + buf * TILE_N, make_desc_sw128(aA + (k >> 2) * 16384 + (k & 3) * 32),
                              make_desc(aW + k * 256, 128, SBO_W), (h > 0 || k > 0) ? 1u : 0u);
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_free + slot * 8)
                             : "memory");
                if (h == SPT - 1)
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_full + buf * 8)
                                 : "memory");
            }
        }
    } else {
        // ================= epilogue =================
        float* stg = sStg + warp * 32 * STG_W;
        const int quad = warp & 3, half = warp >> 2;
        const int sub = lane >> 3, c4 = lane & 7;
        // column sums of this lane's rows over all tiles of the CTA.  AGG keeps them in FP32 (<= ~150 tiles x 8 rows per lane, then FP64
        // across lanes and CTAs): the 16 registers this frees are what keeps its epilogue off the spill cliff
        using Acc = typename std::conditional<AGG, float, double>::type;
        Acc csum[2][4] = {}, csq[2][4] = {};
        const float4 b0 = *reinterpret_cast<const float4*>(s_bias + half * 64 + c4 * 4);
        const float4 b1 = *reinterpret_cast<const float4*>(s_bias + half * 64 + 32 + c4 * 4);
        long long i = 0;
        for (long long tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, i++) {
            const int buf = (int)(i & 1);
            if constexpr (AGG) {
                // the tile's adjacency rows, fetched while the products are still being formed
                const int tr = tid;  // 256 epilogue threads, 128 tile rows
                float2 aw = make_float2(0.f, 0.f);
                int as = -1;
                const long long gr = tile * rpt + tr;
                if (tr < rpt && gr < rows) {
                    aw = __ldg(adj_w + gr);
                    const int sr = __ldg(adj_src + gr);
                    as = sr >= 0 ? (tr / nodes) * nodes + sr : -1;
                }
                mbar_wait(bar_full + buf * 8, (uint32_t)((i >> 1) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                asm volatile("bar.sync 2, %0;" ::"n"(NEPI * 32) : "memory");  // the previous tile's rows have been read
                if (tr < TILE_M) { s_adjw[tr] = aw; s_adjs[tr] = (int16_t)as; }
                // product rows -> the full-tile buffer (16-byte pieces XOR-swizzled by row within each 128-byte group)
                const int yrow = quad * 32 + lane;
#pragma unroll
                for (int c2 = 0; c2 < 2; c2++) {
                    uint32_t r[32];
                    TMEM_LD32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * TILE_N + half * 64 + c2 * 32), r);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 8; j++)
                        *reinterpret_cast<uint4*>(sStg + yrow * TILE_N + (((half * 16 + c2 * 8 + j) ^ (yrow & 7)) << 2)) =
                            make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                if (lane == 0) mbar_arrive(bar_empty + buf * 8);  // TMEM[buf] may be overwritten
                asm volatile("bar.sync 2, %0;" ::"n"(NEPI * 32) : "memory");  // every product row of the tile is in place
                const int rbase = quad * 32;
                // this lane's eight rows: weights, predecessor rows and the scale of the mean, once for both column chunks
                float wj[8], wm[8], half_or_one[8], dvs[8];
                int prow[8];  // tile row of the machine predecessor | valid << 17
#pragma unroll
                for (int it = 0; it < 8; it++) {
                    const int tr2 = rbase + it * 4 + sub;
                    const bool ok = tr2 < rpt && tile * rpt + tr2 < rows;
                    const float2 w = s_adjw[tr2];
                    const int sr = s_adjs[tr2];
                    const bool hj = w.x != 0.f, hm = sr >= 0;
                    wj[it] = w.x;              // 0 without a job predecessor: the row read below is then multiplied away ...
                    wm[it] = hm ? w.y : 0.f;   // ... and row tr2 itself stands in for a missing machine predecessor
                    const int n = 1 + (hj ? 1 : 0) + (hm ? 1 : 0);
                    half_or_one[it] = n == 3 ? 0.333333343f : n == 2 ? 0.5f : 1.f;  // reciprocal of the member count ...
                    dvs[it] = (float)n;                                               // ... and the count itself
                    prow[it] = (hm ? sr : tr2) | (ok ? 1 << 17 : 0);
                }
#pragma unroll
                for (int c2 = 0; c2 < 2; c2++) {
                    const int piece = half * 16 + c2 * 8 + c4;  // 16-byte piece of the row this lane combines
                    const float4 bb = c2 == 0 ? b0 : b1;
                    float4 s = make_float4(0.f, 0.f, 0.f, 0.f), q = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int it = 0; it < 8; it++) {
                        const int tr2 = rbase + it * 4 + sub;
                        const int sr = prow[it] & 0xffff, jr = tr2 > 0 ? tr2 - 1 : 0;
                        const float4 xs = *reinterpret_cast<const float4*>(sStg + tr2 * TILE_N + ((piece ^ (tr2 & 7)) << 2));
                        const float4 xj = *reinterpret_cast<const float4*>(sStg + jr * TILE_N + ((piece ^ (jr & 7)) << 2));
                        const float4 xm = *reinterpret_cast<const float4*>(sStg + sr * TILE_N + ((piece ^ (sr & 7)) << 2));
                        float4 v;
                        v.x = fmaf(wm[it], xm.x, fmaf(wj[it], xj.x, xs.x)); v.y = fmaf(wm[it], xm.y, fmaf(wj[it], xj.y, xs.y));
                        v.z = fmaf(wm[it], xm.z, fmaf(wj[it], xj.z, xs.z)); v.w = fmaf(wm[it], xm.w, fmaf(wj[it], xj.w, xs.w));
                        {   // mean over the 1, 2 or 3 members; / 3 correctly rounded by one residual step on the reciprocal
                            // product (the residual is exactly zero for the factors 1 and 0.5: one branch-free sequence)
                            const float t = half_or_one[it], d = dvs[it];
                            const float qx = v.x * t, qy = v.y * t, qz = v.z * t, qw = v.w * t;
                            v.x = fmaf(fmaf(-d, qx, v.x), t, qx); v.y = fmaf(fmaf(-d, qy, v.y), t, qy);
                            v.z = fmaf(fmaf(-d, qz, v.z), t, qz); v.w = fmaf(fmaf(-d, qw, v.w), t, qw);
                        }
                        v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
                        if (prow[it] & (1 << 17)) {
                            *reinterpret_cast<float4*>(Z + (tile * rpt + tr2) * TILE_N + piece * 4) = v;
                            if (!GROUPED) {
                                s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
                                q.x = fmaf(v.x, v.x, q.x); q.y = fmaf(v.y, v.y, q.y); q.z = fmaf(v.z, v.z, q.z); q.w = fmaf(v.w, v.w, q.w);
                            }
                        }
                    }
                    if (!GROUPED) {
                        csum[c2][0] += (Acc)s.x; csum[c2][1] += (Acc)s.y; csum[c2][2] += (Acc)s.z; csum[c2][3] += (Acc)s.w;
                        csq[c2][0] += (Acc)q.x; csq[c2][1] += (Acc)q.y; csq[c2][2] += (Acc)q.z; csq[c2][3] += (Acc)q.w;
                    }
                }
                if (GROUPED) {
                    asm volatile("bar.sync 3, %0;" ::"n"(NEPI * 32) : "memory");  // the tile's rows are stored
                    env_stats_tile(Z, stats, tile, tile * rpt, gtile_rows(tile, tile * rpt, rows, rpt, nodes, 1), nodes, 1, tid);
                }
                continue;
            }
            mbar_wait(bar_full + buf * 8, (uint32_t)((i >> 1) & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const long long trow0 = GROUPED ? gtile_row0(tile, rpt, nodes, g_P) : tile * TILE_M;
            const int tnrows = GROUPED ? gtile_rows(tile, trow0, rows, rpt, nodes, g_P) : 0;
            const long long rend = GROUPED ? trow0 + tnrows : rows;  // rows past rend belong to another tile (or none)
            const long long row0 = trow0 + quad * 32;
#pragma unroll
            for (int c2 = 0; c2 < 2; c2++) {
                const int cc = half * 2 + c2;
                uint32_t r[32];
                const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * TILE_N + cc * 32);
                TMEM_LD32(taddr, r);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (c2 == 1) {
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    if (lane == 0) mbar_arrive(bar_empty + buf * 8);
                }
#pragma unroll
                for (int j = 0; j < 8; j++)
                    *reinterpret_cast<uint4*>(stg + lane * STG_W + ((j ^ (lane & 7)) << 2)) =
                        make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                __syncwarp();
                const float4 bb = c2 == 0 ? b0 : b1;
                float* zp = Z + (row0 + sub) * TILE_N + cc * 32 + c4 * 4;
                float4 s = make_float4(0.f, 0.f, 0.f, 0.f), q = make_float4(0.f, 0.f, 0.f, 0.f);
                const bool full = row0 + 32 <= rend;
#pragma unroll
                for (int it = 0; it < 8; it++) {
                    const int rr = it * 4 + sub;
                    float4 v = *reinterpret_cast<const float4*>(stg + rr * STG_W + ((c4 ^ (rr & 7)) << 2));
                    v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
                    if (full || row0 + rr < rend) {
                        *reinterpret_cast<float4*>(zp + (size_t)it * 4 * TILE_N) = v;
                        if (!GROUPED) {
                            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
                            q.x = fmaf(v.x, v.x, q.x); q.y = fmaf(v.y, v.y, q.y); q.z = fmaf(v.z, v.z, q.z); q.w = fmaf(v.w, v.w, q.w);
                        }
                    }
                }
                if (!GROUPED) {
                    if (!GROUPED) {
                        csum[c2][0] += (Acc)s.x; csum[c2][1] += (Acc)s.y; csum[c2][2] += (Acc)s.z; csum[c2][3] += (Acc)s.w;
                        csq[c2][0] += (Acc)q.x; csq[c2][1] += (Acc)q.y; csq[c2][2] += (Acc)q.z; csq[c2][3] += (Acc)q.w;
                    }
                }
                __syncwarp();
            }
            if (GROUPED) {
                asm volatile("bar.sync 3, %0;" ::"n"(NEPI * 32) : "memory");  // the tile's rows are stored
                env_stats_tile(Z, stats, tile, trow0, tnrows, nodes, g_P, tid);
            }
        }
        if (!GROUPED && stats) {
#pragma unroll
            for (int c2 = 0; c2 < 2; c2++)
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    double a = (double)csum[c2][j], b = (double)csq[c2][j];
                    a += __shfl_xor_sync(0xffffffffu, a, 8); a += __shfl_xor_sync(0xffffffffu, a, 16);
                    b += __shfl_xor_sync(0xffffffffu, b, 8); b += __shfl_xor_sync(0xffffffffu, b, 16);
                    if (sub == 0) {
                        atomicAdd(stats + half * 64 + c2 * 32 + c4 * 4 + j, a);
                        atomicAdd(stats + TILE_N + half * 64 + c2 * 32 + c4 * 4 + j, b);
                    }
                }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256));
}

// BatchNorm1d with batch statistics folded into a per-column affine: scale = gamma / sqrt(var + eps),
// shift = beta - mean * scale (biased variance, as torch uses for normalisation in training mode)
__global__ void bn_finalize_kernel(const double* __restrict__ stats, double inv_rows, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float eps, float* scale, float* shift, int C) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double mean = stats[c] * inv_rows;
    double var = stats[C + c] * inv_rows - mean * mean;
    if (var < 0) var = 0;
    const double sc = (double)gamma[c] / sqrt(var + (double)eps);
    scale[c] = (float)sc;
    shift[c] = (float)((double)beta[c] - mean * sc);
}
// grouped: env_stats [B,P,2,C] -> scale, shift [G,C]; a group's sums are its envs' sums (each the sum of its pieces),
// added in index order
__global__ void bn_finalize_grouped_kernel(const double* __restrict__ env_stats, long long G, int P, int epg, double inv_rows,
                                           const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float* scale,
                                           float* shift, int C) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= G * C) return;
    const long long g = idx / C;
    const int c = (int)(idx - g * C);
    double s = 0.0, q = 0.0;
    for (int e = 0; e < epg; e++) {
        const double* st = env_stats + (g * epg + e) * P * 2 * C + c;
        double es = 0.0, eq = 0.0;
        for (int p = 0; p < P; p++) { es += st[(size_t)p * 2 * C]; eq += st[(size_t)p * 2 * C + C]; }
        s += es;
        q += eq;
    }
    const double mean = s * inv_rows;  // as bn_finalize_kernel
    double var = q * inv_rows - mean * mean;
    if (var < 0) var = 0;
    const double sc = (double)gamma[c] / sqrt(var + (double)eps);
    scale[idx] = (float)sc;
    shift[idx] = (float)((double)beta[c] - mean * sc);
}


// =====================================================================================================================
// Weight gradient of the layer above, for the PPO update (ppo_algorithm.py:918-1003 backward passes):
//     dW[128, K] = dY^T X        db[128] = column sums of dY          dY [rows,128], X [rows,K] row-major f32
// The reduction runs over ROWS, so both operands enter the MMA transposed: A(m, r) = dY[r, m], B(n, r) = X[r, n], both
// "K-major" with K = r.  Four consecutive r of one feature must sit in one 16-byte piece, while global memory has four
// consecutive FEATURES of one r in a piece: every thread loads a 4 x 4 block (four rows, one feature quad; a warp
// instruction reads one whole 512-byte row), transposes it by register naming and stores four 16-byte pieces.  The
// 8-feature groups are 16 bytes further apart than the data needs (SBO = 2064), which makes those stores
// bank-conflict-free.  One CTA per SM walks 64-row stages (ring of 3), accumulates ALL of them into one TMEM
// accumulator and writes its partial [128, NP] once; a second small kernel adds the partials in CTA order, so the
// result does not depend on scheduling.
constexpr int WG_KS = 64, WG_NSTAGE = 3, WG_WARPS = 16;
constexpr int WG_SBO = (WG_KS / 4) * 128 + 16;

__device__ __forceinline__ void umma_tf32_desc(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate));
}

template <int NP>
__global__ void __launch_bounds__(WG_WARPS * 32, 1) wgrad_tf32_kernel(const float* __restrict__ dY, const float* __restrict__ X,
                                                                      long long rows, int K, float* __restrict__ parts,
                                                                      float* __restrict__ dbparts, long long num_stages) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr int A_BYTES = 16 * WG_SBO, B_BYTES = (NP / 8) * WG_SBO;
    constexpr int TCOLS = NP < 32 ? 32 : NP;
    constexpr uint32_t IDESC_W = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(NP >> 3) << 17) | ((TILE_M >> 4) << 24);
    unsigned char* sA = smem;
    unsigned char* sB = smem + WG_NSTAGE * A_BYTES;
    double* s_db = reinterpret_cast<double*>(sB + WG_NSTAGE * B_BYTES);          // [WG_WARPS][128]
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_db + WG_WARPS * 128);         // sfree[NSTAGE], done
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + WG_NSTAGE + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int st = 0; st <= WG_NSTAGE; st++) mbar_init(smem_u32(s_bar + st), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(TCOLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *s_tmem;
    const uint32_t bar_free = smem_u32(s_bar), bar_done = smem_u32(s_bar + WG_NSTAGE);

    // unit of this thread: A (dY): row quad `warp`, feature quad `lane`;  B (X): NP/4 feature quads x 16 row quads
    constexpr int BQ = NP / 4;
    const bool b_on = tid < BQ * 16;
    const int b_fq = tid % BQ, b_rq = tid / BQ;
    const bool b_col_ok = b_fq * 4 < K;

    float4 va[4], vb[4];
    auto load = [&](long long stage, float4* a, float4* b) {
        const long long r0 = stage * WG_KS;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const long long ra = r0 + warp * 4 + j;
            a[j] = ra < rows ? __ldg(reinterpret_cast<const float4*>(dY + ra * TILE_N + lane * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
            const long long rb = r0 + b_rq * 4 + j;
            b[j] = (b_on && b_col_ok && rb < rows) ? __ldg(reinterpret_cast<const float4*>(X + rb * K + b_fq * 4))
                                                  : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    // transposed store of a 4 x 4 block: piece i = feature 4*fq + i, rows 4*rq .. 4*rq+3
    auto store = [&](unsigned char* base, int fq, int rq, const float4* v) {
        const int f0 = fq * 4;
        unsigned char* p = base + (f0 >> 3) * WG_SBO + rq * 128 + (f0 & 7) * 16;
        *reinterpret_cast<float4*>(p) = make_float4(to_tf32(v[0].x), to_tf32(v[1].x), to_tf32(v[2].x), to_tf32(v[3].x));
        *reinterpret_cast<float4*>(p + 16) = make_float4(to_tf32(v[0].y), to_tf32(v[1].y), to_tf32(v[2].y), to_tf32(v[3].y));
        *reinterpret_cast<float4*>(p + 32) = make_float4(to_tf32(v[0].z), to_tf32(v[1].z), to_tf32(v[2].z), to_tf32(v[3].z));
        *reinterpret_cast<float4*>(p + 48) = make_float4(to_tf32(v[0].w), to_tf32(v[1].w), to_tf32(v[2].w), to_tf32(v[3].w));
    };

    double dbacc[4] = {0.0, 0.0, 0.0, 0.0};
    const long long my_n = (num_stages - blockIdx.x + gridDim.x - 1) / gridDim.x;
    if (my_n > 0) load(blockIdx.x, va, vb);
    for (long long i = 0; i < my_n; i++) {
        float4 na[4], nb[4];
        const bool more = i + 1 < my_n;
        if (more) load(blockIdx.x + (i + 1) * (long long)gridDim.x, na, nb);
        const int slot = (int)(i % WG_NSTAGE);
        if (i >= WG_NSTAGE) mbar_wait(bar_free + slot * 8, (uint32_t)((i / WG_NSTAGE - 1) & 1));  // the MMAs that read it are done
        store(sA + slot * A_BYTES, lane, warp, va);
        if (b_on) store(sB + slot * B_BYTES, b_fq, b_rq, vb);
        dbacc[0] += (double)((va[0].x + va[1].x) + (va[2].x + va[3].x));
        dbacc[1] += (double)((va[0].y + va[1].y) + (va[2].y + va[3].y));
        dbacc[2] += (double)((va[0].z + va[1].z) + (va[2].z + va[3].z));
        dbacc[3] += (double)((va[0].w + va[1].w) + (va[2].w + va[3].w));
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t aA = smem_u32(sA + slot * A_BYTES), aB = smem_u32(sB + slot * B_BYTES);
#pragma unroll
            for (int k = 0; k < WG_KS / 8; k++)
                umma_tf32_desc(tmem_base, make_desc(aA + k * 256, 128, WG_SBO), make_desc(aB + k * 256, 128, WG_SBO), IDESC_W,
                               (i > 0 || k > 0) ? 1u : 0u);
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_free + slot * 8)
                         : "memory");
            if (!more)
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_done) : "memory");
        }
        if (more) {
#pragma unroll
            for (int j = 0; j < 4; j++) { va[j] = na[j]; vb[j] = nb[j]; }
        }
    }
    // bias gradient: warp partials in a fixed order
#pragma unroll
    for (int j = 0; j < 4; j++) s_db[warp * 128 + lane * 4 + j] = dbacc[j];
    __syncthreads();
    if (tid < 128 && dbparts) {
        double t = 0.0;
        for (int w = 0; w < WG_WARPS; w++) t += s_db[w * 128 + tid];
        dbparts[(size_t)blockIdx.x * 128 + tid] = (float)t;
    }
    // accumulator -> this CTA's partial
    if (warp < 4) {
        float* out = parts + ((size_t)blockIdx.x * TILE_M + warp * 32 + lane) * NP;
        if (my_n > 0) {
            mbar_wait(bar_done, 0);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int c0 = 0; c0 < NP; c0 += 32) {
                uint32_t r[32];
                TMEM_LD32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, r);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int j = 0; j < 32 && c0 + j < NP; j += 4)
                    *reinterpret_cast<uint4*>(out + c0 + j) = make_uint4(r[j], r[j + 1], r[j + 2], r[j + 3]);
            }
        } else {
            for (int j = 0; j < NP; j += 4) *reinterpret_cast<float4*>(out + j) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TCOLS));
}

// dW[m, k] = sum over CTAs (in order) of parts[c][m][k]; db likewise
__global__ void wgrad_reduce_kernel(const float* __restrict__ parts, const float* __restrict__ dbparts, int nparts, int NP, int K,
                                    float* __restrict__ dW, float* __restrict__ db) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < TILE_M * K) {
        const int m = idx / K, k = idx % K;
        float t = 0.f;
        for (int c = 0; c < nparts; c++) t += parts[((size_t)c * TILE_M + m) * NP + k];
        dW[idx] = t;
    }
    if (db && idx < TILE_M) {
        float t = 0.f;
        for (int c = 0; c < nparts; c++) t += dbparts[(size_t)c * 128 + idx];
        db[idx] = t;
    }
}


// =====================================================================================================================
// Policy head in ONE kernel (model/gcn_mlp.py:258-320 MLPActor over cat(per-row, per-env, per-env) features,
// actor_critic.py:244-268 and :455-470):
//     out[r] = tanh( tanh( act(X[src(r)]) Wa^T + bias_env[r / rpe] ) W1^T + b1 ) . w2 + b2
// Nothing in this chain couples rows, so a 128-row tile goes through both products without leaving the SM: the rows are
// gathered (candidate op of each job, or the row itself), the producing layer's BatchNorm + ReLU is applied, the tile is
// staged as the A operand; `tcgen05.mma` -> TMEM; the first epilogue adds the per-env bias (the per-env column blocks of
// the first weight matrix, applied once per env by the caller), takes tanh and writes the result back INTO the A buffer
// (the first product has finished reading it) as the second product's operand; the second epilogue takes tanh, dots the
// row with w2 and writes one float per row: one gathered read of [rows,128] in all.  Both weight matrices stay in shared memory (2 x 64 KB), one CTA per SM.
// tanh / ELU for operands that are rounded to TF32 next (or summed into a score next to TF32 products): one ex2.approx
// and one fast division instead of the ~25-instruction accurate routines; absolute error < 3e-7
__device__ __forceinline__ float tanh_fast(float x) {
    const float t = __expf(2.f * fminf(x, 44.f));
    return 1.f - __fdividef(2.f, t + 1.f);
}
__device__ __forceinline__ float elu_fast(float x) { return x > 0.f ? x : __expf(x) - 1.f; }

constexpr int HEAD_WARPS = 16;

// GROUPED: in_scale / in_shift are [G,128], one affine per BatchNorm group of epg envs
template <bool GROUPED>
__global__ void __launch_bounds__(HEAD_WARPS * 32, 1) head_tf32_kernel(
    const float* __restrict__ X, const int32_t* __restrict__ cand, long long rows, int rpe, int nodes_per_env,
    const float* __restrict__ in_scale, const float* __restrict__ in_shift, int in_relu, const float* __restrict__ Wa,
    const float* __restrict__ bias_env, long long bias_rows, const float* __restrict__ W1, const float* __restrict__ b1,
    const float* __restrict__ w2, const float* __restrict__ b2, float* __restrict__ out, long long num_tiles, int epg = 1) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr size_t WBYTES = (size_t)TILE_N * 128 * 4;
    float* sWa = reinterpret_cast<float*>(smem);
    float* sW1 = reinterpret_cast<float*>(smem + WBYTES);
    float* sA = reinterpret_cast<float*>(smem + 2 * WBYTES);
    float* s_part = reinterpret_cast<float*>(smem + 3 * WBYTES);  // [4][128] partial dots of the second epilogue
    float* s_b1 = s_part + 4 * 128;
    float* s_w2 = s_b1 + 128;
    float* s_scale = s_w2 + 128;
    float* s_shift = s_scale + 128;
    int* s_row = reinterpret_cast<int*>(s_shift + 128);  // [2][128] source row of each tile row (-1 past the end)
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_row + 256);
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool affine = in_scale != nullptr;
    if (tid < 128) {
        s_b1[tid] = b1 ? b1[tid] : 0.f;
        s_w2[tid] = w2[tid];
        s_scale[tid] = affine ? in_scale[tid] : 1.f;
        s_shift[tid] = affine ? in_shift[tid] : 0.f;
    }
    if (tid == 0) {
        mbar_init(smem_u32(s_bar + 0), 1);
        mbar_init(smem_u32(s_bar + 1), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(256));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    stage_block<false, HEAD_WARPS>(sWa, Wa, 0, TILE_N, 128, 128, 128, nullptr, nullptr, false, warp, lane);
    stage_block<false, HEAD_WARPS>(sW1, W1, 0, TILE_N, 128, 128, 128, nullptr, nullptr, false, warp, lane);
    auto fill_rows = [&](long long tile, int slot) {  // threads 0..127
        const long long r = tile * TILE_M + tid;
        int src = -1;
        if (tile < num_tiles && r < rows) src = cand ? (int)((r / rpe) * nodes_per_env + __ldg(cand + r)) : (int)r;
        s_row[slot * 128 + tid] = src;
    };
    if (tid < 128) fill_rows(blockIdx.x, 0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *s_tmem;
    const uint32_t bar0 = smem_u32(s_bar), bar1 = smem_u32(s_bar + 1);
    const float b2v = b2 ? __ldg(b2) : 0.f;

    // tile rows -> registers: iteration it = warp + 16 u covers rows 8 (it / 8) .., columns 16 (it % 8) ..; lane = (row % 8,
    // 16-byte piece): the mapping of stage_block (conflict-free 512-byte shared-memory runs per warp)
    const int r8 = lane & 7, c4 = lane >> 3;
    float4 v[8];
    auto gather = [&](int slot) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int it = warp + u * HEAD_WARPS, grp = it >> 3, q = it & 7;
            const int src = s_row[slot * 128 + grp * 8 + r8];
            v[u] = src >= 0 ? __ldg(reinterpret_cast<const float4*>(X + (size_t)src * 128 + q * 16 + c4 * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto store_a = [&](int slot) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int it = warp + u * HEAD_WARPS, grp = it >> 3, q = it & 7, k = q * 16 + c4 * 4;
            float4 x = v[u];
            if (affine && s_row[slot * 128 + grp * 8 + r8] >= 0) {
                float4 sc, sh;
                if (GROUPED) {
                    const int src = s_row[slot * 128 + grp * 8 + r8];
                    const long long g = (long long)(cand ? src / nodes_per_env : src / rpe) / epg;
                    sc = __ldg(reinterpret_cast<const float4*>(in_scale + g * 128 + k));
                    sh = __ldg(reinterpret_cast<const float4*>(in_shift + g * 128 + k));
                } else {
                    sc = *reinterpret_cast<const float4*>(s_scale + k); sh = *reinterpret_cast<const float4*>(s_shift + k);
                }
                x.x = x.x * sc.x + sh.x; x.y = x.y * sc.y + sh.y; x.z = x.z * sc.z + sh.z; x.w = x.w * sc.w + sh.w;
                if (in_relu) { x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f); }
            }
            x.x = to_tf32(x.x); x.y = to_tf32(x.y); x.z = to_tf32(x.z); x.w = to_tf32(x.w);
            *reinterpret_cast<float4*>(reinterpret_cast<char*>(sA) + grp * 4096 + (q * 4 + c4) * 128 + r8 * 16) = x;
        }
    };
    auto mma_tile = [&](const float* sW, uint32_t dcol) {  // one elected thread: D[dcol..] = A W^T over K = 128
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t aA = smem_u32(sA), aW = smem_u32(sW);
#pragma unroll
        for (int k = 0; k < 16; k++)
            umma_tf32(tmem_base + dcol, make_desc(aA + k * 256, 128, 4096), make_desc(aW + k * 256, 128, 4096), k > 0 ? 1u : 0u);
    };

    const int quad = warp & 3, cg = warp >> 2;  // this warp's TMEM lanes 32 quad .., columns 32 cg ..
    const int trow = quad * 32 + lane;          // its thread's tile row
    gather(0);
    long long i = 0;
    for (long long tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, i++) {
        const int slot = (int)(i & 1);
        const uint32_t par = (uint32_t)(i & 1);
        store_a(slot);
        if (tid < 128) fill_rows(tile + gridDim.x, slot ^ 1);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (tid == 0) {
            mma_tile(sWa, 0);
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar0) : "memory");
        }
        gather(slot ^ 1);  // the next tile's rows travel while this tile is multiplied
        mbar_wait(bar0, par);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const long long grow = tile * TILE_M + trow;
        const bool rok = grow < rows;
        {   // first epilogue: + per-env bias, tanh, back into the A buffer as the second product's operand
            uint32_t r[32];
            TMEM_LD32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(cg * 32), r);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            const long long brow = bias_rows == 1 ? 0 : (rok ? grow / rpe : 0);
            const float4* bp = reinterpret_cast<const float4*>(bias_env + brow * 128 + cg * 32);
            char* dst = reinterpret_cast<char*>(sA) + (trow >> 3) * 4096 + (cg * 8) * 128 + (trow & 7) * 16;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const float4 bb = __ldg(bp + j);
                float4 x;
                x.x = to_tf32(tanh_fast(__uint_as_float(r[4 * j]) + bb.x)); x.y = to_tf32(tanh_fast(__uint_as_float(r[4 * j + 1]) + bb.y));
                x.z = to_tf32(tanh_fast(__uint_as_float(r[4 * j + 2]) + bb.z)); x.w = to_tf32(tanh_fast(__uint_as_float(r[4 * j + 3]) + bb.w));
                if (!rok) x = make_float4(0.f, 0.f, 0.f, 0.f);
                *reinterpret_cast<float4*>(dst + j * 128) = x;
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (tid == 0) {
            mma_tile(sW1, TILE_N);
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar1) : "memory");
        }
        mbar_wait(bar1, par);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        {   // second epilogue: + b1, tanh, dot with w2 over this warp's 32 columns
            uint32_t r[32];
            TMEM_LD32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(TILE_N + cg * 32), r);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            float acc = 0.f;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const float4 bb = *reinterpret_cast<const float4*>(s_b1 + cg * 32 + 4 * j);
                const float4 ww = *reinterpret_cast<const float4*>(s_w2 + cg * 32 + 4 * j);
                acc = fmaf(tanh_fast(__uint_as_float(r[4 * j]) + bb.x), ww.x, acc);
                acc = fmaf(tanh_fast(__uint_as_float(r[4 * j + 1]) + bb.y), ww.y, acc);
                acc = fmaf(tanh_fast(__uint_as_float(r[4 * j + 2]) + bb.z), ww.z, acc);
                acc = fmaf(tanh_fast(__uint_as_float(r[4 * j + 3]) + bb.w), ww.w, acc);
            }
            s_part[cg * 128 + trow] = acc;
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (tid < 128) {
            const long long orow = tile * TILE_M + tid;
            if (orow < rows) out[orow] = ((s_part[tid] + s_part[128 + tid]) + (s_part[256 + tid] + s_part[384 + tid])) + b2v;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256));
}


// =====================================================================================================================
// Machine-node trunk in ONE kernel (model/actor_critic.py:381-420: m_fea_1_fcl, m_fea_2_fcl, three applications of the
// GAT layer model/gat.py:82-159 on the fixed 2-node graph with ELU between them, mean over the two node sets):
//     h1 = f1 W1p^T, h2 = f2 W2p^T;   3 x { t = [h1; h2] W;  att = softmax(lrelu(t1.a_src + t1.a_dst), lrelu(t1.a_src + t2.a_dst));
//                                          h1 = att0 t1 + att1 t2, h2 = t2;  (ELU on both between layers) };   out = (h1 + h2) / 2
// Nothing couples machines before the BatchNorm that follows, so 128 machines run through all three layers on one SM: the
// input projections (K = 6 / 8) on the CUDA cores straight into the A operands, each layer's product on `tcgen05.mma` into
// TMEM, the attention / combination / ELU in the epilogue, written back into the A buffers for the next layer; one [R,128]
// write in all.  The two node sets are TWO products per layer (t1 = h1 W into TMEM columns 0..127, t2 = h2 W into
// 128..255), so that the thread that owns a machine's TMEM lane holds both of its rows: no exchange of node-2 rows through
// shared memory, every thread does the same work.
// GROUPED (per-env BatchNorm statistics): a tile is rpt = (128 / M) * M machines of whole envs (lanes >= rpt idle), and
// instead of the batch-wide atomics `stats` is env_stats [B,1,2,128]: the last layer also parks the output rows in the
// (then free) first A buffer, and one thread per (env, column) adds the env's rows from there in row order in FP64, so
// an env's statistics are the same bits at any batch position.
constexpr int TRUNK_WARPS = 16;
template <bool GROUPED>
__global__ void __launch_bounds__(TRUNK_WARPS * 32, 1) gat_trunk2_tf32_kernel(
    const float* __restrict__ f1, const float* __restrict__ f2, const float* __restrict__ W1p, const float* __restrict__ W2p,
    const float* __restrict__ Wt, const float* __restrict__ a_src, const float* __restrict__ a_dst, float* __restrict__ out,
    double* __restrict__ stats, long long R, long long num_tiles, int rpt, int M) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr size_t WBYTES = (size_t)TILE_N * 128 * 4;
    float* sW = reinterpret_cast<float*>(smem);
    float* sA1 = reinterpret_cast<float*>(smem + WBYTES);
    float* sA2 = reinterpret_cast<float*>(smem + 2 * WBYTES);
    float* s_dot = reinterpret_cast<float*>(smem + 3 * WBYTES);          // [3][4][128]: s1, d1, d2 partials per column group
    float* s_as = s_dot + 3 * 4 * 128;
    float* s_ad = s_as + 128;
    float* s_w1p = s_ad + 128;                                           // [128][6]
    float* s_w2p = s_w1p + 128 * 6;                                      // [128][8]
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_w2p + 128 * 8);
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid < 128) { s_as[tid] = a_src[tid]; s_ad[tid] = a_dst[tid]; }
    for (int i = tid; i < 128 * 6; i += blockDim.x) s_w1p[i] = W1p[i];
    for (int i = tid; i < 128 * 8; i += blockDim.x) s_w2p[i] = W2p[i];
    if (tid == 0) {
        mbar_init(smem_u32(s_bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(256));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    stage_block<false, TRUNK_WARPS>(sW, Wt, 0, TILE_N, 128, 128, 128, nullptr, nullptr, false, warp, lane);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *s_tmem;
    const uint32_t bar = smem_u32(s_bar);

    const int quad = warp & 3, cg = warp >> 2;   // TMEM lanes 32 quad .., columns 32 cg ..
    const int mloc = quad * 32 + lane;           // this thread's machine within the tile
    const size_t arow = (size_t)(mloc >> 3) * 4096 + (cg * 8) * 128 + (mloc & 7) * 16;  // its 32 columns in an A buffer
    uint32_t phase = 0;
    double st_sum = 0.0, st_sq = 0.0;
    for (long long tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const long long m = tile * (GROUPED ? rpt : 128) + mloc;
        const bool mok = m < R && (!GROUPED || mloc < rpt);
        {   // input projections on the CUDA cores, straight into the two A operands
            float fa[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, fb[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (mok) {
                const float2* p2 = reinterpret_cast<const float2*>(f1 + m * 6);
                const float2 u0 = __ldg(p2), u1 = __ldg(p2 + 1), u2 = __ldg(p2 + 2);
                fa[0] = u0.x; fa[1] = u0.y; fa[2] = u1.x; fa[3] = u1.y; fa[4] = u2.x; fa[5] = u2.y;
                const float4 v0 = __ldg(reinterpret_cast<const float4*>(f2 + m * 8)), v1 = __ldg(reinterpret_cast<const float4*>(f2 + m * 8) + 1);
                fb[0] = v0.x; fb[1] = v0.y; fb[2] = v0.z; fb[3] = v0.w; fb[4] = v1.x; fb[5] = v1.y; fb[6] = v1.z; fb[7] = v1.w;
            }
#pragma unroll
            for (int j = 0; j < 8; j++) {
                float o1[4], o2[4];
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    const int col = cg * 32 + j * 4 + c;
                    const float2 wa = *reinterpret_cast<const float2*>(s_w1p + col * 6), wb = *reinterpret_cast<const float2*>(s_w1p + col * 6 + 2),
                                 wc = *reinterpret_cast<const float2*>(s_w1p + col * 6 + 4);
                    o1[c] = to_tf32(fmaf(fa[5], wc.y, fmaf(fa[4], wc.x, fmaf(fa[3], wb.y, fmaf(fa[2], wb.x, fmaf(fa[1], wa.y, fa[0] * wa.x))))));
                    const float4 xa = *reinterpret_cast<const float4*>(s_w2p + col * 8), xb = *reinterpret_cast<const float4*>(s_w2p + col * 8 + 4);
                    o2[c] = to_tf32(fmaf(fb[7], xb.w, fmaf(fb[6], xb.z, fmaf(fb[5], xb.y, fmaf(fb[4], xb.x,
                                    fmaf(fb[3], xa.w, fmaf(fb[2], xa.z, fmaf(fb[1], xa.y, fb[0] * xa.x))))))));
                }
                *reinterpret_cast<float4*>(reinterpret_cast<char*>(sA1) + arow + j * 128) = make_float4(o1[0], o1[1], o1[2], o1[3]);
                *reinterpret_cast<float4*>(reinterpret_cast<char*>(sA2) + arow + j * 128) = make_float4(o2[0], o2[1], o2[2], o2[3]);
            }
        }
#pragma unroll 1
        for (int layer = 0; layer < 3; layer++) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            if (tid == 0) {
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a1 = smem_u32(sA1), a2 = smem_u32(sA2), aW = smem_u32(sW);
#pragma unroll
                for (int k = 0; k < 16; k++)
                    umma_tf32(tmem_base, make_desc(a1 + k * 256, 128, 4096), make_desc(aW + k * 256, 128, 4096), k > 0 ? 1u : 0u);
#pragma unroll
                for (int k = 0; k < 16; k++)
                    umma_tf32(tmem_base + TILE_N, make_desc(a2 + k * 256, 128, 4096), make_desc(aW + k * 256, 128, 4096), k > 0 ? 1u : 0u);
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
            }
            mbar_wait(bar, phase);
            phase ^= 1;
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            uint32_t r1[32], r2[32];
            TMEM_LD32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(cg * 32), r1);
            TMEM_LD32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(TILE_N + cg * 32), r2);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            float ps = 0.f, pd1 = 0.f, pd2 = 0.f;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const float4 va = *reinterpret_cast<const float4*>(s_as + cg * 32 + 4 * j), vd = *reinterpret_cast<const float4*>(s_ad + cg * 32 + 4 * j);
                const float x0 = __uint_as_float(r1[4 * j]), x1 = __uint_as_float(r1[4 * j + 1]), x2 = __uint_as_float(r1[4 * j + 2]),
                            x3 = __uint_as_float(r1[4 * j + 3]);
                const float y0 = __uint_as_float(r2[4 * j]), y1 = __uint_as_float(r2[4 * j + 1]), y2 = __uint_as_float(r2[4 * j + 2]),
                            y3 = __uint_as_float(r2[4 * j + 3]);
                ps = fmaf(x3, va.w, fmaf(x2, va.z, fmaf(x1, va.y, fmaf(x0, va.x, ps))));
                pd1 = fmaf(x3, vd.w, fmaf(x2, vd.z, fmaf(x1, vd.y, fmaf(x0, vd.x, pd1))));
                pd2 = fmaf(y3, vd.w, fmaf(y2, vd.z, fmaf(y1, vd.y, fmaf(y0, vd.x, pd2))));
            }
            s_dot[(0 * 4 + cg) * 128 + mloc] = ps;
            s_dot[(1 * 4 + cg) * 128 + mloc] = pd1;
            s_dot[(2 * 4 + cg) * 128 + mloc] = pd2;
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            const float s1 = (s_dot[0 * 128 + mloc] + s_dot[1 * 128 + mloc]) + (s_dot[2 * 128 + mloc] + s_dot[3 * 128 + mloc]);
            const float d1 = (s_dot[4 * 128 + mloc] + s_dot[5 * 128 + mloc]) + (s_dot[6 * 128 + mloc] + s_dot[7 * 128 + mloc]);
            const float d2 = (s_dot[8 * 128 + mloc] + s_dot[9 * 128 + mloc]) + (s_dot[10 * 128 + mloc] + s_dot[11 * 128 + mloc]);
            float e11 = s1 + d1, e12 = s1 + d2;
            e11 = e11 > 0.f ? e11 : 0.2f * e11;
            e12 = e12 > 0.f ? e12 : 0.2f * e12;
            const float mx = fmaxf(e11, e12);
            const float p1 = expf(e11 - mx), p2 = expf(e12 - mx);
            const float a0 = p1 / (p1 + p2), a1 = p2 / (p1 + p2);
            if (layer < 2) {  // next layer's operands: elu(h1'), elu(h2') back into the A buffers (the products are done with them)
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    float4 x, y;
                    y.x = __uint_as_float(r2[4 * j]); y.y = __uint_as_float(r2[4 * j + 1]); y.z = __uint_as_float(r2[4 * j + 2]); y.w = __uint_as_float(r2[4 * j + 3]);
                    x.x = a0 * __uint_as_float(r1[4 * j]) + a1 * y.x; x.y = a0 * __uint_as_float(r1[4 * j + 1]) + a1 * y.y;
                    x.z = a0 * __uint_as_float(r1[4 * j + 2]) + a1 * y.z; x.w = a0 * __uint_as_float(r1[4 * j + 3]) + a1 * y.w;
                    x.x = to_tf32(elu_fast(x.x)); x.y = to_tf32(elu_fast(x.y)); x.z = to_tf32(elu_fast(x.z)); x.w = to_tf32(elu_fast(x.w));
                    y.x = to_tf32(elu_fast(y.x)); y.y = to_tf32(elu_fast(y.y)); y.z = to_tf32(elu_fast(y.z)); y.w = to_tf32(elu_fast(y.w));
                    *reinterpret_cast<float4*>(reinterpret_cast<char*>(sA1) + arow + j * 128) = x;
                    *reinterpret_cast<float4*>(reinterpret_cast<char*>(sA2) + arow + j * 128) = y;
                }
            } else {  // mean over the two node sets, written out; column sums for the BatchNorm that follows
                float4* op = reinterpret_cast<float4*>(out + m * 128 + cg * 32);
                float o[32];
#pragma unroll
                for (int j = 0; j < 32; j++) {
                    const float y = __uint_as_float(r2[j]);
                    o[j] = mok ? 0.5f * ((a0 * __uint_as_float(r1[j]) + a1 * y) + y) : 0.f;
                }
                if (mok) {
#pragma unroll
                    for (int j = 0; j < 8; j++) op[j] = make_float4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
                }
                if (GROUPED) {  // row mloc of the tile, 16-byte pieces XOR-swizzled by the row (the products are done with sA1)
#pragma unroll
                    for (int j = 0; j < 8; j++)
                        *reinterpret_cast<float4*>(sA1 + mloc * 128 + (((cg * 8 + j) ^ (mloc & 7)) << 2)) =
                            make_float4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
                }
                if (!GROUPED && stats) {  // recursive halving over the warp's 32 machines: lane l ends up with column cg * 32 + l
                    float q[32];
#pragma unroll
                    for (int j = 0; j < 32; j++) q[j] = o[j] * o[j];
#pragma unroll
                    for (int off = 16, n = 16; off >= 1; off >>= 1, n >>= 1) {
                        const bool up = (lane & off) != 0;
#pragma unroll
                        for (int j = 0; j < n; j++) {
                            const float so = up ? o[j] : o[j + n], ko = up ? o[j + n] : o[j];
                            const float sq = up ? q[j] : q[j + n], kq = up ? q[j + n] : q[j];
                            o[j] = ko + __shfl_xor_sync(0xffffffffu, so, off);
                            q[j] = kq + __shfl_xor_sync(0xffffffffu, sq, off);
                        }
                    }
                    st_sum += (double)o[0];
                    st_sq += (double)q[0];
                }
            }
        }
        __syncthreads();  // s_dot and the A buffers are rewritten by the next tile
        if (GROUPED) {    // the tile's rows are parked in sA1 (the barrier above): per-env sums in row order, FP64
            const long long row0 = tile * rpt, env0 = row0 / M;
            const int nenv = (int)(R - row0 < rpt ? R - row0 : rpt) / M;
            for (int item = tid; item < nenv * 128; item += TRUNK_WARPS * 32) {
                const int e = item >> 7, c = item & 127;
                double sum = 0.0, sq = 0.0;
                for (int j = 0; j < M; j++) {
                    const int r = e * M + j;
                    const double v = (double)sA1[r * 128 + ((((c >> 2) ^ (r & 7))) << 2) + (c & 3)];
                    sum += v;
                    sq = fma(v, v, sq);
                }
                stats[(env0 + e) * 256 + c] = sum;
                stats[(env0 + e) * 256 + 128 + c] = sq;
            }
            __syncthreads();  // sA1 is the next tile's operand
        }
    }
    if (!GROUPED && stats) {
        atomicAdd(stats + cg * 32 + lane, st_sum);
        atomicAdd(stats + 128 + cg * 32 + lane, st_sq);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256));
}


// =====================================================================================================================
// ESA machine actor (model/actor_critic.py:1207-1404 esa_Machine_Actor) in two launches.  Its per-row network is
//     h1 = BN(f1 W1^T), h2 = BN(f2 W2^T)  (one BatchNorm module, statistics of each call over its own R rows)
//     s  = 10 ( tanh( tanh( W0 cat(h1, h2, pooled, h_pooled_o) + b0 ) W1m^T + b1 ) . w2 + b2 )
// BatchNorm is a per-column affine and both projections are linear, so the per-row part of the first layer is ONE K = 14
// product on the raw features: W0a diag(sc1) W1 f1 + W0b diag(sc2) W2 f2, the shifts join the per-env bias.  The column
// statistics follow from the feature moments: mean_c = w_c . mu_f, var_c = w_c^T Sigma_f w_c.
//
// esa_stats_kernel: feature sums and second moments (the 6 x 6 and 8 x 8 blocks) in FP64, plus the per-env feature means.
// A CTA stages whole envs (<= 256 rows) of both feature sets in shared memory; thread (m, half) owns moment m over every
// other row; the CTA's partial goes to workspace[blockIdx] and esa_stats_reduce_kernel adds the partials in block order,
// so the moments do not depend on scheduling.
constexpr int ESA_MOMENTS = 14 + 36 + 64, ESA_STATS_THREADS = 256, ESA_STATS_ROWS = 256, ESA_STATS_BLOCKS = 592;

__global__ void __launch_bounds__(ESA_STATS_THREADS) esa_stats_kernel(const float* __restrict__ f1, const float* __restrict__ f2,
                                                                       long long B, int M, int epc, double* __restrict__ parts,
                                                                       float* __restrict__ env_mean) {
    __shared__ float s_f[ESA_STATS_ROWS * 14];
    __shared__ double s_acc[128];
    const int tid = threadIdx.x, mom = tid & 127, half = tid >> 7;
    // moment `mom`: < 14 column sum, < 50 f1 block (i, j), < 114 f2 block (i, j); columns 0..5 = f1, 6..13 = f2
    int ca = 0, cb = -1;
    if (mom < 14) ca = mom;
    else if (mom < 50) { ca = (mom - 14) / 6; cb = (mom - 14) % 6; }
    else if (mom < ESA_MOMENTS) { ca = 6 + (mom - 50) / 8; cb = 6 + (mom - 50) % 8; }
    double acc = 0.0;
    const long long chunks = (B + epc - 1) / epc;
    for (long long ch = blockIdx.x; ch < chunks; ch += gridDim.x) {
        const long long e0 = ch * epc;
        const int ne = (int)(B - e0 < epc ? B - e0 : epc), nr = ne * M;
        const long long r0 = e0 * M;
        __syncthreads();  // the previous chunk's readers are done
        for (int i = tid; i < nr * 6; i += ESA_STATS_THREADS) s_f[(i / 6) * 14 + i % 6] = __ldg(f1 + r0 * 6 + i);
        for (int i = tid; i < nr * 8; i += ESA_STATS_THREADS) s_f[(i / 8) * 14 + 6 + i % 8] = __ldg(f2 + r0 * 8 + i);
        __syncthreads();
        if (mom < ESA_MOMENTS) {
            if (cb < 0) {
                for (int r = half; r < nr; r += 2) acc += (double)s_f[r * 14 + ca];
            } else {
                for (int r = half; r < nr; r += 2) acc = fma((double)s_f[r * 14 + ca], (double)s_f[r * 14 + cb], acc);
            }
        }
        for (int i = tid; i < ne * 16; i += ESA_STATS_THREADS) {  // per-env means, [B,16] with two zero columns
            const int e = i >> 4, c = i & 15;
            double s = 0.0;
            if (c < 14)
                for (int m = 0; m < M; m++) s += (double)s_f[(e * M + m) * 14 + c];
            env_mean[(e0 + e) * 16 + c] = (float)(s / M);
        }
    }
    if (half == 1) s_acc[mom] = acc;
    __syncthreads();
    if (half == 0) parts[(size_t)blockIdx.x * 128 + mom] = acc + s_acc[mom];
}

__global__ void esa_stats_reduce_kernel(const double* __restrict__ parts, int nparts, double* __restrict__ moments) {
    const int m = threadIdx.x;
    if (m >= ESA_MOMENTS) return;
    double t = 0.0;
    for (int c = 0; c < nparts; c++) t += parts[(size_t)c * 128 + m];
    moments[m] = t;
}

// esa_fold_kernel: moments -> BatchNorm affine of both calls -> folded first-layer weights, one thread per hidden column
// c, FP64 throughout:  sc = gamma / sqrt(w_c^T Sigma w_c + eps), sh = beta - (w_c . mu) sc,  A = diag(sc) W  (so
// BN(f W^T) = f A^T + sh);  Wf = [W0a A1 | W0b A2 | 0 0],  b0f = b0 + W0a sh1 + W0b sh2,  Wp = [A1 | A2 | 0 0] / 2,
// bp = (sh1 + sh2) / 2  (the mean over machines commutes with the affine: pooled = env_mean Wp^T + bp).
__global__ void __launch_bounds__(128) esa_fold_kernel(const double* __restrict__ moments, double inv_rows, const float* __restrict__ W1,
                                                       const float* __restrict__ W2, const float* __restrict__ gamma,
                                                       const float* __restrict__ beta, float eps, const float* __restrict__ W0,
                                                       const float* __restrict__ b0, float* __restrict__ Wf, float* __restrict__ Wp,
                                                       float* __restrict__ bp, float* __restrict__ b0f) {
    __shared__ double s_m[ESA_MOMENTS];
    __shared__ double s_A[128][15];
    __shared__ double s_sh[2][128];
    const int c = threadIdx.x;
    if (c < ESA_MOMENTS) s_m[c] = moments[c] * inv_rows;
    __syncthreads();
    double sh[2];
#pragma unroll
    for (int set = 0; set < 2; set++) {
        const int K = set ? 8 : 6, off = set ? 6 : 0;
        const double* S = s_m + (set ? 50 : 14);
        const float* W = (set ? W2 : W1) + c * K;
        double mean = 0.0, var = 0.0;
        for (int i = 0; i < K; i++) {
            const double wi = W[i];
            mean += wi * s_m[off + i];
            for (int j = 0; j < K; j++) var += wi * (double)W[j] * (S[i * K + j] - s_m[off + i] * s_m[off + j]);
        }
        const double sc = (double)gamma[c] / sqrt(fmax(var, 0.0) + (double)eps);
        sh[set] = (double)beta[c] - mean * sc;
        for (int i = 0; i < K; i++) s_A[c][off + i] = sc * (double)W[i];
        s_sh[set][c] = sh[set];
    }
    for (int k = 0; k < 16; k++) Wp[c * 16 + k] = k < 14 ? (float)(0.5 * s_A[c][k]) : 0.f;
    bp[c] = (float)(0.5 * (sh[0] + sh[1]));
    __syncthreads();
    double acc[14], accb = (double)b0[c];
#pragma unroll
    for (int k = 0; k < 14; k++) acc[k] = 0.0;
    const float* w0 = W0 + (size_t)c * 512;
    for (int j = 0; j < 128; j++) {
        const double a = w0[j], b = w0[128 + j];
#pragma unroll
        for (int k = 0; k < 6; k++) acc[k] = fma(a, s_A[j][k], acc[k]);
#pragma unroll
        for (int k = 6; k < 14; k++) acc[k] = fma(b, s_A[j][k], acc[k]);
        accb = fma(a, s_sh[0][j], fma(b, s_sh[1][j], accb));
    }
    for (int k = 0; k < 16; k++) Wf[c * 16 + k] = k < 14 ? (float)acc[k] : 0.f;
    b0f[c] = (float)accb;
}

// esa_head_tf32_kernel: the machine policy head per 128-row tile, both products on tcgen05.mma kind::tf32:
//   D1 = [f1 | f2 | 0 0] W0f^T (K = 16, W0f = the folded first-layer weights [128,16]) -> TMEM columns 0..127;
//   epilogue 1: + bias_env[r / M], tanh, into the A buffer of the second product;  D2 = A2 W1^T -> TMEM 128..255;
//   epilogue 2: + b1, tanh, . w2, + b2, x 10 -> one float per row.
// The structure of head_tf32_kernel with its first product replaced: the rows are 56 bytes of raw features instead of
// a gathered 512-byte embedding, so no [R,128] tensor is read or written.
constexpr int ESA_HEAD_WARPS = 16;

__global__ void __launch_bounds__(ESA_HEAD_WARPS * 32, 1) esa_head_tf32_kernel(
    const float* __restrict__ f1, const float* __restrict__ f2, long long rows, int M, const float* __restrict__ W0f,
    const float* __restrict__ bias_env, const float* __restrict__ W1, const float* __restrict__ b1,
    const float* __restrict__ w2, const float* __restrict__ b2, float* __restrict__ out, long long num_tiles) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr size_t WBYTES = (size_t)TILE_N * 128 * 4, SBYTES = (size_t)TILE_M * 16 * 4;
    float* sW1 = reinterpret_cast<float*>(smem);
    float* sA2 = reinterpret_cast<float*>(smem + WBYTES);
    float* sW0 = reinterpret_cast<float*>(smem + 2 * WBYTES);
    float* sA1 = reinterpret_cast<float*>(smem + 2 * WBYTES + SBYTES);
    float* s_part = reinterpret_cast<float*>(smem + 2 * WBYTES + 2 * SBYTES);  // [4][128] partial dots of epilogue 2
    float* s_b1 = s_part + 4 * 128;
    float* s_w2 = s_b1 + 128;
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_w2 + 128);
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid < 128) {
        s_b1[tid] = b1 ? b1[tid] : 0.f;
        s_w2[tid] = w2[tid];
    }
    if (tid == 0) {
        mbar_init(smem_u32(s_bar + 0), 1);
        mbar_init(smem_u32(s_bar + 1), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(256));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    stage_block<false, ESA_HEAD_WARPS>(sW1, W1, 0, TILE_N, 128, 128, 128, nullptr, nullptr, false, warp, lane);
    stage_block<false, ESA_HEAD_WARPS>(sW0, W0f, 0, TILE_N, 16, 16, 16, nullptr, nullptr, false, warp, lane);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *s_tmem;
    const uint32_t bar0 = smem_u32(s_bar), bar1 = smem_u32(s_bar + 1);
    const float b2v = b2 ? __ldg(b2) : 0.f;

    // A1 staging: thread -> (tile row tid / 4, 16-byte piece tid % 4 = features 4p .. 4p+3), UMMA K-major layout with
    // SBO = 512 (8 rows x 4 pieces); features 0..5 from f1, 6..13 from f2, 14..15 zero
    const int arow = tid >> 2, apiece = tid & 3;
    char* const a1dst = reinterpret_cast<char*>(sA1) + (arow >> 3) * 512 + apiece * 128 + (arow & 7) * 16;
    float v[4];
    auto fetch = [&](long long tile) {
        const long long r = tile * TILE_M + arow;
        const bool ok = tile < num_tiles && r < rows;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int k = apiece * 4 + j;
            v[j] = !ok ? 0.f : k < 6 ? __ldg(f1 + r * 6 + k) : k < 14 ? __ldg(f2 + r * 8 + (k - 6)) : 0.f;
        }
    };
    auto mma = [&](const float* sA, const float* sW, int ksteps, uint32_t sbo, uint32_t dcol) {  // one elected thread
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t aA = smem_u32(sA), aW = smem_u32(sW);
        for (int k = 0; k < ksteps; k++)
            umma_tf32(tmem_base + dcol, make_desc(aA + k * 256, 128, sbo), make_desc(aW + k * 256, 128, sbo), k > 0 ? 1u : 0u);
    };

    const int quad = warp & 3, cg = warp >> 2;  // this warp's TMEM lanes 32 quad .., columns 32 cg ..
    const int trow = quad * 32 + lane;          // its thread's tile row
    fetch(blockIdx.x);
    long long i = 0;
    for (long long tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, i++) {
        const uint32_t par = (uint32_t)(i & 1);
        *reinterpret_cast<float4*>(a1dst) = make_float4(to_tf32(v[0]), to_tf32(v[1]), to_tf32(v[2]), to_tf32(v[3]));
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (tid == 0) {
            mma(sA1, sW0, 2, 512, 0);
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar0) : "memory");
        }
        fetch(tile + gridDim.x);  // the next tile's features travel while this tile is multiplied
        mbar_wait(bar0, par);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const long long grow = tile * TILE_M + trow;
        const bool rok = grow < rows;
        {   // first epilogue: + per-env bias, tanh, into A2 as the second product's operand
            uint32_t r[32];
            TMEM_LD32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(cg * 32), r);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            const long long brow = rok ? grow / M : 0;
            const float4* bp = reinterpret_cast<const float4*>(bias_env + brow * 128 + cg * 32);
            char* dst = reinterpret_cast<char*>(sA2) + (trow >> 3) * 4096 + (cg * 8) * 128 + (trow & 7) * 16;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const float4 bb = __ldg(bp + j);
                float4 x;
                x.x = to_tf32(tanh_fast(__uint_as_float(r[4 * j]) + bb.x)); x.y = to_tf32(tanh_fast(__uint_as_float(r[4 * j + 1]) + bb.y));
                x.z = to_tf32(tanh_fast(__uint_as_float(r[4 * j + 2]) + bb.z)); x.w = to_tf32(tanh_fast(__uint_as_float(r[4 * j + 3]) + bb.w));
                if (!rok) x = make_float4(0.f, 0.f, 0.f, 0.f);
                *reinterpret_cast<float4*>(dst + j * 128) = x;
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (tid == 0) {
            mma(sA2, sW1, 16, 4096, TILE_N);
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar1) : "memory");
        }
        mbar_wait(bar1, par);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        {   // second epilogue: + b1, tanh, dot with w2 over this warp's 32 columns
            uint32_t r[32];
            TMEM_LD32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(TILE_N + cg * 32), r);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            float acc = 0.f;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const float4 bb = *reinterpret_cast<const float4*>(s_b1 + cg * 32 + 4 * j);
                const float4 ww = *reinterpret_cast<const float4*>(s_w2 + cg * 32 + 4 * j);
                acc = fmaf(tanh_fast(__uint_as_float(r[4 * j]) + bb.x), ww.x, acc);
                acc = fmaf(tanh_fast(__uint_as_float(r[4 * j + 1]) + bb.y), ww.y, acc);
                acc = fmaf(tanh_fast(__uint_as_float(r[4 * j + 2]) + bb.z), ww.z, acc);
                acc = fmaf(tanh_fast(__uint_as_float(r[4 * j + 3]) + bb.w), ww.w, acc);
            }
            s_part[cg * 128 + trow] = acc;
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (tid < 128) {
            const long long orow = tile * TILE_M + tid;
            if (orow < rows) out[orow] = 10.f * (((s_part[tid] + s_part[128 + tid]) + (s_part[256 + tid] + s_part[384 + tid])) + b2v);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256));
}

// Operand alignment, checked on the host before any launch: cp.async, TMA and the float4 loads / stores move 16 bytes at a
// time, adj_w and fea1 are read as float2.  NULL passes (optional pointers are checked for presence separately).
template <class... P>
bool al16(P... p) { return ((((uintptr_t)p & 15) == 0) && ...); }
bool al8(const void* p) { return ((uintptr_t)p & 7) == 0; }

}  // namespace

// nodes > 0: the grouped form (env-aligned tiles of `nodes`-row envs, per-env statistics; see linear_tf32_kernel)
template <int KP, bool GROUPED = false>
static int launch_linear(const float* X, int64_t rows, int K, const float* W, const float* bias, const float* in_scale,
                         const float* in_shift, int in_relu, float* Z, double* stats, cudaStream_t stream, int nodes = 0) {
    const size_t smem = (size_t)TILE_N * KP * 4 + (size_t)NSTAGE * TILE_M * (KP > 64 ? 64 : KP) * 4 +
                        (size_t)NEPI * 32 * STG_W * 4 + (TILE_N + 256) * 4 + (4 + NSTAGE) * 8 + 16;
    static thread_local bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(linear_tf32_kernel<KP, GROUPED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return MTFJSP_E_CUDA;
        configured = true;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int P = GROUPED ? (nodes + TILE_M - 1) / TILE_M : 1, rpt = GROUPED && P == 1 ? (TILE_M / nodes) * nodes : TILE_M;
    const long long tiles = GROUPED ? (P == 1 ? (rows + rpt - 1) / rpt : rows / nodes * P) : (rows + TILE_M - 1) / TILE_M;
    const int grid = (int)(tiles < sms ? tiles : sms);
    if constexpr (GROUPED)
        linear_tf32_kernel<KP, true><<<grid, GEMM_WARPS * 32, smem, stream>>>(X, rows, K, W, bias, nullptr, nullptr, 0, Z, stats,
                                                                             tiles, rpt, nodes, P);
    else
        linear_tf32_kernel<KP, false><<<grid, GEMM_WARPS * 32, smem, stream>>>(X, rows, K, W, bias, in_scale, in_shift, in_relu, Z,
                                                                              stats, tiles);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

// K = 128 through the TMA kernel (X 16-byte aligned, checked by the caller); returns 1 if launched, 0 if the driver entry
// point is not available (caller falls back)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        return (EncodeTiledFn)p;
    }();
    return fn;
}

static int launch_linear_tma(const float* X, int64_t rows, const float* W, const float* bias, const float* in_scale,
                             const float* in_shift, int in_relu, float* Z, double* stats, cudaStream_t stream) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return 0;
    CUtensorMap map;
    const cuuint64_t dims[2] = {128, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {512};
    const cuuint32_t box[2] = {32, 128};
    const cuuint32_t estr[2] = {1, 1};
    if (enc(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)X, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return 0;
    const size_t smem = (size_t)TILE_N * 128 * 4 + (size_t)NSTAGE * TILE_M * 64 * 4 + (size_t)NEPI * 32 * STG_W * 4 +
                        (TILE_N + 256) * 4 + (4 + 2 * NSTAGE) * 8 + 16 + 128 * 10;
    static thread_local bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(linear_tf32_tma_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return MTFJSP_E_CUDA;
        configured = true;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long tiles = (rows + TILE_M - 1) / TILE_M;
    const int grid = (int)(tiles < sms ? tiles : sms);
    linear_tf32_tma_kernel<false, false><<<grid, GEMM_WARPS * 32, smem, stream>>>(map, rows, W, bias, in_scale, in_shift, in_relu, Z, stats, tiles,
                                                                         TILE_M, 0, nullptr, nullptr);
    return cudaGetLastError() == cudaSuccess ? 1 : MTFJSP_E_CUDA;
}

// aggregation + layer in one launch (K = 128, N <= 128 nodes per env); 1 launched, 0 not available, < 0 error
static int launch_linear_tma_agg(const float* X, int64_t B, int N, const float* adj_w, const int16_t* adj_src, const float* W,
                                 const float* bias, const float* in_scale, const float* in_shift, int in_relu, float* Z,
                                 double* stats, cudaStream_t stream) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc || N > TILE_M) return 0;
    const int rpt = (TILE_M / N) * N;
    const long long rows = (long long)B * N;
    CUtensorMap map;
    const cuuint64_t dims[2] = {128, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {512};
    const cuuint32_t box[2] = {32, (cuuint32_t)rpt};
    const cuuint32_t estr[2] = {1, 1};
    if (enc(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)X, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return 0;
    const size_t smem = (size_t)TILE_N * 128 * 4 + (size_t)3 * TILE_M * 64 * 4 + (size_t)TILE_M * TILE_N * 4 + (TILE_N + 256) * 4 +
                        (4 + 2 * 3) * 8 + 16 + 128 * 10;
    static thread_local bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(linear_tf32_tma_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return MTFJSP_E_CUDA;
        configured = true;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long tiles = (rows + rpt - 1) / rpt;
    const int grid = (int)(tiles < sms ? tiles : sms);
    linear_tf32_tma_kernel<true, false><<<grid, GEMM_WARPS * 32, smem, stream>>>(map, rows, W, bias, in_scale, in_shift, in_relu, Z, stats, tiles, rpt,
                                                                        N, reinterpret_cast<const float2*>(adj_w), adj_src);
    return cudaGetLastError() == cudaSuccess ? 1 : MTFJSP_E_CUDA;
}

// the grouped K = 128 layers (both forms: agg = the aggregation + layer of launch_linear_tma_agg, nodes <= 128); in_scale /
// in_shift [G,128]; 1 launched, 0 TMA not available, < 0 error
static int launch_linear_tma_grouped(bool agg, const float* X, int64_t B, int N, const float* adj_w, const int16_t* adj_src,
                                     const float* W, const float* bias, const float* in_scale, const float* in_shift, int in_relu,
                                     int epg, float* Z, double* env_stats, cudaStream_t stream) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return 0;
    const int P = (N + TILE_M - 1) / TILE_M, rpt = P == 1 ? (TILE_M / N) * N : TILE_M;
    const long long rows = (long long)B * N;
    CUtensorMap map;
    const cuuint64_t dims[2] = {128, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {512};
    const cuuint32_t box[2] = {32, (cuuint32_t)rpt};
    const cuuint32_t estr[2] = {1, 1};
    if (enc(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)X, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return 0;
    const size_t smem_agg = (size_t)TILE_N * 128 * 4 + (size_t)3 * TILE_M * 64 * 4 + (size_t)TILE_M * TILE_N * 4 + (TILE_N + 256) * 4 +
                            (4 + 2 * 3) * 8 + 16 + 128 * 10;
    const size_t smem_lin = (size_t)TILE_N * 128 * 4 + (size_t)NSTAGE * TILE_M * 64 * 4 + (size_t)NEPI * 32 * STG_W * 4 +
                            (TILE_N + 256) * 4 + (4 + 2 * NSTAGE) * 8 + 16 + 128 * 10;
    static thread_local bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(linear_tf32_tma_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_agg) != cudaSuccess ||
            cudaFuncSetAttribute(linear_tf32_tma_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_lin) != cudaSuccess)
            return MTFJSP_E_CUDA;
        configured = true;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long tiles = P == 1 ? (rows + rpt - 1) / rpt : B * P;
    const int grid = (int)(tiles < sms ? tiles : sms);
    if (agg)
        linear_tf32_tma_kernel<true, true><<<grid, GEMM_WARPS * 32, smem_agg, stream>>>(
            map, rows, W, bias, in_scale, in_shift, in_relu, Z, env_stats, tiles, rpt, N, reinterpret_cast<const float2*>(adj_w), adj_src,
            P, epg);
    else
        linear_tf32_tma_kernel<false, true><<<grid, GEMM_WARPS * 32, smem_lin, stream>>>(
            map, rows, W, bias, in_scale, in_shift, in_relu, Z, env_stats, tiles, rpt, N, nullptr, nullptr, P, epg);
    return cudaGetLastError() == cudaSuccess ? 1 : MTFJSP_E_CUDA;
}

extern "C" {

int mtfjsp_enc_linear_tf32(const float* X, int64_t rows, int K, const float* W, const float* bias, const float* in_scale,
                           const float* in_shift, int in_relu, float* Z, double* stats, void* stream) {
    if (!X || !W || !Z || rows < 1 || K < 4 || K > 128 || (K % 4) != 0) return MTFJSP_E_ARG;
    if ((in_scale == nullptr) != (in_shift == nullptr)) return MTFJSP_E_ARG;
    if (!al16(X, W, Z) || !al8(stats)) return MTFJSP_E_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    if (K == 128 && rows >= 4096) {  // the big layers: A operand by TMA (falls through when the driver lacks the entry point)
        const int rc = launch_linear_tma(X, rows, W, bias, in_scale, in_shift, in_relu, Z, stats, s);
        if (rc != 0) return rc < 0 ? rc : MTFJSP_OK;
    }
    if (K <= 16) return launch_linear<16>(X, rows, K, W, bias, in_scale, in_shift, in_relu, Z, stats, s);
    if (K <= 32) return launch_linear<32>(X, rows, K, W, bias, in_scale, in_shift, in_relu, Z, stats, s);
    if (K <= 64) return launch_linear<64>(X, rows, K, W, bias, in_scale, in_shift, in_relu, Z, stats, s);
    return launch_linear<128>(X, rows, K, W, bias, in_scale, in_shift, in_relu, Z, stats, s);
}

int mtfjsp_enc_head_tf32(const float* X, const int32_t* cand, int64_t B, int rows_per_env, int nodes_per_env,
                         const float* in_scale, const float* in_shift, int in_relu, const float* Wa, const float* bias_env,
                         int64_t bias_rows, const float* W1, const float* b1, const float* w2, const float* b2, float* out,
                         void* stream) {
    if (!X || !Wa || !bias_env || !W1 || !w2 || !out || B < 1 || rows_per_env < 1) return MTFJSP_E_ARG;
    if ((in_scale == nullptr) != (in_shift == nullptr)) return MTFJSP_E_ARG;
    if (!al16(X, Wa, bias_env, W1)) return MTFJSP_E_ARG;
    if (bias_rows != 1 && bias_rows != B) return MTFJSP_E_ARG;
    if (cand && (nodes_per_env < 1 || (long long)B * nodes_per_env > 0x7fffffffLL)) return MTFJSP_E_ARG;
    const long long rows = (long long)B * rows_per_env;
    if (rows > 0x7fffffffLL) return MTFJSP_E_ARG;
    const size_t smem = 3 * (size_t)TILE_N * 128 * 4 + (4 * 128 + 4 * 128) * 4 + 256 * 4 + 2 * 8 + 16;
    static thread_local bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(head_tf32_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return MTFJSP_E_CUDA;
        configured = true;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long tiles = (rows + TILE_M - 1) / TILE_M;
    const int grid = (int)(tiles < sms ? tiles : sms);
    head_tf32_kernel<false><<<grid, HEAD_WARPS * 32, smem, (cudaStream_t)stream>>>(X, cand, rows, rows_per_env, nodes_per_env, in_scale,
                                                                          in_shift, in_relu, Wa, bias_env, bias_rows, W1, b1, w2, b2,
                                                                          out, tiles);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_gat_trunk_tf32(const float* fea1, const float* fea2, const float* W1p, const float* W2p, const float* Wt,
                              const float* a_src, const float* a_dst, float* out, double* stats, int64_t R, void* stream) {
    if (!fea1 || !fea2 || !W1p || !W2p || !Wt || !a_src || !a_dst || !out || R < 1) return MTFJSP_E_ARG;
    if (!al16(fea2, Wt, out) || !al8(fea1) || !al8(stats)) return MTFJSP_E_ARG;
    const size_t smem = 3 * (size_t)TILE_N * 128 * 4 + (3 * 4 * 128 + 256 + 128 * 14) * 4 + 8 + 16;
    static thread_local bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(gat_trunk2_tf32_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return MTFJSP_E_CUDA;
        configured = true;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long tiles = (R + 127) / 128;
    const int grid = (int)(tiles < sms ? tiles : sms);
    gat_trunk2_tf32_kernel<false><<<grid, TRUNK_WARPS * 32, smem, (cudaStream_t)stream>>>(fea1, fea2, W1p, W2p, Wt, a_src, a_dst, out,
                                                                                          stats, R, tiles, 128, 1);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_gat_trunk_tf32_grouped(const float* fea1, const float* fea2, const float* W1p, const float* W2p, const float* Wt,
                                      const float* a_src, const float* a_dst, float* out, double* env_stats, int64_t B, int M,
                                      void* stream) {
    if (!fea1 || !fea2 || !W1p || !W2p || !Wt || !a_src || !a_dst || !out || !env_stats || B < 1 || M < 1 || M > 128 ||
        B * M > 0x7fffff00LL)
        return MTFJSP_E_ARG;
    if (!al16(fea2, Wt, out) || !al8(fea1) || !al8(env_stats)) return MTFJSP_E_ARG;
    const size_t smem = 3 * (size_t)TILE_N * 128 * 4 + (3 * 4 * 128 + 256 + 128 * 14) * 4 + 8 + 16;
    static thread_local bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(gat_trunk2_tf32_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return MTFJSP_E_CUDA;
        configured = true;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int epT = 128 / M;  // whole envs per tile
    const long long tiles = (B + epT - 1) / epT;
    const int grid = (int)(tiles < sms ? tiles : sms);
    gat_trunk2_tf32_kernel<true><<<grid, TRUNK_WARPS * 32, smem, (cudaStream_t)stream>>>(fea1, fea2, W1p, W2p, Wt, a_src, a_dst, out,
                                                                                         env_stats, B * M, tiles, epT * M, M);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_aggregate_linear_tf32(const float* X, int64_t B, int N, const float* adj_w, const int16_t* adj_src, const float* W,
                                     const float* bias, const float* in_scale, const float* in_shift, int in_relu, float* Z,
                                     double* stats, void* stream) {
    if (!X || !adj_w || !adj_src || !W || !Z || B < 1 || N < 1) return MTFJSP_E_ARG;
    if ((in_scale == nullptr) != (in_shift == nullptr)) return MTFJSP_E_ARG;
    if (!al16(X, W, Z) || !al8(adj_w) || !al8(stats)) return MTFJSP_E_ARG;
    const int rc = launch_linear_tma_agg(X, B, N, adj_w, adj_src, W, bias, in_scale, in_shift, in_relu, Z, stats, (cudaStream_t)stream);
    if (rc == 0) return MTFJSP_E_STATE;  // not available for this size / driver: the caller runs the two kernels
    return rc < 0 ? rc : MTFJSP_OK;
}

static bool grouped_args_ok(int64_t B, int N, int epg) { return B >= 1 && N >= 1 && epg >= 1 && B % epg == 0 && B * N <= 0x7fffff00LL; }

int mtfjsp_enc_linear_tf32_grouped(const float* X, int64_t B, int rows_per_env, int K, const float* W, const float* bias,
                                   const float* in_scale, const float* in_shift, int in_relu, int envs_per_group, float* Z,
                                   double* env_stats, void* stream) {
    if (!X || !W || !Z || !env_stats || !grouped_args_ok(B, rows_per_env, envs_per_group)) return MTFJSP_E_ARG;
    if ((in_scale == nullptr) != (in_shift == nullptr)) return MTFJSP_E_ARG;
    if (!al16(X, W, Z, in_scale, in_shift) || !al8(env_stats)) return MTFJSP_E_ARG;
    if (K == 128) {
        const int rc = launch_linear_tma_grouped(false, X, B, rows_per_env, nullptr, nullptr, W, bias, in_scale, in_shift, in_relu,
                                                 envs_per_group, Z, env_stats, (cudaStream_t)stream);
        return rc == 0 ? MTFJSP_E_STATE : rc < 0 ? rc : MTFJSP_OK;
    }
    if (K < 4 || K > 16 || (K % 4) != 0 || in_scale) return MTFJSP_E_ARG;
    return launch_linear<16, true>(X, B * rows_per_env, K, W, bias, nullptr, nullptr, 0, Z, env_stats, (cudaStream_t)stream, rows_per_env);
}

int mtfjsp_enc_aggregate_linear_tf32_grouped(const float* X, int64_t B, int N, const float* adj_w, const int16_t* adj_src,
                                             const float* W, const float* bias, const float* in_scale, const float* in_shift,
                                             int in_relu, int envs_per_group, float* Z, double* env_stats, void* stream) {
    if (!X || !adj_w || !adj_src || !W || !Z || !env_stats || !grouped_args_ok(B, N, envs_per_group)) return MTFJSP_E_ARG;
    if ((in_scale == nullptr) != (in_shift == nullptr)) return MTFJSP_E_ARG;
    if (!al16(X, W, Z, in_scale, in_shift) || !al8(adj_w) || !al8(env_stats)) return MTFJSP_E_ARG;
    if (N > TILE_M) return MTFJSP_E_STATE;  // the caller runs mtfjsp_enc_aggregate_grouped + mtfjsp_enc_linear_tf32_grouped
    const int rc = launch_linear_tma_grouped(true, X, B, N, adj_w, adj_src, W, bias, in_scale, in_shift, in_relu, envs_per_group, Z,
                                             env_stats, (cudaStream_t)stream);
    return rc == 0 ? MTFJSP_E_STATE : rc < 0 ? rc : MTFJSP_OK;
}

int mtfjsp_enc_head_tf32_grouped(const float* X, const int32_t* cand, int64_t B, int rows_per_env, int nodes_per_env,
                                 const float* in_scale, const float* in_shift, int in_relu, int envs_per_group, const float* Wa,
                                 const float* bias_env, int64_t bias_rows, const float* W1, const float* b1, const float* w2,
                                 const float* b2, float* out, void* stream) {
    if (!X || !in_scale || !in_shift || !Wa || !bias_env || !W1 || !w2 || !out || B < 1 || rows_per_env < 1) return MTFJSP_E_ARG;
    if (envs_per_group < 1 || B % envs_per_group != 0) return MTFJSP_E_ARG;
    if (bias_rows != 1 && bias_rows != B) return MTFJSP_E_ARG;
    if (!al16(X, Wa, bias_env, W1, in_scale, in_shift)) return MTFJSP_E_ARG;
    if (cand && (nodes_per_env < 1 || (long long)B * nodes_per_env > 0x7fffffffLL)) return MTFJSP_E_ARG;
    const long long rows = (long long)B * rows_per_env;
    if (rows > 0x7fffffffLL) return MTFJSP_E_ARG;
    const size_t smem = 3 * (size_t)TILE_N * 128 * 4 + (4 * 128 + 4 * 128) * 4 + 256 * 4 + 2 * 8 + 16;
    static thread_local bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(head_tf32_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return MTFJSP_E_CUDA;
        configured = true;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long tiles = (rows + TILE_M - 1) / TILE_M;
    const int grid = (int)(tiles < sms ? tiles : sms);
    head_tf32_kernel<true><<<grid, HEAD_WARPS * 32, smem, (cudaStream_t)stream>>>(X, cand, rows, rows_per_env, nodes_per_env, in_scale,
                                                                                in_shift, in_relu, Wa, bias_env, bias_rows, W1, b1, w2,
                                                                                b2, out, tiles, envs_per_group);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_bn_finalize_grouped(const double* env_stats, int64_t B, int rows_per_env, int envs_per_group, const float* gamma,
                                   const float* beta, float eps, float* scale, float* shift, int C, void* stream) {
    if (!env_stats || !gamma || !beta || !scale || !shift || C < 1 || !grouped_args_ok(B, rows_per_env, envs_per_group))
        return MTFJSP_E_ARG;
    const long long G = B / envs_per_group;
    const int P = (rows_per_env + TILE_M - 1) / TILE_M;
    bn_finalize_grouped_kernel<<<(unsigned)((G * C + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        env_stats, G, P, envs_per_group, 1.0 / ((double)envs_per_group * rows_per_env), gamma, beta, eps, scale, shift, C);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_bn_finalize(const double* stats, int64_t rows, const float* gamma, const float* beta, float eps,
                           float* scale, float* shift, int C, void* stream) {
    if (!stats || !gamma || !beta || !scale || !shift || rows < 1 || C < 1) return MTFJSP_E_ARG;
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(stats, 1.0 / (double)rows, gamma, beta, eps, scale,
                                                                        shift, C);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int64_t mtfjsp_enc_esa_mach_stats_workspace_doubles(void) { return (int64_t)ESA_STATS_BLOCKS * 128; }

int mtfjsp_enc_esa_mach_stats(const float* fea1, const float* fea2, int64_t B, int M, double* moments, float* env_mean,
                              double* workspace, void* stream) {
    if (!fea1 || !fea2 || !moments || !env_mean || !workspace || B < 1 || M < 1 || M > ESA_STATS_ROWS) return MTFJSP_E_ARG;
    const int epc = ESA_STATS_ROWS / M;
    const long long chunks = (B + epc - 1) / epc;
    const int grid = (int)(chunks < ESA_STATS_BLOCKS ? chunks : ESA_STATS_BLOCKS);
    esa_stats_kernel<<<grid, ESA_STATS_THREADS, 0, (cudaStream_t)stream>>>(fea1, fea2, B, M, epc, workspace, env_mean);
    if (cudaGetLastError() != cudaSuccess) return MTFJSP_E_CUDA;
    esa_stats_reduce_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(workspace, grid, moments);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_esa_mach_fold(const double* moments, int64_t rows, const float* W1, const float* W2, const float* gamma,
                             const float* beta, float eps, const float* W0, const float* b0, float* Wf, float* Wp, float* bp,
                             float* b0f, void* stream) {
    if (!moments || !W1 || !W2 || !gamma || !beta || !W0 || !b0 || !Wf || !Wp || !bp || !b0f || rows < 1) return MTFJSP_E_ARG;
    esa_fold_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(moments, 1.0 / (double)rows, W1, W2, gamma, beta, eps, W0, b0, Wf, Wp, bp, b0f);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_esa_mach_head_tf32(const float* fea1, const float* fea2, int64_t B, int M, const float* W0f, const float* bias_env,
                                  const float* W1, const float* b1, const float* w2, const float* b2, float* out, void* stream) {
    if (!fea1 || !fea2 || !W0f || !bias_env || !W1 || !w2 || !out || B < 1 || M < 1) return MTFJSP_E_ARG;
    if (!al16(W0f, bias_env, W1)) return MTFJSP_E_ARG;
    const long long rows = (long long)B * M;
    const size_t smem = 2 * (size_t)TILE_N * 128 * 4 + 2 * (size_t)TILE_M * 16 * 4 + (4 * 128 + 2 * 128) * 4 + 2 * 8 + 16;
    static thread_local bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(esa_head_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return MTFJSP_E_CUDA;
        configured = true;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long tiles = (rows + TILE_M - 1) / TILE_M;
    const int grid = (int)(tiles < sms ? tiles : sms);
    esa_head_tf32_kernel<<<grid, ESA_HEAD_WARPS * 32, smem, (cudaStream_t)stream>>>(fea1, fea2, rows, M, W0f, bias_env, W1, b1, w2, b2,
                                                                                  out, tiles);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

}  // extern "C"

template <int NP>
static int launch_wgrad(const float* dY, const float* X, int64_t rows, int K, float* dW, float* db, float* ws, int sms,
                        cudaStream_t stream) {
    const size_t smem = (size_t)WG_NSTAGE * (16 + NP / 8) * WG_SBO + (size_t)WG_WARPS * 128 * 8 + (WG_NSTAGE + 1) * 8 + 16;
    static thread_local bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(wgrad_tf32_kernel<NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return MTFJSP_E_CUDA;
        configured = true;
    }
    const long long stages = (rows + WG_KS - 1) / WG_KS;
    const int grid = (int)(stages < sms ? stages : sms);
    float* parts = ws;
    float* dbparts = ws + (size_t)sms * TILE_M * NP;
    wgrad_tf32_kernel<NP><<<grid, WG_WARPS * 32, smem, stream>>>(dY, X, rows, K, parts, dbparts, stages);
    if (cudaGetLastError() != cudaSuccess) return MTFJSP_E_CUDA;
    wgrad_reduce_kernel<<<(TILE_M * K + 255) / 256, 256, 0, stream>>>(parts, dbparts, grid, NP, K, dW, db);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

static int wgrad_sms() {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}
static int wgrad_np(int K) { return K <= 16 ? 16 : K <= 32 ? 32 : K <= 64 ? 64 : 128; }

extern "C" {

int64_t mtfjsp_enc_wgrad_workspace_floats(int K) {
    if (K < 4 || K > 128) return 0;
    return (int64_t)wgrad_sms() * (TILE_M * wgrad_np(K) + 128);
}

int mtfjsp_enc_wgrad_tf32(const float* dY, const float* X, int64_t rows, int K, float* dW, float* db, float* workspace,
                          void* stream) {
    if (!dY || !X || !dW || !workspace || rows < 1 || K < 4 || K > 128 || (K % 4) != 0) return MTFJSP_E_ARG;
    if (!al16(dY, X, workspace)) return MTFJSP_E_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const int sms = wgrad_sms();
    switch (wgrad_np(K)) {
        case 16: return launch_wgrad<16>(dY, X, rows, K, dW, db, workspace, sms, s);
        case 32: return launch_wgrad<32>(dY, X, rows, K, dW, db, workspace, sms, s);
        case 64: return launch_wgrad<64>(dY, X, rows, K, dW, db, workspace, sms, s);
        default: return launch_wgrad<128>(dY, X, rows, K, dW, db, workspace, sms, s);
    }
}

}  // extern "C"
