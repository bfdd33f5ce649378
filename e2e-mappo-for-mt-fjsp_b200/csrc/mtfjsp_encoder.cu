// mtfjsp_encoder.cu -- encoder-side kernels for sm_100a: batched adjacency aggregation over the compact ELL
// adjacency the env kernel emits (no [B*N, B*N] COO matrix, no cuSPARSE).
//
// Replaces (reference file:line):
//   model/actor_critic.py:139-140, 155-156   dense adj -> to_sparse -> aggr_obs block-diagonal COO   (eliminated)
//   model/gcn_mlp.py:125                     torch.mm(Adj.double(), h.double())                       weighted neighbour sum, FP64
//   model/gcn_mlp.py:133-149                 degree via a second SpMM with ones                       fused (slot count)
//   model/gcn_mlp.py:192                     torch.sparse.mm(graph_pool, h)                           per-env mean over nodes
//
// Numerics: the reference forms the <= 3-term row sum and the division by the in-degree (self included) in FP64 and
// rounds once to FP32 for the MLP that follows.  This kernel uses FP32 fused multiply-adds and a correctly rounded
// FP32 division: at most 2 FP32 ulp from the reference value (tests: rtol 1e-6 against a dense FP64 product).  An
// FP64 version of the same gather was instruction-bound on the FP64/conversion pipes (1.46 ms per 128-channel layer
// at 2.36 M rows, 20 % of HBM peak); the layers downstream are FP32/TF32 GEMMs, so the extra bits were not observable.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mtfjsp.h"

namespace {

// one thread per (row, 4 channels): out[row] = (h[row] + wj*h[row-1] + wm*h[src]) / deg
// GROUPED: in_scale / in_shift [G,C], the affine of group (env0 + row / N) / epg
template <bool GROUPED>
__global__ void __launch_bounds__(256) aggregate_kernel(const float4* __restrict__ h, const float2* __restrict__ adj_w,
                                                        const int16_t* __restrict__ adj_src, float4* __restrict__ out,
                                                        unsigned total, int N, int C4, int c4_shift,
                                                        const float4* __restrict__ in_scale,
                                                        const float4* __restrict__ in_shift, int in_relu, long long env0 = 0,
                                                        int epg = 1) {
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;  // one thread per (row, 4 channels); total < 2^31
    if (idx >= total) return;
    const unsigned row = c4_shift >= 0 ? idx >> c4_shift : idx / (unsigned)C4;
    const unsigned c = idx - row * (unsigned)C4;
    const unsigned v = row % (unsigned)N;
    const float2 w = __ldg(adj_w + row);
    const int src = __ldg(adj_src + row);
    const bool hj = w.x != 0.f, hm = src >= 0;
    // the three gathers are independent: issue them together
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 xs = __ldg(h + idx);
    float4 xj = hj ? __ldg(h + (idx - (unsigned)C4)) : z4;
    float4 xm = hm ? __ldg(h + ((size_t)(row - v + (unsigned)src) * C4 + c)) : z4;
    if (in_scale) {  // BatchNorm (+ReLU) of the producing layer, folded into the gather
        const size_t ga = GROUPED ? (size_t)((env0 + row / (unsigned)N) / epg) * C4 + c : c;
        const float4 sc = __ldg(in_scale + ga), sh = __ldg(in_shift + ga);
        auto bn = [&](float4& x) {
            x.x = fmaf(x.x, sc.x, sh.x); x.y = fmaf(x.y, sc.y, sh.y); x.z = fmaf(x.z, sc.z, sh.z); x.w = fmaf(x.w, sc.w, sh.w);
            if (in_relu) { x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f); }
        };
        bn(xs);
        if (hj) bn(xj);
        if (hm) bn(xm);
    }
    // self + w_job * h[v-1] + w_mach * h[src], FP32 fused multiply-adds (the reference's dense bmm is FP32 as well),
    // then the mean over the neighbourhood (1, 2 or 3 members)
    float4 a;
    a.x = fmaf(w.y, xm.x, fmaf(w.x, xj.x, xs.x)); a.y = fmaf(w.y, xm.y, fmaf(w.x, xj.y, xs.y));
    a.z = fmaf(w.y, xm.z, fmaf(w.x, xj.z, xs.z)); a.w = fmaf(w.y, xm.w, fmaf(w.x, xj.w, xs.w));
    const int n = 1 + (hj ? 1 : 0) + (hm ? 1 : 0);
    if (n == 3) {
        a.x = __fdiv_rn(a.x, 3.f); a.y = __fdiv_rn(a.y, 3.f); a.z = __fdiv_rn(a.z, 3.f); a.w = __fdiv_rn(a.w, 3.f);
    } else if (n == 2) {
        a.x *= 0.5f; a.y *= 0.5f; a.z *= 0.5f; a.w *= 0.5f;
    }
    out[idx] = a;
}

// machine-successor index: adj_dst[b,u] = v with adj_src[b,v] == u, else -1 (a machine route gives every op at most
// one successor, so the gather below has at most one machine term as well)
__global__ void ell_invert_kernel(const int16_t* __restrict__ adj_src, int16_t* __restrict__ adj_dst, unsigned rows, int N) {
    const unsigned row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    const int src = adj_src[row];
    if (src >= 0) adj_dst[row - row % (unsigned)N + (unsigned)src] = (int16_t)(row % (unsigned)N);
}

// transpose of aggregate_kernel, again a gather: dL/dx[u] = g[u]/deg[u] + w_job[u+1]*g[u+1]/deg[u+1]
//                                                           + w_mach[d]*g[d]/deg[d],  d = adj_dst[u]
__global__ void __launch_bounds__(256) aggregate_bwd_kernel(const float4* __restrict__ g, const float2* __restrict__ adj_w,
                                                            const int16_t* __restrict__ adj_src,
                                                            const int16_t* __restrict__ adj_dst, float4* __restrict__ out,
                                                            unsigned total, int N, int C4, int c4_shift) {
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const unsigned row = c4_shift >= 0 ? idx >> c4_shift : idx / (unsigned)C4;
    const unsigned c = idx - row * (unsigned)C4;
    const unsigned v = row % (unsigned)N;
    auto inv_deg = [&](unsigned r, float2 w) {
        const int n = 1 + (w.x != 0.f ? 1 : 0) + (__ldg(adj_src + r) >= 0 ? 1 : 0);
        return n == 3 ? (1.0f / 3.0f) : n == 2 ? 0.5f : 1.0f;
    };
    const float2 w0 = __ldg(adj_w + row);
    const float s0 = inv_deg(row, w0);
    const float4 g0 = __ldg(g + idx);
    float4 a = make_float4(g0.x * s0, g0.y * s0, g0.z * s0, g0.w * s0);
    if (v + 1 < (unsigned)N) {
        const float2 w1 = __ldg(adj_w + row + 1);
        if (w1.x != 0.f) {
            const float s1 = w1.x * inv_deg(row + 1, w1);
            const float4 g1 = __ldg(g + idx + (unsigned)C4);
            a.x = fmaf(s1, g1.x, a.x); a.y = fmaf(s1, g1.y, a.y); a.z = fmaf(s1, g1.z, a.z); a.w = fmaf(s1, g1.w, a.w);
        }
    }
    const int d = __ldg(adj_dst + row);
    if (d >= 0) {
        const unsigned r2 = row - v + (unsigned)d;
        const float2 w2 = __ldg(adj_w + r2);
        const float s2 = w2.y * inv_deg(r2, w2);
        const float4 g2 = __ldg(g + ((size_t)r2 * C4 + c));
        a.x = fmaf(s2, g2.x, a.x); a.y = fmaf(s2, g2.y, a.y); a.z = fmaf(s2, g2.z, a.z); a.w = fmaf(s2, g2.w, a.w);
    }
    out[idx] = a;
}

// per-env mean over the N node rows (graph_pool average): one block per env, thread per channel
// GROUPED: in_scale / in_shift [G,C], the affine of group b / epg
template <bool GROUPED>
__global__ void graph_mean_kernel(const float* __restrict__ h, float* __restrict__ out, int N, int C,
                                  const float* __restrict__ in_scale, const float* __restrict__ in_shift, int in_relu, int epg = 1) {
    const long long b = blockIdx.x;
    const float inv = 1.0f / (float)N;  // the reference multiplies each row by the float32 value 1/N and sums
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float acc = 0.f;
        const long long ga = GROUPED ? (b / epg) * C + c : c;
        const float sc = in_scale ? in_scale[ga] : 1.f, sh = in_scale ? in_shift[ga] : 0.f;
        for (int v = 0; v < N; v++) {
            float x = h[(b * N + v) * C + c];
            if (in_scale) { x = x * sc + sh; if (in_relu) x = fmaxf(x, 0.f); }
            acc += inv * x;
        }
        out[b * C + c] = acc;
    }
}

// ---- grouped BatchNorm1d (+ReLU) with batch statistics, forward and backward ------------------------------------
// x [G, R, C] f32: G row groups (one per buffered step of a PPO minibatch), each normalised with its own statistics
// (the reference re-forwards one step at a time, so every step has its own BatchNorm batch: gcn_mlp.py:154, 248,
// actor_critic.py:434 inside the loops of ppo_algorithm.py:739-775).  HBM-bound: forward = one statistics pass
// (read x) + one apply pass (read x, write y); backward = one sums pass (read x, gy) + one apply pass (read x, gy,
// write dx).  Nothing but x is kept for the backward: y's sign (ReLU mask) is recomputed from x.
constexpr int BN_ROWS = 512;  // rows of one group per block

// column sums of (a, b) over this block's rows -> FP64 atomics into acc[g][0][C], acc[g][1][C]
// MODE 0: a = x - p, b = (x - p)^2 with p the group's first row (statistics, shifted so that E[a^2] - E[a]^2 does not
//         cancel when |mean| >> std);  MODE 1: a = g', b = g' * xhat (backward sums), g' = gy * [y > 0]
template <int MODE>
__global__ void __launch_bounds__(256) bn_reduce_kernel(const float4* __restrict__ x, const float4* __restrict__ gy,
                                                        const float* __restrict__ w, const float* __restrict__ b,
                                                        const float* __restrict__ mean, const float* __restrict__ rstd,
                                                        double* __restrict__ acc, long long R, int C4, int relu) {
    extern __shared__ double s_red[];  // [2][ty][C]
    const int g = blockIdx.y;
    const int cq = threadIdx.x % C4, ty = threadIdx.x / C4, ny = blockDim.x / C4;
    const long long r0 = (long long)blockIdx.x * BN_ROWS;
    const long long r1 = r0 + BN_ROWS < R ? r0 + BN_ROWS : R;
    const int C = C4 * 4;
    float4 sa = make_float4(0.f, 0.f, 0.f, 0.f), sb = sa;
    float4 mu = sa, rs = sa, ww = sa, bb = sa;
    if (MODE == 0) mu = __ldg(x + (size_t)g * R * C4 + cq);  // the shift p
    if (MODE == 1) {
        mu = reinterpret_cast<const float4*>(mean + (size_t)g * C)[cq];
        rs = reinterpret_cast<const float4*>(rstd + (size_t)g * C)[cq];
        ww = reinterpret_cast<const float4*>(w)[cq];
        bb = reinterpret_cast<const float4*>(b)[cq];
    }
    if (ty < ny) {
        for (long long r = r0 + ty; r < r1; r += ny) {
            const size_t i = ((size_t)g * R + r) * C4 + cq;
            const float4 v = __ldg(x + i);
            if (MODE == 0) {
                const float4 d = make_float4(v.x - mu.x, v.y - mu.y, v.z - mu.z, v.w - mu.w);
                sa.x += d.x; sa.y += d.y; sa.z += d.z; sa.w += d.w;
                sb.x = fmaf(d.x, d.x, sb.x); sb.y = fmaf(d.y, d.y, sb.y); sb.z = fmaf(d.z, d.z, sb.z); sb.w = fmaf(d.w, d.w, sb.w);
            } else {
                float4 d = __ldg(gy + i);
                const float4 xh = make_float4((v.x - mu.x) * rs.x, (v.y - mu.y) * rs.y, (v.z - mu.z) * rs.z, (v.w - mu.w) * rs.w);
                if (relu) {
                    if (!(fmaf(xh.x, ww.x, bb.x) > 0.f)) d.x = 0.f;
                    if (!(fmaf(xh.y, ww.y, bb.y) > 0.f)) d.y = 0.f;
                    if (!(fmaf(xh.z, ww.z, bb.z) > 0.f)) d.z = 0.f;
                    if (!(fmaf(xh.w, ww.w, bb.w) > 0.f)) d.w = 0.f;
                }
                sa.x += d.x; sa.y += d.y; sa.z += d.z; sa.w += d.w;
                sb.x = fmaf(d.x, xh.x, sb.x); sb.y = fmaf(d.y, xh.y, sb.y); sb.z = fmaf(d.z, xh.z, sb.z); sb.w = fmaf(d.w, xh.w, sb.w);
            }
        }
        double* pa = s_red + (size_t)ty * C + cq * 4;
        double* pb = s_red + (size_t)(ny + ty) * C + cq * 4;
        pa[0] = sa.x; pa[1] = sa.y; pa[2] = sa.z; pa[3] = sa.w;
        pb[0] = sb.x; pb[1] = sb.y; pb[2] = sb.z; pb[3] = sb.w;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 2 * C; c += blockDim.x) {
        const int which = c / C, col = c - which * C;
        double t = 0.0;
        for (int y = 0; y < ny; y++) t += s_red[(size_t)(which * ny + y) * C + col];
        atomicAdd(acc + ((size_t)g * 2 + which) * C + col, t);
    }
}

// acc holds the sums of x - p and (x - p)^2 with p = x[g, 0, c] (bn_reduce_kernel<0>)
__global__ void bn_stats_finalize_kernel(const double* __restrict__ acc, const float* __restrict__ x, long long R, double inv_rows,
                                         float eps, float* mean, float* rstd, int G, int C) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= G * C) return;
    const int g = i / C, c = i - g * C;
    const double m = acc[((size_t)g * 2) * C + c] * inv_rows;
    double var = acc[((size_t)g * 2 + 1) * C + c] * inv_rows - m * m;  // biased, as torch normalises in training mode
    if (var < 0) var = 0;
    mean[i] = (float)((double)__ldg(x + (size_t)g * R * C + c) + m);
    rstd[i] = (float)(1.0 / sqrt(var + (double)eps));
}

// MODE 0: y = relu?(xhat*w + b);  MODE 1: dx = (g' - (sg + xhat*sgx)/R) * rstd * w
template <int MODE>
__global__ void __launch_bounds__(256) bn_apply_kernel(const float4* __restrict__ x, const float4* __restrict__ gy,
                                                       const float* __restrict__ w, const float* __restrict__ b,
                                                       const float* __restrict__ mean, const float* __restrict__ rstd,
                                                       const double* __restrict__ sums, float4* __restrict__ out, long long R,
                                                       int C4, int relu, float inv_rows) {
    const int g = blockIdx.y;
    const int cq = threadIdx.x % C4, ty = threadIdx.x / C4, ny = blockDim.x / C4;
    if (ty >= ny) return;
    const int C = C4 * 4;
    const long long r0 = (long long)blockIdx.x * BN_ROWS;
    const long long r1 = r0 + BN_ROWS < R ? r0 + BN_ROWS : R;
    const float4 mu = reinterpret_cast<const float4*>(mean + (size_t)g * C)[cq];
    const float4 rs = reinterpret_cast<const float4*>(rstd + (size_t)g * C)[cq];
    const float4 ww = reinterpret_cast<const float4*>(w)[cq];
    const float4 bb = reinterpret_cast<const float4*>(b)[cq];
    float4 sg = make_float4(0.f, 0.f, 0.f, 0.f), sx = sg;
    if (MODE == 1) {
        const double* p0 = sums + ((size_t)g * 2) * C + cq * 4;
        const double* p1 = sums + ((size_t)g * 2 + 1) * C + cq * 4;
        sg = make_float4((float)(p0[0] * inv_rows), (float)(p0[1] * inv_rows), (float)(p0[2] * inv_rows), (float)(p0[3] * inv_rows));
        sx = make_float4((float)(p1[0] * inv_rows), (float)(p1[1] * inv_rows), (float)(p1[2] * inv_rows), (float)(p1[3] * inv_rows));
    }
    for (long long r = r0 + ty; r < r1; r += ny) {
        const size_t i = ((size_t)g * R + r) * C4 + cq;
        const float4 v = __ldg(x + i);
        const float4 xh = make_float4((v.x - mu.x) * rs.x, (v.y - mu.y) * rs.y, (v.z - mu.z) * rs.z, (v.w - mu.w) * rs.w);
        float4 y = make_float4(fmaf(xh.x, ww.x, bb.x), fmaf(xh.y, ww.y, bb.y), fmaf(xh.z, ww.z, bb.z), fmaf(xh.w, ww.w, bb.w));
        if (MODE == 0) {
            if (relu) { y.x = fmaxf(y.x, 0.f); y.y = fmaxf(y.y, 0.f); y.z = fmaxf(y.z, 0.f); y.w = fmaxf(y.w, 0.f); }
            out[i] = y;
        } else {
            float4 d = __ldg(gy + i);
            if (relu) {
                if (!(y.x > 0.f)) d.x = 0.f;
                if (!(y.y > 0.f)) d.y = 0.f;
                if (!(y.z > 0.f)) d.z = 0.f;
                if (!(y.w > 0.f)) d.w = 0.f;
            }
            out[i] = make_float4((d.x - (sg.x + xh.x * sx.x)) * (rs.x * ww.x), (d.y - (sg.y + xh.y * sx.y)) * (rs.y * ww.y),
                                 (d.z - (sg.z + xh.z * sx.z)) * (rs.z * ww.z), (d.w - (sg.w + xh.w * sx.w)) * (rs.w * ww.w));
        }
    }
}

// 4-stream generalised advantage estimation (algorithm/ppo_algorithm.py:438-536): per env and reward stream a
// backward scan over the buffered steps, delta = r + gamma*v_next - v, gae = delta + gamma*lambda*gae*(1-done).
// Layout [T,B,4] (stream innermost), one thread per (env, stream): every step's load/store is coalesced.
// Also accumulates sum / sum of squares per stream (FP64) for the block-wide advantage normalisation.
__global__ void gae4_kernel(const float* __restrict__ r, const float* __restrict__ v, const float* __restrict__ vn,
                            const float* __restrict__ done, float* __restrict__ adv, double* __restrict__ stats, int T,
                            long long B, float gamma, float lam) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double s = 0.0, q = 0.0;
    const int k = (int)(threadIdx.x & 3);  // blockDim.x is a multiple of 4, so idx % 4 == threadIdx.x % 4
    if (idx < B * 4) {
        const long long b = idx >> 2;
        float gae = 0.f;
        for (int t = T - 1; t >= 0; t--) {
            const long long o = (long long)t * B * 4 + idx;
            const float delta = r[o] + gamma * vn[o] - v[o];
            gae = delta + gamma * lam * gae * (1.0f - done[(long long)t * B + b]);
            adv[o] = gae;
            s += (double)gae;
            q += (double)gae * (double)gae;
        }
    }
    // lanes with equal k hold the same stream: reduce over the warp with stride-4 shuffles, one atomic per warp and stream
    for (int o = 16; o >= 4; o >>= 1) {
        s += __shfl_down_sync(0xffffffffu, s, o);
        q += __shfl_down_sync(0xffffffffu, q, o);
    }
    if ((threadIdx.x & 31) < 4 && stats) {
        atomicAdd(stats + k, s);
        atomicAdd(stats + 4 + k, q);
    }
}

// adv <- (adv - mean) / (std + 1e-5) per stream, std unbiased (torch.std), ppo_algorithm.py:485, 532
__global__ void adv_normalize_kernel(float* __restrict__ adv, const double* __restrict__ stats, double count, long long total) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int k = (int)(idx & 3);
    const double mean = stats[k] / count;
    double var = (stats[4 + k] - count * mean * mean) / (count - 1.0);
    if (var < 0) var = 0;
    adv[idx] = (float)(((double)adv[idx] - mean) / (sqrt(var) + 1e-5));
}


// ---------------------------------------------------------------------------------------------------------------------
// Rollout-path fusions of the machine actor and the policy heads (H = 128; one warp per row, one float4 per lane).
// Each replaces a chain of library elementwise / gemv / cat launches that re-read [rows,128] tensors between them.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float dot4(const float4 a, const float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
__device__ __forceinline__ float elu1(float x) { return x > 0.f ? x : expm1f(x); }

// GATLayer.forward on the fixed 2-node graph after the projection (model/gat.py:82-159): t = [t1; t2] ([2R,128]),
//   e11 = lrelu(t1.a_src + t1.a_dst), e12 = lrelu(t1.a_src + t2.a_dst), att = softmax(e11, e12),
//   h1' = att0 t1 + att1 t2, h2' = t2.
// mode 0: out [2R,128] = [h1'; h2'];  mode 1: out = [elu(h1'); elu(h2')] (input of the next layer, actor_critic.py:
// 400-418);  mode 2: out [R,128] = (h1' + h2') / 2 (mean over the two node sets, :420).
__global__ void __launch_bounds__(256) gat_attend_kernel(const float4* __restrict__ t, const float4* __restrict__ a_src,
                                                         const float4* __restrict__ a_dst, float4* __restrict__ out,
                                                         long long R, int mode) {
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= R) return;
    const float4 x1 = __ldg(t + row * 32 + lane), x2 = __ldg(t + (R + row) * 32 + lane);
    const float4 as = __ldg(a_src + lane), ad = __ldg(a_dst + lane);
    const float s1 = warp_sum(dot4(x1, as)), d1 = warp_sum(dot4(x1, ad)), d2 = warp_sum(dot4(x2, ad));
    float e11 = s1 + d1, e12 = s1 + d2;
    e11 = e11 > 0.f ? e11 : 0.2f * e11;
    e12 = e12 > 0.f ? e12 : 0.2f * e12;
    const float mx = fmaxf(e11, e12);
    const float p1 = expf(e11 - mx), p2 = expf(e12 - mx);
    const float a0 = p1 / (p1 + p2), a1 = p2 / (p1 + p2);
    float4 h1 = make_float4(a0 * x1.x + a1 * x2.x, a0 * x1.y + a1 * x2.y, a0 * x1.z + a1 * x2.z, a0 * x1.w + a1 * x2.w);
    float4 h2 = x2;
    if (mode == 2) {
        out[row * 32 + lane] = make_float4(0.5f * (h1.x + h2.x), 0.5f * (h1.y + h2.y), 0.5f * (h1.z + h2.z), 0.5f * (h1.w + h2.w));
        return;
    }
    if (mode == 1) {
        h1 = make_float4(elu1(h1.x), elu1(h1.y), elu1(h1.z), elu1(h1.w));
        h2 = make_float4(elu1(h2.x), elu1(h2.y), elu1(h2.z), elu1(h2.w));
    }
    out[row * 32 + lane] = h1;
    out[(R + row) * 32 + lane] = h2;
}

// Backward of gat_attend_kernel for the PPO update (torch autograd runs ~20 elementwise kernels per GAT layer there).
// g: gradient of the forward's output ([2R,128], or [R,128] in mode 2); recomputes the attention from t, writes
// dt [2R,128] and accumulates the gradients of a_src / a_dst per block (dparts [gridDim.x][2][128], summed by the caller).
__global__ void __launch_bounds__(256) gat_attend_bwd_kernel(const float4* __restrict__ t, const float4* __restrict__ a_src,
                                                             const float4* __restrict__ a_dst, const float4* __restrict__ g,
                                                             float4* __restrict__ dt, float* __restrict__ dparts, long long R,
                                                             int mode) {
    __shared__ float4 s_acc[8][2][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float4 as = __ldg(a_src + lane), ad = __ldg(a_dst + lane);
    float4 das = make_float4(0.f, 0.f, 0.f, 0.f), dad = das;
    const long long nw = (long long)gridDim.x * 8;
    for (long long row = (long long)blockIdx.x * 8 + warp; row < R; row += nw) {
        const float4 x1 = __ldg(t + row * 32 + lane), x2 = __ldg(t + (R + row) * 32 + lane);
        const float s1 = warp_sum(dot4(x1, as)), d1 = warp_sum(dot4(x1, ad)), d2 = warp_sum(dot4(x2, ad));
        const float r11 = s1 + d1, r12 = s1 + d2;
        const float e11 = r11 > 0.f ? r11 : 0.2f * r11, e12 = r12 > 0.f ? r12 : 0.2f * r12;
        const float mx = fmaxf(e11, e12);
        const float p1 = expf(e11 - mx), p2 = expf(e12 - mx);
        const float a0 = p1 / (p1 + p2), a1 = p2 / (p1 + p2);
        float4 gh1, gh2;
        if (mode == 2) {
            const float4 gv = __ldg(g + row * 32 + lane);
            gh1 = make_float4(0.5f * gv.x, 0.5f * gv.y, 0.5f * gv.z, 0.5f * gv.w);
            gh2 = gh1;
        } else {
            gh1 = __ldg(g + row * 32 + lane);
            gh2 = __ldg(g + (R + row) * 32 + lane);
            if (mode == 1) {  // out = elu(h): d/dh = 1 for h > 0, exp(h) otherwise
                const float4 h1 = make_float4(a0 * x1.x + a1 * x2.x, a0 * x1.y + a1 * x2.y, a0 * x1.z + a1 * x2.z, a0 * x1.w + a1 * x2.w);
                gh1.x *= h1.x > 0.f ? 1.f : expf(h1.x); gh1.y *= h1.y > 0.f ? 1.f : expf(h1.y);
                gh1.z *= h1.z > 0.f ? 1.f : expf(h1.z); gh1.w *= h1.w > 0.f ? 1.f : expf(h1.w);
                gh2.x *= x2.x > 0.f ? 1.f : expf(x2.x); gh2.y *= x2.y > 0.f ? 1.f : expf(x2.y);
                gh2.z *= x2.z > 0.f ? 1.f : expf(x2.z); gh2.w *= x2.w > 0.f ? 1.f : expf(x2.w);
            }
        }
        const float da0 = warp_sum(dot4(gh1, x1)), da1 = warp_sum(dot4(gh1, x2));
        const float mean = a0 * da0 + a1 * da1;
        const float de11 = a0 * (da0 - mean) * (r11 > 0.f ? 1.f : 0.2f), de12 = a1 * (da1 - mean) * (r12 > 0.f ? 1.f : 0.2f);
        const float ds1 = de11 + de12;
        dt[row * 32 + lane] = make_float4(a0 * gh1.x + ds1 * as.x + de11 * ad.x, a0 * gh1.y + ds1 * as.y + de11 * ad.y,
                                          a0 * gh1.z + ds1 * as.z + de11 * ad.z, a0 * gh1.w + ds1 * as.w + de11 * ad.w);
        dt[(R + row) * 32 + lane] = make_float4(a1 * gh1.x + gh2.x + de12 * ad.x, a1 * gh1.y + gh2.y + de12 * ad.y,
                                                a1 * gh1.z + gh2.z + de12 * ad.z, a1 * gh1.w + gh2.w + de12 * ad.w);
        das.x += ds1 * x1.x; das.y += ds1 * x1.y; das.z += ds1 * x1.z; das.w += ds1 * x1.w;
        dad.x += de11 * x1.x + de12 * x2.x; dad.y += de11 * x1.y + de12 * x2.y;
        dad.z += de11 * x1.z + de12 * x2.z; dad.w += de11 * x1.w + de12 * x2.w;
    }
    s_acc[warp][0][lane] = das;
    s_acc[warp][1][lane] = dad;
    __syncthreads();
    if (threadIdx.x < 64) {  // warps' partials in a fixed order: deterministic
        const int which = threadIdx.x >> 5;
        float4 a = s_acc[0][which][lane];
        for (int w = 1; w < 8; w++) {
            const float4 b = s_acc[w][which][lane];
            a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
        }
        reinterpret_cast<float4*>(dparts)[((size_t)blockIdx.x * 2 + which) * 32 + lane] = a;
    }
}


// Action selection of the rollout (algorithm/agent_func.py:22-63 select_action / sample_select_action): masked softmax over
// the <= 32 scores of an env, one draw from it (inverse CDF on a counter-based uniform keyed by (seed, step counter, env))
// or the arg-max, the log-probability of the drawn entry and, for the job actor, the candidate op behind the drawn job.
// One warp per env, lane j = entry j.  Replaces masked_fill + softmax + torch.multinomial (eleven validity / draw launches)
// + gather + log + gather: ~25 launches per actor and step.
__device__ __forceinline__ uint64_t sel_mix(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
__global__ void __launch_bounds__(256) select_kernel(const float* __restrict__ scores, const uint8_t* __restrict__ mask,
                                                     const int32_t* __restrict__ cand, float scale, int R, long long B, int greedy,
                                                     uint64_t seed, const int64_t* __restrict__ counter, int stream_id,
                                                     float* __restrict__ prob, int64_t* __restrict__ action,
                                                     float* __restrict__ log_a, int64_t* __restrict__ task) {
    const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (b >= B) return;
    const bool in = lane < R;
    const bool open = in && mask[b * R + lane] == 0;
    const float sc = open ? scores[b * R + lane] * scale : -INFINITY;
    float mx = sc;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    const float e = open ? expf(sc - mx) : 0.f;
    const float tot = warp_sum(e);
    const float p = tot > 0.f ? e / tot : 0.f;
    if (in) prob[b * R + lane] = p;
    int a;
    if (greedy) {
        const unsigned best = __ballot_sync(0xffffffffu, open && sc == mx);  // first entry that attains the maximum
        a = best ? __ffs(best) - 1 : 0;
    } else {
        // inclusive prefix sum of p over the lanes; the drawn entry is the first open one whose prefix exceeds u
        float c = p;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float t = __shfl_up_sync(0xffffffffu, c, o);
            if (lane >= o) c += t;
        }
        const uint64_t r = sel_mix(seed ^ sel_mix((uint64_t)b * 0x100000001B3ULL + (uint64_t)(*counter) * 0x9E3779B1ULL + (uint64_t)stream_id));
        const float total = __shfl_sync(0xffffffffu, c, 31);
        const float u = (float)(r >> 40) * (1.0f / 16777216.0f) * total;  // [0, total)
        const unsigned hit = __ballot_sync(0xffffffffu, open && c > u);
        const unsigned any = __ballot_sync(0xffffffffu, open);
        a = hit ? __ffs(hit) - 1 : (any ? 31 - __clz(any) : 0);  // rounding at the top end: the last open entry
    }
    const float pa = __shfl_sync(0xffffffffu, p, a);
    if (lane == 0) {
        action[b] = a;
        log_a[b] = logf(pa);
        if (task) task[b] = cand ? (int64_t)cand[b * R + a] : (int64_t)a;
    }
}

// Operand alignment, checked on the host before any launch: the kernels read and write 16 bytes (float4) or 8 bytes
// (float2: adj_w) at a time.  NULL passes (optional pointers are checked for presence separately).
template <class... P>
bool al16(P... p) { return ((((uintptr_t)p & 15) == 0) && ...); }
bool al8(const void* p) { return ((uintptr_t)p & 7) == 0; }

}  // namespace

extern "C" {

int mtfjsp_enc_select(const float* scores, const uint8_t* mask, const int32_t* cand, float scale, int R, int64_t B, int greedy,
                      uint64_t seed, const int64_t* counter, int stream_id, float* prob, int64_t* action, float* log_a,
                      int64_t* task, void* stream) {
    if (!scores || !mask || !prob || !action || !log_a || R < 1 || R > 32 || B < 1 || (!greedy && !counter)) return MTFJSP_E_ARG;
    select_kernel<<<(unsigned)((B + 7) / 8), 256, 0, (cudaStream_t)stream>>>(scores, mask, cand, scale, R, B, greedy, seed, counter,
                                                                           stream_id, prob, action, log_a, task);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_gae4(const float* r, const float* v, const float* v_next, const float* done, float* adv, double* stats, int T,
                int64_t B, float gamma, float lam, void* stream) {
    if (!r || !v || !v_next || !done || !adv || T < 1 || B < 1) return MTFJSP_E_ARG;
    const long long n = (long long)B * 4;
    gae4_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(r, v, v_next, done, adv, stats, T, B, gamma, lam);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_adv_normalize(float* adv, const double* stats, double count, int T, int64_t B, void* stream) {
    if (!adv || !stats || count < 2 || T < 1 || B < 1) return MTFJSP_E_ARG;
    const long long total = (long long)T * B * 4;
    adv_normalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(adv, stats, count, total);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}


int mtfjsp_enc_aggregate(const float* h, const float* adj_w, const int16_t* adj_src, float* out, int64_t B, int N,
                         int C, const float* in_scale, const float* in_shift, int in_relu, void* stream) {
    if (!h || !adj_w || !adj_src || !out || B < 1 || N < 1 || C < 4 || (C % 4) != 0) return MTFJSP_E_ARG;
    if ((in_scale == nullptr) != (in_shift == nullptr)) return MTFJSP_E_ARG;
    if (!al16(h, out, in_scale, in_shift) || !al8(adj_w)) return MTFJSP_E_ARG;
    const int C4 = C / 4;
    int c4_shift = -1;
    for (int k = 0; k < 16; k++)
        if ((1 << k) == C4) c4_shift = k;
    // 32-bit indexing inside a launch; whole envs per launch (the machine-predecessor gather stays inside an env)
    const long long per_env = (long long)N * C4;
    const long long chunk = (long long)0x7fffff00 / per_env;
    if (chunk < 1) return MTFJSP_E_ARG;
    for (long long b0 = 0; b0 < B; b0 += chunk) {
        const long long nb = B - b0 < chunk ? B - b0 : chunk;
        const unsigned total = (unsigned)(nb * per_env);
        const long long r0 = b0 * N;
        aggregate_kernel<false><<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
            reinterpret_cast<const float4*>(h) + r0 * C4, reinterpret_cast<const float2*>(adj_w) + r0, adj_src + r0,
            reinterpret_cast<float4*>(out) + r0 * C4, total, N, C4, c4_shift, reinterpret_cast<const float4*>(in_scale),
            reinterpret_cast<const float4*>(in_shift), in_relu);
    }
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_ell_invert(const int16_t* adj_src, int16_t* adj_dst, int64_t B, int N, void* stream) {
    if (!adj_src || !adj_dst || B < 1 || N < 1 || (long long)B * N > 0x7fffff00LL) return MTFJSP_E_ARG;
    const unsigned rows = (unsigned)(B * N);
    if (cudaMemsetAsync(adj_dst, 0xff, (size_t)rows * 2, (cudaStream_t)stream) != cudaSuccess) return MTFJSP_E_CUDA;
    ell_invert_kernel<<<(rows + 255) / 256, 256, 0, (cudaStream_t)stream>>>(adj_src, adj_dst, rows, N);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_aggregate_bwd(const float* g, const float* adj_w, const int16_t* adj_src, const int16_t* adj_dst, float* out,
                             int64_t B, int N, int C, void* stream) {
    if (!g || !adj_w || !adj_src || !adj_dst || !out || B < 1 || N < 1 || C < 4 || (C % 4) != 0) return MTFJSP_E_ARG;
    if (!al16(g, out) || !al8(adj_w)) return MTFJSP_E_ARG;
    const int C4 = C / 4;
    int c4_shift = -1;
    for (int k = 0; k < 16; k++)
        if ((1 << k) == C4) c4_shift = k;
    const long long per_env = (long long)N * C4;
    const long long chunk = (long long)0x7fffff00 / per_env;
    if (chunk < 1) return MTFJSP_E_ARG;
    for (long long b0 = 0; b0 < B; b0 += chunk) {
        const long long nb = B - b0 < chunk ? B - b0 : chunk;
        const unsigned total = (unsigned)(nb * per_env);
        const long long r0 = b0 * N;
        aggregate_bwd_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
            reinterpret_cast<const float4*>(g) + r0 * C4, reinterpret_cast<const float2*>(adj_w) + r0, adj_src + r0,
            adj_dst + r0, reinterpret_cast<float4*>(out) + r0 * C4, total, N, C4, c4_shift);
    }
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

static bool bn_args_ok(int64_t G, int64_t R, int C) { return G >= 1 && G <= 65535 && R >= 1 && C >= 4 && C <= 1024 && (C % 4) == 0; }

int mtfjsp_enc_bn_fwd(const float* x, const float* w, const float* b, float eps, int64_t G, int64_t R, int C, int relu, float* y,
                      float* mean, float* rstd, double* workspace, void* stream) {
    if (!x || !w || !b || !y || !mean || !rstd || !workspace || !bn_args_ok(G, R, C)) return MTFJSP_E_ARG;
    if (!al16(x, w, b, y, mean, rstd) || !al8(workspace)) return MTFJSP_E_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const int C4 = C / 4, ny = 256 / C4 > 0 ? 256 / C4 : 1;
    const int threads = C4 * ny > 256 ? C4 : 256;
    const dim3 grid((unsigned)((R + BN_ROWS - 1) / BN_ROWS), (unsigned)G);
    const size_t smem = (size_t)2 * (threads / C4) * C * sizeof(double);
    if (cudaMemsetAsync(workspace, 0, (size_t)G * 2 * C * sizeof(double), s) != cudaSuccess) return MTFJSP_E_CUDA;
    bn_reduce_kernel<0><<<grid, threads, smem, s>>>(reinterpret_cast<const float4*>(x), nullptr, w, b, nullptr, nullptr, workspace,
                                                    R, C4, 0);
    bn_stats_finalize_kernel<<<(unsigned)((G * C + 255) / 256), 256, 0, s>>>(workspace, x, R, 1.0 / (double)R, eps, mean, rstd,
                                                                          (int)G, C);
    bn_apply_kernel<0><<<grid, threads, 0, s>>>(reinterpret_cast<const float4*>(x), nullptr, w, b, mean, rstd, nullptr,
                                                reinterpret_cast<float4*>(y), R, C4, relu, 0.f);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_bn_bwd(const float* x, const float* gy, const float* w, const float* b, const float* mean, const float* rstd,
                      int64_t G, int64_t R, int C, int relu, float* dx, double* sums, void* stream) {
    if (!x || !gy || !w || !b || !mean || !rstd || !dx || !sums || !bn_args_ok(G, R, C)) return MTFJSP_E_ARG;
    if (!al16(x, gy, w, b, mean, rstd, dx) || !al8(sums)) return MTFJSP_E_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const int C4 = C / 4, ny = 256 / C4 > 0 ? 256 / C4 : 1;
    const int threads = C4 * ny > 256 ? C4 : 256;
    const dim3 grid((unsigned)((R + BN_ROWS - 1) / BN_ROWS), (unsigned)G);
    const size_t smem = (size_t)2 * (threads / C4) * C * sizeof(double);
    if (cudaMemsetAsync(sums, 0, (size_t)G * 2 * C * sizeof(double), s) != cudaSuccess) return MTFJSP_E_CUDA;
    bn_reduce_kernel<1><<<grid, threads, smem, s>>>(reinterpret_cast<const float4*>(x), reinterpret_cast<const float4*>(gy), w, b, mean,
                                                    rstd, sums, R, C4, relu);
    bn_apply_kernel<1><<<grid, threads, 0, s>>>(reinterpret_cast<const float4*>(x), reinterpret_cast<const float4*>(gy), w, b, mean,
                                                rstd, sums, reinterpret_cast<float4*>(dx), R, C4, relu, 1.0f / (float)R);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_graph_mean(const float* h, float* out, int64_t B, int N, int C, const float* in_scale,
                          const float* in_shift, int in_relu, void* stream) {
    if (!h || !out || B < 1 || N < 1 || C < 1) return MTFJSP_E_ARG;
    if ((in_scale == nullptr) != (in_shift == nullptr)) return MTFJSP_E_ARG;
    graph_mean_kernel<false><<<(unsigned)B, C < 128 ? 32 * ((C + 31) / 32) : 128, 0, (cudaStream_t)stream>>>(h, out, N, C, in_scale,
                                                                                                   in_shift, in_relu);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_aggregate_grouped(const float* h, const float* adj_w, const int16_t* adj_src, float* out, int64_t B, int N, int C,
                                 const float* in_scale, const float* in_shift, int in_relu, int envs_per_group, void* stream) {
    if (!h || !adj_w || !adj_src || !out || !in_scale || !in_shift || B < 1 || N < 1 || C < 4 || (C % 4) != 0) return MTFJSP_E_ARG;
    if (envs_per_group < 1 || B % envs_per_group != 0) return MTFJSP_E_ARG;
    if (!al16(h, out, in_scale, in_shift) || !al8(adj_w)) return MTFJSP_E_ARG;
    const int C4 = C / 4;
    int c4_shift = -1;
    for (int k = 0; k < 16; k++)
        if ((1 << k) == C4) c4_shift = k;
    const long long per_env = (long long)N * C4;
    const long long chunk = (long long)0x7fffff00 / per_env;
    if (chunk < 1) return MTFJSP_E_ARG;
    for (long long b0 = 0; b0 < B; b0 += chunk) {
        const long long nb = B - b0 < chunk ? B - b0 : chunk;
        const unsigned total = (unsigned)(nb * per_env);
        const long long r0 = b0 * N;
        aggregate_kernel<true><<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
            reinterpret_cast<const float4*>(h) + r0 * C4, reinterpret_cast<const float2*>(adj_w) + r0, adj_src + r0,
            reinterpret_cast<float4*>(out) + r0 * C4, total, N, C4, c4_shift, reinterpret_cast<const float4*>(in_scale),
            reinterpret_cast<const float4*>(in_shift), in_relu, b0, envs_per_group);
    }
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_graph_mean_grouped(const float* h, float* out, int64_t B, int N, int C, const float* in_scale, const float* in_shift,
                                  int in_relu, int envs_per_group, void* stream) {
    if (!h || !out || !in_scale || !in_shift || B < 1 || N < 1 || C < 1) return MTFJSP_E_ARG;
    if (envs_per_group < 1 || B % envs_per_group != 0) return MTFJSP_E_ARG;
    graph_mean_kernel<true><<<(unsigned)B, C < 128 ? 32 * ((C + 31) / 32) : 128, 0, (cudaStream_t)stream>>>(h, out, N, C, in_scale,
                                                                                                         in_shift, in_relu,
                                                                                                         envs_per_group);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_gat_attend(const float* t, const float* a_src, const float* a_dst, float* out, int64_t R, int mode,
                          void* stream) {
    if (!t || !a_src || !a_dst || !out || R < 1 || mode < 0 || mode > 2) return MTFJSP_E_ARG;
    if (!al16(t, a_src, a_dst, out)) return MTFJSP_E_ARG;
    gat_attend_kernel<<<(unsigned)((R + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(t), reinterpret_cast<const float4*>(a_src), reinterpret_cast<const float4*>(a_dst),
        reinterpret_cast<float4*>(out), R, mode);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}

int mtfjsp_enc_gat_attend_bwd_blocks(int64_t R) {
    const long long b = (R + 7) / 8;
    return (int)(b < 148 * 8 ? b : 148 * 8);
}

int mtfjsp_enc_gat_attend_bwd(const float* t, const float* a_src, const float* a_dst, const float* g, float* dt, float* dparts,
                              int64_t R, int mode, void* stream) {
    if (!t || !a_src || !a_dst || !g || !dt || !dparts || R < 1 || mode < 0 || mode > 2) return MTFJSP_E_ARG;
    if (!al16(t, a_src, a_dst, g, dt, dparts)) return MTFJSP_E_ARG;
    gat_attend_bwd_kernel<<<mtfjsp_enc_gat_attend_bwd_blocks(R), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(t), reinterpret_cast<const float4*>(a_src), reinterpret_cast<const float4*>(a_dst),
        reinterpret_cast<const float4*>(g), reinterpret_cast<float4*>(dt), dparts, R, mode);
    return cudaGetLastError() == cudaSuccess ? MTFJSP_OK : MTFJSP_E_CUDA;
}


}  // extern "C"
