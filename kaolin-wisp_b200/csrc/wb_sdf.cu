// wb_sdf.cu -- NeuralSDF(OctreeGrid) evaluation and the sphere tracer of app/nglod as ONE persistent kernel.
//
//   wb_sdf_eval   NeuralSDF.sdf (wisp/models/nefs/neural_sdf.py:120-155) = OctreeGrid.interpolate (octree_grid.py:130-219)
//                 + [position embedding first, features second] + BasicDecoder (basic_decoders.py:73-101), one thread per
//                 point, the decoder's weights staged in shared memory.  The reference runs a query, one Kaolin launch per
//                 LOD, a cat and two cuBLAS GEMMs per call.
//   wb_sdf_trace  PackedSDFTracer.trace (wisp/tracers/packed_sdf_tracer.py:78-174) + find_depth_bound
//                 (wisp/csrc/render/find_depth_bound_cuda.cu:16-45) + finitediff_gradient (wisp/ops/differential/gradients.py:29-45).
//                 The reference is a Python loop of ~15 masked torch kernels, a boolean-mask gather and one nef call per
//                 step.  Here: one cooperative kernel, one thread per pack (ray with >= 1 nugget) and step, per-pack state in a
//                 40-byte SoA record, grid-wide barriers where the reference's semantics are grid-wide:
//                   * the loop ends when NO pack is alive anywhere (`if not mask.any(): break`, :129,:143) -- terminated packs
//                     keep adding their last `dist` to `t` on every iteration that is still executed (:121 is unmasked), so the
//                     reported depth of a hit depends on the global iteration count;
//                   * find_depth_bound bounds the scan of pack p by the CURRENT cursor of pack p+1 (cu:29) -- cursors are
//                     double buffered and exchanged at the barrier.
//                 Normals by central differences (6 more evaluations at the finest LOD) in the epilogue of the same kernel.
//   Numerics: fp32 decoder (the tracer runs under torch.no_grad() without autocast); octree features rounded to fp16 on load and
//   per-LOD results rounded to fp16, as the call site does (octree_grid.py:147-149).  The decoder's summation order differs from
//   cuBLAS: results agree to fp32 rounding, hit decisions can differ only where |sdf| is within ~1e-6 of a threshold.
#include "wb_common.cuh"
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

constexpr int WB_SDF_MAX_IN = 132;        // 3 + 6*freq position embedding + features
constexpr int WB_SDF_MAX_H = 128;
constexpr int WB_SDF_THREADS = 256;

struct WbSdf {
    // octree grid
    const int16_t* points; const int32_t* trinkets;
    const float* feats[WB_MAX_LODS];
    int F, base_lod, num_lods, multiscale, half_round;
    // decoder
    int pos_mode, pos_freq, pos_dim, feat_dim, in_dim, in_pad, H, nh;      // nh hidden layers (>= 1), all H wide
    const float* params;                                                     // packed [W0, b0, W1, b1, ..., Wout, bout] (nn.Linear layout)
    int smem_floats;
};

static int sdf_embed_dim(int mode, int freq) { return mode == 0 ? 0 : mode == 1 ? 3 : mode == 2 ? 6 * freq : 3 + 6 * freq; }

static int wb_make_sdf(const wb_sdf_desc* d, WbSdf* m)
{
    WB_CHECK_ARG(d != nullptr && d->points && d->trinkets && d->feats && d->params, "null pointer in wb_sdf_desc");
    WB_CHECK_ARG(d->num_lods >= 1 && d->num_lods <= WB_MAX_LODS && d->base_lod >= 0, "bad LOD range");
    WB_CHECK_ARG(d->feature_dim >= 1 && d->feature_dim <= 64, "feature_dim must be in [1,64]");
    WB_CHECK_ARG(d->multiscale == 0 || d->multiscale == 1, "multiscale must be 0 ('cat') or 1 ('sum')");
    WB_CHECK_ARG(d->num_layers >= 1 && d->num_layers <= 4 && d->hidden_dim >= 1 && d->hidden_dim <= WB_SDF_MAX_H, "decoder: 1..4 hidden layers, <= 128 wide");
    WB_CHECK_ARG(d->pos_mode >= 0 && d->pos_mode <= 3 && d->pos_freq >= 0 && d->pos_freq <= 10, "bad position embedding");
    m->points = d->points; m->trinkets = d->trinkets;
    for (int k = 0; k < d->num_lods; ++k) { WB_CHECK_ARG(d->feats[k] != nullptr, "null feature level"); m->feats[k] = d->feats[k]; }
    m->F = d->feature_dim; m->base_lod = d->base_lod; m->num_lods = d->num_lods; m->multiscale = d->multiscale; m->half_round = d->half_round;
    m->pos_mode = d->pos_mode; m->pos_freq = d->pos_freq; m->pos_dim = sdf_embed_dim(d->pos_mode, d->pos_freq);
    m->feat_dim = d->multiscale ? d->feature_dim : d->feature_dim * d->num_lods;
    m->in_dim = m->pos_dim + m->feat_dim; m->in_pad = (m->in_dim + 3) & ~3;
    WB_CHECK_ARG(m->in_dim <= WB_SDF_MAX_IN, "decoder input too wide");
    m->H = d->hidden_dim; m->nh = d->num_layers; m->params = d->params;
    WB_CHECK_ARG(m->nh == 1 || (m->H % 4) == 0, "hidden_dim must be a multiple of 4 for multi-layer decoders");
    m->smem_floats = m->H * m->in_pad + m->H + (m->nh - 1) * (m->H * m->H + m->H) + m->H + 4;
    WB_CHECK_ARG(m->smem_floats * 4 <= 200 * 1024, "decoder does not fit in shared memory");
    return WB_OK;
}

// shared-memory image: W0 rows padded to in_pad floats | b0 | (W_k [H x H] | b_k) ... | Wout [H] | bout
__device__ __forceinline__ void sdf_stage(const WbSdf& m, float* sw)
{
    const float* p = m.params;
    int o = 0, src = 0;
    for (int e = threadIdx.x; e < m.H * m.in_pad; e += blockDim.x) {
        const int j = e / m.in_pad, k = e - j * m.in_pad;
        sw[e] = k < m.in_dim ? __ldg(p + j * m.in_dim + k) : 0.0f;
    }
    o += m.H * m.in_pad; src += m.H * m.in_dim;
    for (int e = threadIdx.x; e < m.H; e += blockDim.x) sw[o + e] = __ldg(p + src + e);
    o += m.H; src += m.H;
    for (int l = 1; l < m.nh; ++l) {
        for (int e = threadIdx.x; e < m.H * m.H + m.H; e += blockDim.x) sw[o + e] = __ldg(p + src + e);
        o += m.H * m.H + m.H; src += m.H * m.H + m.H;
    }
    for (int e = threadIdx.x; e < m.H + 1; e += blockDim.x) sw[o + e] = __ldg(p + src + e);
    __syncthreads();
}

__device__ __forceinline__ float sdf_h(float v) { return __half2float(__float2half_rn(v)); }

// positional_embedder.py:51-66 / neural_sdf.py:86-99: [x (include_input), sin(winded), cos(winded)], winded freq-major coord-minor
__device__ __forceinline__ int sdf_embed(int mode, int freq, float x, float y, float z, float* out)
{
    if (mode == 0) return 0;
    int o = 0;
    if (mode == 1 || mode == 3) { out[0] = x; out[1] = y; out[2] = z; o = 3; }
    if (mode == 1) return 3;
    float band = 1.0f;
    for (int f = 0; f < freq; ++f) {
        out[o + f * 3 + 0] = sinf(x * band); out[o + f * 3 + 1] = sinf(y * band); out[o + f * 3 + 2] = sinf(z * band);
        out[o + 3 * freq + f * 3 + 0] = cosf(x * band); out[o + 3 * freq + f * 3 + 1] = cosf(y * band); out[o + 3 * freq + f * 3 + 2] = cosf(z * band);
        band *= 2.0f;
    }
    return o + 6 * freq;
}

// OctreeGrid.interpolate for LODs 0..nl-1 of one point -> feat[] (zeros where the point leaves the octree); FT > 0: compile-time
// feature width of a 'sum' grid (accumulators in registers)
template <int FT>
__device__ __forceinline__ void sdf_features(const WbOct& oc, const WbSdf& m, int nl, float cx, float cy, float cz, float* feat)
{
    const int F = FT > 0 ? FT : m.F;
    const bool sum = FT > 0 ? true : (m.multiscale != 0 && nl > 1);         // lod_idx == 0: a single LOD either way (octree_grid.py:190-198)
    const int width = sum ? F : nl * F;
#pragma unroll
    for (int f = 0; f < (FT > 0 ? FT : 1); ++f) feat[f] = 0.0f;
    if (FT == 0) for (int f = 0; f < width; ++f) feat[f] = 0.0f;
    const int L = m.base_lod + nl - 1;                                       // level of the finest LOD used
    const float h = ldexpf(1.0f, L - 1), inv_h = ldexpf(1.0f, -(L - 1)), maxq = (float)((1 << L) - 1);
    int qx, qy, qz;
    if (!(wb_quantize(cx, h, inv_h, maxq, qx) && wb_quantize(cy, h, inv_h, maxq, qy) && wb_quantize(cz, h, inv_h, maxq, qz))) return;
    int node = 0;
    for (int l = 0; l <= L; ++l) {
        if (l > 0) {
            const int d = L - l;
            const int ci = (((qx >> d) & 1) << 2) | (((qy >> d) & 1) << 1) | ((qz >> d) & 1);
            const uint32_t b = __ldg(oc.octree + node);
            if (!(b & (1u << ci))) return;
            node = __ldg(oc.prefix + node) + __popc(b & ((2u << ci) - 1u));
        }
        const int k = l - m.base_lod;
        if (k < 0) continue;
        const float hl = ldexpf(1.0f, l - 1);
        const float ux = __fmaf_rn(cx, hl, hl) - (float)__ldg(m.points + 3 * (int64_t)node);
        const float uy = __fmaf_rn(cy, hl, hl) - (float)__ldg(m.points + 3 * (int64_t)node + 1);
        const float uz = __fmaf_rn(cz, hl, hl) - (float)__ldg(m.points + 3 * (int64_t)node + 2);
        const float ix = 1.0f - ux, iy = 1.0f - uy, iz = 1.0f - uz;
        float cf[8];
        cf[0] = (ix * iy) * iz; cf[1] = (ix * iy) * uz; cf[2] = (ix * uy) * iz; cf[3] = (ix * uy) * uz;
        cf[4] = (ux * iy) * iz; cf[5] = (ux * iy) * uz; cf[6] = (ux * uy) * iz; cf[7] = (ux * uy) * uz;
        const int4 t0 = __ldg(reinterpret_cast<const int4*>(m.trinkets + 8 * (int64_t)node));
        const int4 t1 = __ldg(reinterpret_cast<const int4*>(m.trinkets + 8 * (int64_t)node) + 1);
        const int tk[8] = { t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w };
        const float* ft = m.feats[k];
        if (FT > 0 && (FT % 4) == 0) {
            float acc[FT > 0 ? FT : 1];
#pragma unroll
            for (int f = 0; f < FT; ++f) acc[f] = 0.0f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4* row = reinterpret_cast<const float4*>(ft + (int64_t)tk[j] * FT);
#pragma unroll
                for (int q = 0; q < FT / 4; ++q) {
                    float4 v = __ldg(row + q);
                    if (m.half_round) { v.x = sdf_h(v.x); v.y = sdf_h(v.y); v.z = sdf_h(v.z); v.w = sdf_h(v.w); }
                    acc[4 * q] = fmaf(v.x, cf[j], acc[4 * q]); acc[4 * q + 1] = fmaf(v.y, cf[j], acc[4 * q + 1]);
                    acc[4 * q + 2] = fmaf(v.z, cf[j], acc[4 * q + 2]); acc[4 * q + 3] = fmaf(v.w, cf[j], acc[4 * q + 3]);
                }
            }
#pragma unroll
            for (int f = 0; f < FT; ++f) feat[f] += m.half_round ? sdf_h(acc[f]) : acc[f];
        } else {
            for (int f = 0; f < F; ++f) {
                float acc = 0.0f;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float v = __ldg(ft + (int64_t)tk[j] * F + f);
                    if (m.half_round) v = sdf_h(v);
                    acc = fmaf(v, cf[j], acc);
                }
                if (m.half_round) acc = sdf_h(acc);
                if (sum) feat[f] += acc; else feat[k * F + f] = acc;
            }
        }
        if (k == nl - 1) return;
    }
}

// NeuralSDF.sdf at one point.  FT/PT > 0: the app/nglod shape ('sum' grid of FT features, identity position input) with the
// input vector in registers; otherwise the generic path through local arrays.
template <int FT, int PT>
__device__ __forceinline__ float sdf_eval(const WbOct& oc, const WbSdf& m, const float* __restrict__ sw, int nl, float x, float y, float z)
{
    const int H = m.H;
    if constexpr (FT > 0 && PT == 1) {                    // dispatch guarantees nh == 1, 'sum', identity position input
        constexpr int IN = 3 + (FT > 0 ? FT : 1), INP = (IN + 3) & ~3;
        float in[INP];
        in[0] = x; in[1] = y; in[2] = z;
        sdf_features<FT>(oc, m, nl, x, y, z, in + 3);
#pragma unroll
        for (int k = IN; k < INP; ++k) in[k] = 0.0f;
        const float* b0 = sw + H * INP; const float* wo = b0 + H;
        float out = wo[H];
        // four hidden units at a time: four independent FMA chains instead of one 20-deep dependent chain per unit (the evaluation is a
        // latency chain per thread: few packs are alive per CTA, nothing else hides the FMA latency)
        int j = 0;
        for (; j + 4 <= H; j += 4) {
            float a0 = b0[j], a1 = b0[j + 1], a2 = b0[j + 2], a3 = b0[j + 3];
            const float4* w0 = reinterpret_cast<const float4*>(sw + j * INP);
            const float4* w1 = reinterpret_cast<const float4*>(sw + (j + 1) * INP);
            const float4* w2 = reinterpret_cast<const float4*>(sw + (j + 2) * INP);
            const float4* w3 = reinterpret_cast<const float4*>(sw + (j + 3) * INP);
#pragma unroll
            for (int q = 0; q < INP / 4; ++q) {
                const float4 u0 = w0[q], u1 = w1[q], u2 = w2[q], u3 = w3[q];
                const float x0 = in[4 * q], x1 = in[4 * q + 1], x2 = in[4 * q + 2], x3 = in[4 * q + 3];
                a0 = fmaf(u0.x, x0, a0); a1 = fmaf(u1.x, x0, a1); a2 = fmaf(u2.x, x0, a2); a3 = fmaf(u3.x, x0, a3);
                a0 = fmaf(u0.y, x1, a0); a1 = fmaf(u1.y, x1, a1); a2 = fmaf(u2.y, x1, a2); a3 = fmaf(u3.y, x1, a3);
                a0 = fmaf(u0.z, x2, a0); a1 = fmaf(u1.z, x2, a1); a2 = fmaf(u2.z, x2, a2); a3 = fmaf(u3.z, x2, a3);
                a0 = fmaf(u0.w, x3, a0); a1 = fmaf(u1.w, x3, a1); a2 = fmaf(u2.w, x3, a2); a3 = fmaf(u3.w, x3, a3);
            }
            // the output layer sums in unit order, as the single-chain form did
            out = fmaf(wo[j], fmaxf(a0, 0.0f), out); out = fmaf(wo[j + 1], fmaxf(a1, 0.0f), out);
            out = fmaf(wo[j + 2], fmaxf(a2, 0.0f), out); out = fmaf(wo[j + 3], fmaxf(a3, 0.0f), out);
        }
        for (; j < H; ++j) {
            const float4* wr = reinterpret_cast<const float4*>(sw + j * INP);
            float a = b0[j];
#pragma unroll
            for (int q = 0; q < INP / 4; ++q) {
                const float4 w = wr[q];
                a = fmaf(w.x, in[4 * q], a); a = fmaf(w.y, in[4 * q + 1], a); a = fmaf(w.z, in[4 * q + 2], a); a = fmaf(w.w, in[4 * q + 3], a);
            }
            out = fmaf(wo[j], fmaxf(a, 0.0f), out);
        }
        return out;
    } else {
    float in[WB_SDF_MAX_IN];
    const int pd = sdf_embed(m.pos_mode, m.pos_freq, x, y, z, in);
    sdf_features<0>(oc, m, nl, x, y, z, in + pd);
    // a grid evaluated below its finest LOD yields fewer 'cat' features than the decoder expects only when lod_idx < num_lods-1
    // with 'cat'; the reference would fail in nn.Linear -- the host shim rejects that combination
    float ha[WB_SDF_MAX_H], hb[WB_SDF_MAX_H];
    const float* w = sw; const float* b = sw + H * m.in_pad;
    for (int j = 0; j < H; ++j) {
        float a = b[j];
        for (int k = 0; k < m.in_dim; ++k) a = fmaf(w[j * m.in_pad + k], in[k], a);
        ha[j] = fmaxf(a, 0.0f);
    }
    const float* p = b + H;
    float* cur = ha; float* nxt = hb;
    for (int l = 1; l < m.nh; ++l) {
        const float* wl = p; const float* bl = p + H * H;
        for (int j = 0; j < H; ++j) {
            float a = bl[j];
            for (int k = 0; k < H; ++k) a = fmaf(wl[j * H + k], cur[k], a);
            nxt[j] = fmaxf(a, 0.0f);
        }
        p += H * H + H;
        float* t = cur; cur = nxt; nxt = t;
    }
    float out = p[H];
    for (int j = 0; j < H; ++j) out = fmaf(p[j], cur[j], out);
    return out;
    }
}

template <int FT, int PT>
__global__ void __launch_bounds__(WB_SDF_THREADS)
wb_sdf_eval_kernel(WbOct oc, WbSdf m, int nl, const float* __restrict__ coords, int64_t N, float* __restrict__ out)
{
    extern __shared__ __align__(16) float sw[];
    sdf_stage(m, sw);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = sdf_eval<FT, PT>(oc, m, sw, nl, __ldg(coords + 3 * i), __ldg(coords + 3 * i + 1), __ldg(coords + 3 * i + 2));
}

// ---------------------------------------------------------------------------------------------------------------------
// sphere tracer
// ---------------------------------------------------------------------------------------------------------------------
struct WbSdfTrace {
    const float* origins; const float* dirs; int64_t R; float dist_max;
    const float2* nug_depth; int64_t Ng; const int64_t* ray_offsets;     // raw raytrace depths (entry, exit); nuggets of ray r: [off[r], off[r+1])
    wb_sdf_state S;                                                        // per-pack state, owned by the caller
    int num_steps, nl, want_normals; float step_size, min_dis, min_dis5;
    float* o_xyz; float* o_depth; uint8_t* o_hit; float* o_normal; float* o_rgb; float* o_alpha;
};
enum { SDF_ALIVE = 1, SDF_HIT = 2 };

__global__ void wb_sdf_flag_kernel(const int64_t* __restrict__ ray_offsets, int64_t R, int32_t* __restrict__ flags)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < R) flags[r] = ray_offsets[r + 1] > ray_offsets[r] ? 1 : 0;
}

__device__ __forceinline__ void sdf_point(const WbSdfTrace& T, int64_t r, float t, float& x, float& y, float& z)
{
    x = wb_addcmul(__ldg(T.origins + 3 * r), __ldg(T.dirs + 3 * r), t);                 // torch.addcmul(nug_o, nug_d, t) (:104,:122,:140)
    y = wb_addcmul(__ldg(T.origins + 3 * r + 1), __ldg(T.dirs + 3 * r + 1), t);
    z = wb_addcmul(__ldg(T.origins + 3 * r + 2), __ldg(T.dirs + 3 * r + 2), t);
}
// packs = rays with at least one nugget, in ray order (mark_pack_boundaries + nonzero, :93-94)
__device__ __forceinline__ void sdf_pack_list(const WbSdfTrace& T, int64_t tid, int64_t nthr)
{
    for (int64_t r = tid; r < T.R; r += nthr)
        if (T.S.pack_off[r + 1] > T.S.pack_off[r]) T.S.pack_ray[T.S.pack_off[r]] = (int32_t)r;
}
// initial state of pack p (:96-113) except its first distance; returns the start point
__device__ __forceinline__ void sdf_init_pack(const WbSdfTrace& T, int64_t p, float& x, float& y, float& z)
{
    const int64_t r = T.S.pack_ray[p];
    const int32_t first = (int32_t)T.ray_offsets[r];
    const float t = __fadd_rn(__ldg(&T.nug_depth[first]).x, 1e-5f);                     // depth[..., 0:1] += 1e-5 (:91)
    sdf_point(T, r, t, x, y, z);
    T.S.t[p] = t; T.S.x[3 * p] = x; T.S.x[3 * p + 1] = y; T.S.x[3 * p + 2] = z;
    T.S.cursor0[p] = first; T.S.state[p] = SDF_ALIVE;
}
// step 1: march by the SDF (:120-131); returns whether the pack is still alive
__device__ __forceinline__ bool sdf_march_pack(const WbSdfTrace& T, int64_t p)
{
    uint8_t st = T.S.state[p];
    const float d = T.S.dist[p];
    const float t = __fadd_rn(T.S.t[p], d);                                             // unmasked in the reference: dead packs drift too
    T.S.t[p] = t;
    if (!(st & SDF_ALIVE)) return false;
    float x, y, z; sdf_point(T, T.S.pack_ray[p], t, x, y, z);
    T.S.x[3 * p] = x; T.S.x[3 * p + 1] = y; T.S.x[3 * p + 2] = z;
    const bool h = (fabsf(d) < T.min_dis) || (__fmul_rn(fabsf(__fadd_rn(d, T.S.dist_prev[p])), 0.5f) < T.min_dis5);
    st = h ? (uint8_t)(st | SDF_HIT) : (uint8_t)(st & ~SDF_HIT);
    if (!(t < T.dist_max) || h) st &= (uint8_t)~SDF_ALIVE;
    if (st & SDF_ALIVE) T.S.dist_prev[p] = d;
    T.S.state[p] = st;
    return (st & SDF_ALIVE) != 0;
}
// step 2: jump to the next occupied cell (:133-141); returns whether the pack is still alive (then x holds its new point)
__device__ __forceinline__ bool sdf_jump_pack(const WbSdfTrace& T, int64_t p, int64_t P, const int32_t* __restrict__ cin, int32_t* __restrict__ cout,
                                              float& x, float& y, float& z)
{
    uint8_t st = T.S.state[p];
    const int32_t cur = cin[p];
    float t = T.S.t[p];
    int32_t nxt = -1;
    if (cur > -1) {                                                                     // find_depth_bound, for every pack (cu:24-43)
        uint32_t i = (uint32_t)cur;
        const uint32_t mx = (p == P - 1) ? (uint32_t)P : (uint32_t)cin[p + 1];         // reference quirks kept (cu:28-29)
        while (i < mx && (int64_t)i < T.Ng) {
            const float2 dd = __ldg(&T.nug_depth[i]);
            const float en = __fadd_rn(dd.x, 1e-5f);
            if ((t >= en && t <= dd.y) || t < en) { nxt = (int32_t)i; break; }
            ++i;
        }
    }
    bool alive = false;
    int32_t ncur = cur;
    if (st & SDF_ALIVE) {
        if (nxt == -1) st &= (uint8_t)~SDF_ALIVE;
        else {
            if (nxt != cur) { t = __fadd_rn(__ldg(&T.nug_depth[nxt]).x, 1e-5f); T.S.t[p] = t; }
            ncur = nxt;
            sdf_point(T, T.S.pack_ray[p], t, x, y, z);
            T.S.x[3 * p] = x; T.S.x[3 * p + 1] = y; T.S.x[3 * p + 2] = z;
            alive = true;
        }
        T.S.state[p] = st;
    }
    cout[p] = ncur;
    return alive;
}
// outputs (:149-174) of a pack that hit, normals excluded
__device__ __forceinline__ void sdf_write_hit(const WbSdfTrace& T, int64_t p, int64_t r)
{
    T.o_xyz[3 * r] = T.S.x[3 * p]; T.o_xyz[3 * r + 1] = T.S.x[3 * p + 1]; T.o_xyz[3 * r + 2] = T.S.x[3 * p + 2];
    T.o_depth[r] = T.S.t[p]; T.o_hit[r] = 1; T.o_alpha[r] = 1.0f;
}

// register allocation bounded for 2 resident CTAs per SM (threads in flight = packs handled at once): 0.97 ms measured against
// 1.14 / 1.31 / 1.56 ms for 1 / 3 / 4 (profiles/README.md)
template <int FT, int PT>
__global__ void __launch_bounds__(WB_SDF_THREADS, 2)
wb_sdf_trace_kernel(WbOct oc, WbSdf m, WbSdfTrace T)
{
    extern __shared__ __align__(16) float sw[];
    cg::grid_group grid = cg::this_grid();
    sdf_stage(m, sw);
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
    const int64_t P = T.S.pack_off[T.R];
    sdf_pack_list(T, tid, nthr);
    grid.sync();
    int evals = 0;                                    // field evaluations of this thread (bench.py: algorithmic bytes of the launch)
    for (int64_t p = tid; p < P; p += nthr) {
        ++evals;
        float x, y, z; sdf_init_pack(T, p, x, y, z);
        const float d = __fmul_rn(__fmul_rn(sdf_eval<FT, PT>(oc, m, sw, T.nl, x, y, z), 1.0f), T.step_size);   // sdf * invres * step_size (:109)
        T.S.dist[p] = d; T.S.dist_prev[p] = d;
    }
    grid.sync();
    int cb = 0;
    for (int it = 0; it < T.num_steps; ++it) {
        int any = 0;
        for (int64_t p = tid; p < P; p += nthr) any |= sdf_march_pack(T, p) ? 1 : 0;
        if (__syncthreads_or(any) && threadIdx.x == 0) atomicOr(T.S.iterflags + 2 * it, 1);
        grid.sync();
        if (__ldcg(T.S.iterflags + 2 * it) == 0) break;                                 // `if not mask.any(): break` (:129)
        any = 0;
        const int32_t* cin = cb ? T.S.cursor1 : T.S.cursor0; int32_t* cout = cb ? T.S.cursor0 : T.S.cursor1;
        for (int64_t p = tid; p < P; p += nthr) {
            float x, y, z;
            if (sdf_jump_pack(T, p, P, cin, cout, x, y, z)) {
                ++evals;
                T.S.dist[p] = __fmul_rn(__fmul_rn(sdf_eval<FT, PT>(oc, m, sw, T.nl, x, y, z), 1.0f), T.step_size);   // (:145-146)
                any = 1;
            }
        }
        cb ^= 1;
        if (__syncthreads_or(any) && threadIdx.x == 0) atomicOr(T.S.iterflags + 2 * it + 1, 1);
        grid.sync();
        if (__ldcg(T.S.iterflags + 2 * it + 1) == 0) break;                             // (:143)
    }
    for (int64_t p = tid; p < P; p += nthr) {
        if (!(T.S.state[p] & SDF_HIT)) continue;
        const int64_t r = T.S.pack_ray[p];
        sdf_write_hit(T, p, r);
        if (T.want_normals) {
            evals += 6;
            const float x = T.S.x[3 * p], y = T.S.x[3 * p + 1], z = T.S.x[3 * p + 2];
            const float eps = 0.005f, den = (float)(0.005 * 2.0);
            const int nlf = m.num_lods;                                                // lod_idx = None -> finest LOD (gradients.py / neural_sdf.py:136-137)
            float g3[3];
#pragma unroll 1
            for (int a = 0; a < 3; ++a) {                                               // f(x + eps e_a) - f(x - eps e_a)
                const float ex = a == 0 ? eps : 0.0f, ey = a == 1 ? eps : 0.0f, ez = a == 2 ? eps : 0.0f;
                float fp = 0.0f, fm = 0.0f;
#pragma unroll 1
                for (int sgn = 0; sgn < 2; ++sgn) {
                    const float v = sgn == 0 ? sdf_eval<FT, PT>(oc, m, sw, nlf, x + ex, y + ey, z + ez)
                                             : sdf_eval<FT, PT>(oc, m, sw, nlf, x - ex, y - ey, z - ez);
                    if (sgn == 0) fp = v; else fm = v;
                }
                g3[a] = fp - fm;
            }
            float gx = __fdiv_rn(g3[0], den), gy = __fdiv_rn(g3[1], den), gz = __fdiv_rn(g3[2], den);
            const float nrm = fmaxf(sqrtf(gx * gx + gy * gy + gz * gz), 1e-5f);         // F.normalize(p=2, eps=1e-5)
            gx = __fdiv_rn(gx, nrm); gy = __fdiv_rn(gy, nrm); gz = __fdiv_rn(gz, nrm);
            T.o_normal[3 * r] = gx; T.o_normal[3 * r + 1] = gy; T.o_normal[3 * r + 2] = gz;
            T.o_rgb[3 * r] = (gx + 1.0f) / 2.0f; T.o_rgb[3 * r + 1] = (gy + 1.0f) / 2.0f; T.o_rgb[3 * r + 2] = (gz + 1.0f) / 2.0f;
        }
    }
    evals = __reduce_add_sync(0xffffffffu, evals);
    if ((threadIdx.x & 31) == 0 && evals) atomicAdd(T.S.iterflags + 2 * T.num_steps + 2, evals);
}

// The same state machine one phase per launch, for neural fields whose SDF is evaluated outside this library (NeuralSDF over a
// hash or triplanar grid): the caller evaluates the field at S.x of the alive packs between the phases.
//   phase 0: pack list   1: initial state   2: step 1 (march)   3: step 2 (jump)   4: outputs of the packs that hit
__global__ void __launch_bounds__(WB_SDF_THREADS)
wb_sdf_phase_kernel(WbSdfTrace T, int phase, int it, int cb)
{
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
    const int64_t P = T.S.pack_off[T.R];
    if (phase == 0) { sdf_pack_list(T, tid, nthr); return; }
    int any = 0;
    for (int64_t p = tid; p < P; p += nthr) {
        float x, y, z;
        if (phase == 1) sdf_init_pack(T, p, x, y, z);
        else if (phase == 2) any |= sdf_march_pack(T, p) ? 1 : 0;
        else if (phase == 3) any |= sdf_jump_pack(T, p, P, cb ? T.S.cursor1 : T.S.cursor0, cb ? T.S.cursor0 : T.S.cursor1, x, y, z) ? 1 : 0;
        else if (T.S.state[p] & SDF_HIT) sdf_write_hit(T, p, T.S.pack_ray[p]);
    }
    if (phase == 2 || phase == 3)
        if (__syncthreads_or(any) && threadIdx.x == 0) atomicOr(T.S.iterflags + 2 * it + (phase == 3 ? 1 : 0), 1);
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
static bool sdf_fast_shape(const WbSdf& m) { return m.multiscale == 1 && m.F == 16 && m.pos_mode == 1 && m.nh == 1; }

extern "C" int wb_sdf_eval(const wb_octree* oct, const wb_sdf_desc* nef, int32_t lod_idx, const float* coords, int64_t N, float* out, wb_stream s)
{
    if (N == 0) return WB_OK;
    WbSdf m; int rc = wb_make_sdf(nef, &m); if (rc) return rc;
    WB_CHECK_ARG(lod_idx >= 0 && lod_idx < m.num_lods, "lod_idx out of range");
    WB_CHECK_ARG(m.multiscale == 1 || lod_idx == m.num_lods - 1, "'cat' grids feed the decoder all LODs: lod_idx must be num_lods-1");
    WbOct oc; rc = wb_make_oct(oct, m.base_lod + lod_idx, &oc); if (rc) return rc;
    WB_CHECK_ARG(coords && out, "null pointer");
    const int smem = m.smem_floats * 4;
    int64_t ctas = (N + WB_SDF_THREADS - 1) / WB_SDF_THREADS; const int64_t cap = (int64_t)wb_num_sms() * 8; if (ctas > cap) ctas = cap;
    auto kern = sdf_fast_shape(m) ? wb_sdf_eval_kernel<16, 1> : wb_sdf_eval_kernel<0, 0>;
    if (smem > 48 * 1024) WB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<(unsigned)ctas, WB_SDF_THREADS, smem, (cudaStream_t)s>>>(oc, m, lod_idx + 1, coords, N, out);
    WB_LAUNCH_CHECK();
    return WB_OK;
}

static int sdf_make_trace(const wb_rays* rays, const float* nug_depth, int64_t Ng, const int64_t* ray_offsets, int32_t num_steps, float step_size,
                          float min_dis, const wb_sdf_state* st, WbSdfTrace* T)
{
    WB_CHECK_ARG(rays != nullptr && rays->origins && rays->dirs && nug_depth && ray_offsets, "null pointer");
    WB_CHECK_ARG(rays->near_v == nullptr, "the SDF tracer compares t with a scalar dist_max (packed_sdf_tracer.py:127)");
    WB_CHECK_ARG(st && st->flags && st->pack_off && st->scan_ws && st->pack_ray && st->t && st->dist && st->dist_prev && st->x && st->cursor0 && st->cursor1 &&
                 st->state && st->iterflags, "null pointer in wb_sdf_state");
    WB_CHECK_ARG(num_steps >= 0 && num_steps <= 4096, "num_steps out of range");
    WB_CHECK_ARG(st->scan_ws_bytes >= wb_scan_workspace_bytes(rays->num_rays), "scan workspace too small (wb_scan_workspace_bytes)");
    memset(T, 0, sizeof(*T));
    T->origins = rays->origins; T->dirs = rays->dirs; T->R = rays->num_rays; T->dist_max = rays->dist_max;
    T->nug_depth = reinterpret_cast<const float2*>(nug_depth); T->Ng = Ng; T->ray_offsets = ray_offsets; T->S = *st;
    T->num_steps = num_steps; T->step_size = step_size;
    T->min_dis = (float)((double)min_dis * 1.0); T->min_dis5 = (float)(((double)min_dis * 5.0) * 1.0);     // min_dis * invres, (min_dis*5) * invres (:123-126)
    return WB_OK;
}
// rays with nuggets -> exclusive scan (pack_off); iteration flags cleared
static int sdf_scan_packs(const WbSdfTrace& T, int32_t num_steps, cudaStream_t st)
{
    WB_CUDA(cudaMemsetAsync(T.S.iterflags, 0, 4 * (2 * (size_t)num_steps + 4), st));
    wb_sdf_flag_kernel<<<(unsigned)((T.R + 255) / 256), 256, 0, st>>>(T.ray_offsets, T.R, T.S.flags);
    WB_LAUNCH_CHECK();
    return wb_scan_counts(T.S.flags, T.R, T.S.pack_off, T.S.scan_ws, T.S.scan_ws_bytes, (wb_stream)st);
}

extern "C" int wb_sdf_trace(const wb_octree* oct, const wb_sdf_desc* nef, int32_t lod_idx, const wb_rays* rays,
                            const float* nug_depth, int64_t Ng, const int64_t* ray_offsets,
                            int32_t num_steps, float step_size, float min_dis, int32_t want_normals, const wb_sdf_state* state,
                            float* xyz, float* depth, uint8_t* hit, float* normal, float* rgb, float* alpha, wb_stream s)
{
    WB_CHECK_ARG(rays != nullptr, "null rays");
    if (rays->num_rays == 0 || Ng == 0) return WB_OK;
    WbSdf m; int rc = wb_make_sdf(nef, &m); if (rc) return rc;
    WB_CHECK_ARG(lod_idx >= 0 && lod_idx < m.num_lods, "lod_idx out of range");
    WB_CHECK_ARG(m.multiscale == 1 || lod_idx == m.num_lods - 1, "'cat' grids feed the decoder all LODs: lod_idx must be num_lods-1");
    WbOct oc; rc = wb_make_oct(oct, m.base_lod + m.num_lods - 1, &oc); if (rc) return rc;
    WbSdfTrace T; rc = sdf_make_trace(rays, nug_depth, Ng, ray_offsets, num_steps, step_size, min_dis, state, &T); if (rc) return rc;
    WB_CHECK_ARG(xyz && depth && hit && alpha && (!want_normals || (normal && rgb)), "null output");
    T.nl = lod_idx + 1; T.want_normals = want_normals ? 1 : 0;
    T.o_xyz = xyz; T.o_depth = depth; T.o_hit = hit; T.o_normal = normal; T.o_rgb = rgb; T.o_alpha = alpha;
    cudaStream_t st = (cudaStream_t)s;
    rc = sdf_scan_packs(T, num_steps, st); if (rc) return rc;
    const int smem = m.smem_floats * 4;
    const void* kern = sdf_fast_shape(m) ? (const void*)wb_sdf_trace_kernel<16, 1> : (const void*)wb_sdf_trace_kernel<0, 0>;
    if (smem > 48 * 1024) WB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int per_sm = 0;
    WB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WB_SDF_THREADS, smem));
    WB_CHECK_ARG(per_sm >= 1, "sphere-trace kernel does not fit on an SM");
    int64_t ctas = (int64_t)wb_num_sms() * per_sm;                       // cooperative launch: every CTA resident
    const int64_t need = (T.R + WB_SDF_THREADS - 1) / WB_SDF_THREADS; if (ctas > need) ctas = need;
    void* args[] = { &oc, &m, &T };
    WB_CUDA(cudaLaunchCooperativeKernel(kern, dim3((unsigned)ctas), dim3(WB_SDF_THREADS), args, (size_t)smem, st));
    wb_count_launch();
    return WB_OK;
}

extern "C" int wb_sdf_phase(int32_t phase, const wb_rays* rays, const float* nug_depth, int64_t Ng, const int64_t* ray_offsets,
                            int32_t num_steps, int32_t iteration, float min_dis, const wb_sdf_state* state,
                            float* xyz, float* depth, uint8_t* hit, float* alpha, wb_stream s)
{
    WB_CHECK_ARG(rays != nullptr, "null rays");
    WB_CHECK_ARG(phase >= 0 && phase <= 4 && iteration >= 0 && iteration < (num_steps > 0 ? num_steps : 1), "bad phase / iteration");
    if (rays->num_rays == 0 || Ng == 0) return WB_OK;
    WbSdfTrace T; int rc = sdf_make_trace(rays, nug_depth, Ng, ray_offsets, num_steps, 1.0f, min_dis, state, &T); if (rc) return rc;
    WB_CHECK_ARG(phase != 4 || (xyz && depth && hit && alpha), "null output");
    T.o_xyz = xyz; T.o_depth = depth; T.o_hit = hit; T.o_alpha = alpha;
    cudaStream_t st = (cudaStream_t)s;
    if (phase == 0) { rc = sdf_scan_packs(T, num_steps, st); if (rc) return rc; }
    int64_t ctas = (T.R + WB_SDF_THREADS - 1) / WB_SDF_THREADS; const int64_t cap = (int64_t)wb_num_sms() * 8; if (ctas > cap) ctas = cap;
    // cursors alternate between the two buffers once per executed jump phase: iteration `it` reads buffer it & 1
    wb_sdf_phase_kernel<<<(unsigned)ctas, WB_SDF_THREADS, 0, st>>>(T, phase, iteration, iteration & 1);
    WB_LAUNCH_CHECK();
    return WB_OK;
}
