// wb_shade_tc.cu -- fused "shade" stage with tensor-core decoders (precision 1): tcgen05.mma + TMEM + TMA-staged weights.
//
// Numerics = the reference under torch.cuda.amp.autocast (nerf_hash.yaml:76 enable_amp: True): decoder operands in
// fp16, fp32 accumulation; unlike the reference the hash table is read as fp32 master (no per-call .half() copy,
// ops/grid.py:88-89), features are blended in fp32 and table gradients accumulate in fp32.
//
// Unit of work = a 128-sample sub-tile handled by a GROUP of 256 threads: row r of the tile == TMEM lane r is shared by two
// threads (column halves).  Per layer ("round", tc_round):  every thread writes its part of the fp16 operand tile (slab layout,
// wb_tc.cuh) -> fence -> group barrier -> two elected issuer threads launch the round's UMMA chains from a shared-memory issue
// table (A = sample tile, B = TMA-staged weight pack, D in TMEM; the bias is an init UMMA Ones x Bias^T) and commit to the
// group's mbarrier -> the group waits, tcgen05.ld's its accumulator columns, applies the activation, writes the next tile.
// Groups are independent (own named barrier, own mbarrier, own TMEM columns): the forward runs up to 3 one-group CTAs per SM, the
// backward one CTA of two groups (below) or of three / one wide group (wb_shade_tc_bwd3.cuh, the app/nerf decoder shape) per SM.
//
// Forward  (wb_shade_fwd_tc_kernel): gather 15 LODs x 8 corners (fp32 blend) -> decoders -> (r,g,b,sigma).  It also saves
//   the gathered feature rows (fp16, chunk-major [Kp0/8][S] x 16 B: coalesced both ways) for the backward.
// Backward (wb_mlp_bwd_tc_kernel here, wb_mlp_bwd3_tc_kernel in wb_shade_tc_bwd3.cuh): reloads those rows -- it touches neither the
//   hash table nor the octree -- recomputes the decoders (tiles stay in shared memory) and per layer issues
//     weight grad   acc_l[in, out] += X_l^T . dY_l   (both operands MN-major straight from the sample tiles; accumulators
//                                                     stay in TMEM for the whole kernel; a constant-one slab behind every
//                                                     X_l tile makes row `Kp_l` the bias gradient)
//     data grad     dX_l = dY_l . W_l                (weight pack read MN-major: no transposed copy)
//   and writes dL/dfeat as fp16 level-major planes [L][S][F] (the three-group kernel scatters them itself on F == 2 'cat' hash grids).
// Scatter  (wb_table_scatter_kernel, SIMT): lanes = consecutive samples; a thread builds its sample position once and walks all
//   LODs; per LOD, runs of lanes that fall into the same cell are summed with a segmented warp scan and only the last lane of a
//   run issues the reductions (x-neighbour entries that differ only in bit 0 as one 16-byte red.global.add.v4.f32).
//   Neighbouring samples of a ray share cells on all but the finest LODs.
// The per-ray view embedding (positional_embedder.py:51-66) is evaluated once per ray (wb_ray_embed_kernel), not per sample.
// Gradients are carried in fp16 under a power-of-two loss scale supplied on the device (no host sync) and unscaled in fp32
// at the two exits (table scatter, weight-gradient flush).
#include "wb_common.cuh"
#include "wb_featx.cuh"
#include "wb_tc.cuh"
#include <math.h>

#define TC_ML 16
constexpr int TC_ROWS = 128;          // samples per sub-tile (UMMA M)
constexpr int TC_GROUP = 256;         // threads per sub-tile group: 128 rows x 2 column halves
constexpr int TC_BWD_GROUPS = 2;      // sub-tile groups per CTA in the decoder backward
constexpr int TC_ISSUERS = 2;         // issuer warps per group (backward: weight grad | data grad)

struct WbTc {
    int nl_d, nl_c;
    int I[TC_ML], O[TC_ML], Kp[TC_ML], Np[TC_ML];
    int w_off[TC_ML], b_off[TC_ML];            // byte offsets in the parameter blob: weight pack, bias pack [Np x 16] (bias at k = 0)
    int has_bias;
    int ones_off;                              // byte offset (from smem base) of the constant [128 x 16] tile (feature 0 = 1) of the bias UMMA
    int src_w[TC_ML], src_b[TC_ML];
    int blob_bytes;
    int tile_off[TC_ML];                       // byte offset of layer l's INPUT tile inside a sub-tile region
    int dy_off[2];                             // byte offset (from smem base) of the dY tile of sub-tile 0/1
    int sub_off[2];                            // byte offset of the sub-tile regions
    int w_smem_off;                            // byte offset of the staged parameter blob
    int smem_bytes;
    int acc_col[TC_ML];                        // TMEM column of the weight-grad accumulator of layer l
    int work_col[2];                           // TMEM working accumulator of sub-tile 0/1
    int tmem_cols;
    int feat_dim, pos_dim, view_dim, pos_mode, pos_freq, view_mode, view_freq;
    int fits2;                                 // backward: the two-group kernel (all tiles retained) fits in shared memory
};

static int tc_round_up(int v, int m) { return (v + m - 1) / m * m; }

// ---- three-group decoder backward (wb_shade_tc_bwd3.cuh): shared-memory plan ----
constexpr int TC_B3_GROUPS = 3;
struct TcB3Plan {
    int P, Q, R, E, GB, blob_off, ones_off, smem_bytes;          // byte offsets (P..E from the group base, GB = group stride)
    int groups;                                                   // 3: every width <= 64;  1: widths up to 128 (hidden_dim = 128)
    int kind[8], acc_col[8], bias_col[8];                         // weight-grad accumulator of layer l: orientation (see below) and TMEM columns
    int acc_begin, acc_end;                                       // TMEM column range of all accumulators (zeroed at kernel start)
};

// host: shared-memory + tensor-memory plan; returns false when the configuration is outside the kernel's scope.
// Accumulator kinds (one group, 128-wide layers: 416 accumulator columns in the [in, out] orientation + 128 working columns would not
// fit the 512 TMEM columns, and a 128-row X^T leaves no row for the bias gradient):
//   0  acc[in, out] += X^T . dY, the tile's constant-one slab makes row Kp the bias gradient             (Np columns;  Kp < 128)
//   1  the same, bias gradient in a 16-column accumulator of its own: bias[out, 0] += dY^T . Ones         (Np + 16;     Kp == 128)
//   2  acc^T[out, in | 1] += dY^T . [X | 1]                                                              (Kp + 16;     used when Kp + 16 < Np)
// hidden_dim 128 on the app/nerf field: 48 + 32 + 64 + 144 + 32 = 320 accumulator columns + 128 working columns.
static bool tc_b3_plan(const WbTc& m, TcB3Plan* p)
{
    if (m.nl_d != 2 || m.nl_c != 3) return false;
    int maxw = 0, sumN = 0;
    for (int l = 0; l < 5; ++l) { maxw = max(maxw, max(m.Kp[l], m.Np[l])); sumN += m.Np[l]; }
    if (maxw > 128) return false;
    if (maxw > 64 && maxw != 128) return false;      // the one-group layout has been validated on B200 for 128-wide decoders only (hidden_dim 128);
                                                     // widths in between keep training on the fp32 kernels, as before
    // the hidden activation tiles X1, X3, X4 share the buffers P and Q, whose constant-one slab sits behind a maxw-wide tile: the
    // hidden width must BE the widest tile (true for app/nerf: 64-wide hidden layers over 32 / 42 inputs; a 32-wide decoder over a
    // 42-wide colour input would read its bias-gradient row from a stale slab)
    if (m.Kp[1] != maxw || m.Kp[3] != maxw || m.Kp[4] != maxw || m.Np[0] != maxw || m.Np[2] != maxw || m.Np[3] != maxw) return false;
    memset(p, 0, sizeof(*p));
    p->groups = (maxw <= 64 && sumN <= 512 - 3 * 64) ? 3 : 1;    // TMEM: 64 working columns per group (3 groups) / 128 (1 group) + the accumulators
    const int wc = p->groups == 3 ? 64 : 128;
    int col = p->groups * wc;
    p->acc_begin = col;
    for (int l = 0; l < 5; ++l) {
        p->kind[l] = p->groups == 3 ? 0 : (m.Kp[l] + 16 < m.Np[l] ? 2 : (m.Kp[l] >= 128 ? 1 : 0));
        p->acc_col[l] = col; col += p->kind[l] == 2 ? m.Kp[l] + 16 : m.Np[l];
        p->bias_col[l] = col; if (p->kind[l] == 1) col += 16;
    }
    p->acc_end = col;
    if (col > 512) return false;
    const int big = (maxw / 8 + 1) * 2048;                       // a maxw-wide tile + its constant-one slab
    const int small = (max(m.Np[1], m.Np[4]) / 8) * 2048;        // dY1 / dY4
    p->P = 0; p->Q = big; p->R = 2 * big; p->E = 3 * big; p->GB = 3 * big + small;
    p->blob_off = p->groups * p->GB;
    p->ones_off = p->blob_off + m.blob_bytes;
    int end = p->ones_off + 2 * 2048;
    // 16-slab read windows of the MN-major A operands (M = 128 feature rows): X tiles in R, and (kinds 1, 2) dY tiles in E
    const int window = (p->groups - 1) * p->GB + (p->groups == 3 ? p->R : p->E) + 16 * 2048;
    if (end < window) end = window;
    p->smem_bytes = end + 64;
    return p->smem_bytes + 6144 <= 227 * 1024;
}


static int tc_embed_dim(int mode, int freq) { return mode == 0 ? 0 : mode == 1 ? 3 : mode == 2 ? 6 * freq : 3 + 6 * freq; }

// returns WB_OK, or WB_ERR_INVALID with a message when the configuration does not fit the tensor-core path
int wb_tc_make(const wb_nef_desc* d, bool backward, WbTc* m, bool tmem_a = false)
{
    WB_CHECK_ARG(d->dens_layers >= 1 && d->col_layers >= 1 && d->dens_layers + d->col_layers <= TC_ML, "unsupported decoder depth");
    WB_CHECK_ARG(d->dens_params && d->col_params, "null decoder parameters");
    memset(m, 0, sizeof(*m));
    m->nl_d = d->dens_layers; m->nl_c = d->col_layers;
    m->feat_dim = d->multiscale == 0 ? d->num_lods * d->feature_dim : d->feature_dim;
    m->pos_mode = d->pos_mode; m->pos_freq = d->pos_freq; m->view_mode = d->view_mode; m->view_freq = d->view_freq;
    m->pos_dim = tc_embed_dim(d->pos_mode, d->pos_freq); m->view_dim = tc_embed_dim(d->view_mode, d->view_freq);
    WB_CHECK_ARG(d->dens_dims[0] == m->feat_dim + m->pos_dim, "decoder_density input width != grid features + position embedding");
    const int dout = d->dens_dims[d->dens_layers];
    WB_CHECK_ARG(dout >= 2 && dout <= 16, "tensor-core path: decoder_density output must be 2..16 wide");
    WB_CHECK_ARG(d->col_dims[0] == dout - 1 + m->view_dim, "decoder_color input width != density feats - 1 + view embedding");
    WB_CHECK_ARG(d->col_dims[d->col_layers] == 3, "decoder_color output must be 3 wide");
    const int nl = m->nl_d + m->nl_c;
    int off = 0, srcd = 0, srcc = 0, maxw = 0;
    for (int l = 0; l < nl; ++l) {
        const bool dens = l < m->nl_d;
        const int I = dens ? d->dens_dims[l] : d->col_dims[l - m->nl_d];
        const int O = dens ? d->dens_dims[l + 1] : d->col_dims[l - m->nl_d + 1];
        WB_CHECK_ARG(I >= 1 && I <= 128 && O >= 1 && O <= 128, "tensor-core path: layer widths must be <= 128");
        m->I[l] = I; m->O[l] = O; m->Kp[l] = tc_round_up(I, 16); m->Np[l] = tc_round_up(O, 16);
        m->w_off[l] = off; off += m->Kp[l] * m->Np[l] * 2;
        m->b_off[l] = off; off += m->Np[l] * 32;
        int& src = dens ? srcd : srcc;
        m->src_w[l] = src; src += I * O;
        if (d->has_bias) { m->src_b[l] = src; src += O; } else m->src_b[l] = -1;
        maxw = max(maxw, max(m->Kp[l], m->Np[l]));
    }
    m->blob_bytes = tc_round_up(off, 16);
    m->has_bias = d->has_bias ? 1 : 0;
    // shared memory map: [sub0 tiles][sub1 tiles][dY0][dY1][params][pad]
    int sub_bytes = 0;
    if (backward) {
        for (int l = 0; l < nl; ++l) { m->tile_off[l] = sub_bytes; sub_bytes += (m->Kp[l] / 8 + 1) * 2048; }   // + constant-one slab
    } else {
        // forward: every layer's input tile is overwritten in place by its output (the layer's UMMAs have completed before the
        // epilogue writes, and each thread only touches its own row) -> 16 KB per sub-tile, 4 CTAs per SM for the gather
        for (int l = 0; l < nl; ++l) m->tile_off[l] = 0;
        sub_bytes = (maxw / 8) * 2048;
    }
    const int groups = backward ? TC_BWD_GROUPS : 1;             // sub-tile groups per CTA
    m->sub_off[0] = 0; m->sub_off[1] = sub_bytes;
    int p = groups * sub_bytes;
    if (backward) { m->dy_off[0] = p; p += (maxw / 8) * 2048; m->dy_off[1] = p; p += (maxw / 8) * 2048; }
    m->w_smem_off = p; p += m->blob_bytes;
    m->ones_off = p; p += 2 * 2048;
    if (backward) {   // weight-grad MMAs read 16 slabs (M = 128 feature rows) from every X tile: keep that window inside the allocation
        const int need = m->sub_off[groups - 1] + m->tile_off[nl - 1] + 16 * 2048;
        if (p < need) p = need;
    }
    m->smem_bytes = p + 64;
    // static shared memory of the kernels (issue table, barriers): 3 KB forward, 5 KB backward
    const bool smem2 = m->smem_bytes + (backward ? 5632 : 3584) <= 227 * 1024;
    int col = 0;
    for (int gi = 0; gi < groups; ++gi) { m->work_col[gi] = col; col += maxw; }
    // forward TMEM-A variant (one group): work_col[1] is otherwise unused and holds the first column of the fp16 activation tile
    if (tmem_a && !backward) { m->work_col[1] = col; col += maxw / 2; }  // two halfs per 32-bit column
    if (backward) for (int l = 0; l < nl; ++l) { m->acc_col[l] = col; col += m->Np[l]; }
    m->fits2 = (smem2 && col <= 512) ? 1 : 0;
    if (!m->fits2) {       // the two-group backward retains every activation tile and keeps all accumulators [in, out]; the kernel of
        TcB3Plan plan3;    // wb_shade_tc_bwd3.cuh (uniform buffers, three groups or one wide group, mixed accumulator orientation) may still fit
        WB_CHECK_ARG(backward && tc_b3_plan(*m, &plan3),
                     !smem2 ? (backward ? "tensor-core path: decoder backward does not fit in shared memory (use precision 0)"
                                        : "tensor-core path: decoder does not fit in shared memory (use precision 0)")
                            : "tensor-core path: accumulators do not fit in TMEM (use precision 0)");
        col = 512;
    }
    int alloc = 32; while (alloc < col) alloc <<= 1;
    m->tmem_cols = alloc;
    return WB_OK;
}

// number of dL/dfeat planes and halfs per (plane, sample): 'cat' -> one plane per live LOD, 'sum' -> a single plane
static void tc_dfeat_shape(const wb_nef_desc* d, int* planes, int* width)
{
    *width = d->feature_dim;
    *planes = d->multiscale == 0 ? (d->lod_idx < d->num_lods ? d->lod_idx : d->num_lods) : 1;
    if (*planes < 0) *planes = 0;
}
static int64_t tc_align256(int64_t b) { return (b + 255) / 256 * 256; }

// workspace layout (bytes): [ray_embed: R * Kc * 2][dfeat: planes * S * F * 2 (backward only)]
int64_t wb_tc_workspace_bytes(const wb_nef_desc* nef, int64_t R, int64_t S, int backward)
{
    WbTc m; if (wb_tc_make(nef, false, &m)) return -1;
    int planes, width; tc_dfeat_shape(nef, &planes, &width);
    int64_t b = tc_align256(R * m.Kp[m.nl_d] * 2);
    if (backward) b += tc_align256((int64_t)planes * S * width * 2);
    return b + 256;
}
int wb_tc_supported(const wb_nef_desc* nef, int backward)
{
    WbTc m; if (wb_tc_make(nef, false, &m)) return 0;
    if (backward && wb_tc_make(nef, true, &m)) return 0;
    return 1;
}
// the features are only saved for a backward pass: refuse here (at forward time) if that pass cannot run
int64_t wb_tc_feat_bytes(const wb_nef_desc* nef, int64_t S)
{
    WbTc m; if (wb_tc_make(nef, true, &m) || wb_tc_make(nef, false, &m)) return -1;
    return (int64_t)m.Kp[0] * 2 * S + 256;
}

// ---- parameter blob: fp16 weight packs (wb_tc.cuh layout) + fp32 biases -------------------------------------------
__global__ void wb_tc_pack_kernel(WbTc m, const float* __restrict__ dens, const float* __restrict__ col, uint8_t* __restrict__ blob)
{
    const int nl = m.nl_d + m.nl_c;
    for (int l = 0; l < nl; ++l) {
        const float* src = l < m.nl_d ? dens : col;
        const int I = m.I[l], O = m.O[l], Kp = m.Kp[l], Np = m.Np[l];
        __half* w = reinterpret_cast<__half*>(blob + m.w_off[l]);
        for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < Kp * Np; e += gridDim.x * blockDim.x) {
            const int kc = e / (Np * 8), n = (e / 8) % Np, k = kc * 8 + (e & 7);      // element (n,k) at (k/8)*(Np*8) + n*8 + k%8 halves
            w[e] = __float2half_rn((n < O && k < I) ? src[m.src_w[l] + n * I + k] : 0.0f);
        }
        // bias pack B[Np x 16] (K-major, same layout as the weights): column k = 0 holds the bias.  An init UMMA
        // D = Ones[128 x 16] . B^T puts the bias into the accumulator; the layer UMMAs accumulate on top (fp16 bias: what
        // F.linear under autocast does)
        __half* b = reinterpret_cast<__half*>(blob + m.b_off[l]);
        for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < Np * 16; e += gridDim.x * blockDim.x) {
            const int kc = e / (Np * 8), n = (e / 8) % Np, k = kc * 8 + (e & 7);
            b[e] = __float2half_rn((k == 0 && n < O && m.src_b[l] >= 0) ? src[m.src_b[l] + n] : 0.0f);
        }
    }
}

int wb_tc_blob_floats(const wb_nef_desc* nef) { WbTc m; if (wb_tc_make(nef, false, &m)) return -1; return m.blob_bytes / 4; }

int wb_tc_pack(const wb_nef_desc* nef, float* blob, cudaStream_t st)
{
    WbTc m; int rc = wb_tc_make(nef, false, &m); if (rc) return rc;
    wb_tc_pack_kernel<<<16, 256, 0, st>>>(m, nef->dens_params, nef->col_params, reinterpret_cast<uint8_t*>(blob));
    WB_LAUNCH_CHECK();
    return WB_OK;
}

// ---- per-ray colour-input rows: zeros with the view embedding at features [dout-1, dout-1+view_dim) -----------------
__global__ void __launch_bounds__(128)
wb_ray_embed_kernel(WbTc m, const float* __restrict__ dirs, int64_t R, uint4* __restrict__ out)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const int Kc = m.Kp[m.nl_d], f0 = m.O[m.nl_d - 1] - 1;
    __align__(16) __half row[128];
    for (int i = 0; i < Kc; ++i) row[i] = __float2half_rn(0.0f);
    const float x = dirs[3 * r], y = dirs[3 * r + 1], z = dirs[3 * r + 2];
    int o = f0;
    if (m.view_mode == 1 || m.view_mode == 3) { row[o] = __float2half_rn(x); row[o + 1] = __float2half_rn(y); row[o + 2] = __float2half_rn(z); o += 3; }
    if (m.view_mode >= 2) {
        float band = 1.0f;
        for (int f = 0; f < m.view_freq; ++f) {
            const float w3[3] = { x * band, y * band, z * band };
            for (int c = 0; c < 3; ++c) {
                row[o + f * 3 + c] = __float2half_rn(sinf(w3[c]));
                row[o + 3 * m.view_freq + f * 3 + c] = __float2half_rn(cosf(w3[c]));
            }
            band *= 2.0f;
        }
    }
    const uint4* rv = reinterpret_cast<const uint4*>(row);
    for (int c = 0; c < Kc / 8; ++c) out[r * (Kc / 8) + c] = rv[c];
}

// ---------------------------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------------------------
struct TcIn {
    const float* origins; const float* dirs; const float* rec_t; const int32_t* rec_ray; int64_t S;
    const uint4* ray_embed;      // [R][Kc/8] rows prepared by wb_ray_embed_kernel
    uint4* x0_save;              // forward: optional [Kp0/8][S] copy of the density-decoder input rows
    const uint4* x0_saved;       // backward: the same buffer
    int64_t s_begin, s_end;      // backward kernels that take a sample range (a multiple of 128 .. s_end; s_end == 0: the whole [0, S)); S stays the plane stride
};

__device__ __forceinline__ void tile_store1(uint8_t* tile, int r, int f, float v)
{
    *reinterpret_cast<__half*>(tile + tc_slab_off(r, f)) = __float2half_rn(v);
}
__device__ __forceinline__ void tile_store8(uint8_t* tile, int r, int slab, const float v[8])
{
    uint4 q; q.x = tc_pack2(v[0], v[1]); q.y = tc_pack2(v[2], v[3]); q.z = tc_pack2(v[4], v[5]); q.w = tc_pack2(v[6], v[7]);
    *reinterpret_cast<uint4*>(tile + slab * 2048 + r * 16) = q;
}
// embedding (positional_embedder.py:51-66) written into tile features [f0, f0+dim)
__device__ __forceinline__ void tile_embed(uint8_t* tile, int r, int f0, int mode, int freq, float x, float y, float z)
{
    if (mode == 0) return;
    int o = f0;
    if (mode == 1 || mode == 3) { tile_store1(tile, r, o, x); tile_store1(tile, r, o + 1, y); tile_store1(tile, r, o + 2, z); o += 3; }
    if (mode == 1) return;
    float band = 1.0f;
    for (int f = 0; f < freq; ++f) {
        const float wx = x * band, wy = y * band, wz = z * band;
        tile_store1(tile, r, o + f * 3 + 0, sinf(wx)); tile_store1(tile, r, o + f * 3 + 1, sinf(wy)); tile_store1(tile, r, o + f * 3 + 2, sinf(wz));
        tile_store1(tile, r, o + 3 * freq + f * 3 + 0, cosf(wx)); tile_store1(tile, r, o + 3 * freq + f * 3 + 1, cosf(wy)); tile_store1(tile, r, o + 3 * freq + f * 3 + 2, cosf(wz));
        band *= 2.0f;
    }
}
// hash-grid gather of one sample -> features [0, feat_dim) of the X0 tile (fp32 blend, fp16 store)
// `half` (0/1): the two threads of a row split the work -- slab (4 LODs) k goes to half k & 1 on the F == 2 'cat' path, the
// generic paths are done by half 0 alone
__device__ __forceinline__ void tile_gather(const WbGrid& g, uint8_t* tile, int r, int half, float px, float py, float pz)
{
    const int L = g.L, F = g.F;
    if (g.multiscale == 0 && F == 2) {
        for (int l0 = 4 * half; l0 < L; l0 += 8) {              // 4 levels = 8 features = one slab row (16 B store)
            float v[8];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int l = l0 + q;
                if (l >= L || l >= g.lod_idx) { v[2 * q] = 0.0f; v[2 * q + 1] = 0.0f; continue; }       // hash_grid.py:226-229
                uint32_t idx[8]; float cf[8];
                wb_corner_setup(g, l, px, py, pz, idx, cf);
                const float2* tb = reinterpret_cast<const float2*>(g.table + g.begin[l] * 2);
                float2 c[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) c[j] = __ldg(tb + idx[j]);
                float a0 = c[0].x * cf[0], a1 = c[0].y * cf[0];
#pragma unroll
                for (int j = 1; j < 8; ++j) { a0 = fmaf(c[j].x, cf[j], a0); a1 = fmaf(c[j].y, cf[j], a1); }
                v[2 * q] = a0; v[2 * q + 1] = a1;
            }
            tile_store8(tile, r, l0 >> 2, v);
        }
    } else if (half != 0) {
        return;
    } else if (g.multiscale == 0) {
        for (int l = 0; l < L; ++l) {
            if (l >= g.lod_idx) { for (int f = 0; f < F; ++f) tile_store1(tile, r, l * F + f, 0.0f); continue; }
            uint32_t idx[8]; float cf[8];
            wb_corner_setup(g, l, px, py, pz, idx, cf);
            const float* tb = g.table + g.begin[l] * F;
            for (int f = 0; f < F; ++f) {
                float a = __ldg(tb + (int64_t)idx[0] * F + f) * cf[0];
#pragma unroll
                for (int j = 1; j < 8; ++j) a = fmaf(__ldg(tb + (int64_t)idx[j] * F + f), cf[j], a);
                tile_store1(tile, r, l * F + f, a);
            }
        }
    } else {
        float s[8];
#pragma unroll
        for (int f = 0; f < 8; ++f) s[f] = 0.0f;
        for (int l = 0; l < L; ++l) {
            uint32_t idx[8]; float cf[8];
            wb_corner_setup(g, l, px, py, pz, idx, cf);
            const float* tb = g.table + g.begin[l] * F;
#pragma unroll
            for (int f = 0; f < 8; ++f) if (f < F) {
                float a = __ldg(tb + (int64_t)idx[0] * F + f) * cf[0];
#pragma unroll
                for (int j = 1; j < 8; ++j) a = fmaf(__ldg(tb + (int64_t)idx[j] * F + f), cf[j], a);
                s[f] += a;
            }
        }
#pragma unroll
        for (int f = 0; f < 8; ++f) if (f < F) tile_store1(tile, r, f, s[f]);
    }
}
// zero features [f0, f1) of this thread's row
__device__ __forceinline__ void tile_zero(uint8_t* tile, int r, int f0, int f1) { for (int f = f0; f < f1; ++f) tile_store1(tile, r, f, 0.0f); }

// ---- optional phase timestamps (debug builds only: WB_EXTRA_NVCC_FLAGS=-DWB_TC_TIMING, read by tools/tc_timing.py) ----
#ifdef WB_TC_TIMING
#define TC_TS_N 1024
__device__ long long g_tc_ts[2][2][TC_TS_N];      // [kernel: 0 fwd, 1 bwd][thread 0 / (fwd: last thread, bwd: first thread of group 1)][event]
#define TC_TS(c) do { if (blockIdx.x == 0 && (threadIdx.x == 0 || threadIdx.x == ((c).tsk ? TC_GROUP : TC_GROUP - 1)) && (c).tsn < TC_TS_N) \
        g_tc_ts[(c).tsk][threadIdx.x ? 1 : 0][(c).tsn++] = clock64(); } while (0)
__device__ long long g_tc_ts2[2][TC_TS_N];        // thread 0 only: inside the issue branch (after elect+fence, after the UMMAs, after commit)
#define TC_TS2(c, n2) do { if (blockIdx.x == 0 && threadIdx.x == 0 && (n2) < TC_TS_N) g_tc_ts2[(c).tsk][(n2)++] = clock64(); } while (0)
extern "C" int wb_tc_timing_dump2(long long* out)
{ return (int)cudaMemcpyFromSymbol(out, g_tc_ts2, sizeof(long long) * 2 * TC_TS_N); }
__device__ long long g_tc_ts3[2][TC_TS_N];        // thread 0 only: hidden-layer epilogue (before tcgen05.ld, after its wait, after the stores)
#define TC_TS3(c) do { if (blockIdx.x == 0 && threadIdx.x == 0 && (c).tsn3 < TC_TS_N) g_tc_ts3[(c).tsk][(c).tsn3++] = clock64(); } while (0)
extern "C" int wb_tc_timing_dump3(long long* out)
{ return (int)cudaMemcpyFromSymbol(out, g_tc_ts3, sizeof(long long) * 2 * TC_TS_N); }
__device__ long long g_tc_ts4[2][64][16];        // thread 0: stamp before the chain and after every UMMA of the first 64 rounds
__device__ int g_tc_ts4_round[2];
extern "C" int wb_tc_timing_dump4(long long* out)
{ return (int)cudaMemcpyFromSymbol(out, g_tc_ts4, sizeof(long long) * 2 * 64 * 16); }
extern "C" int wb_tc_timing_dump(long long* out)
{ return (int)cudaMemcpyFromSymbol(out, g_tc_ts, sizeof(long long) * 2 * 2 * TC_TS_N); }
#else
#define TC_TS(c) do { } while (0)
#define TC_TS2(c, n2) do { } while (0)
#define TC_TS3(c) do { } while (0)
#endif

// Issue table (shared memory, built once per CTA): everything the issuer needs for one UMMA chain, so that the critical path
// after the group barrier is two LDS.128 (issued BEFORE the barrier) + the UTCHMMAs.  Deriving the descriptors from the
// kernel parameters instead costs ~400 cycles of dependent constant loads / uniform ALU per round (measured).
struct __align__(16) TcRec {
    uint32_t a_lo, a_hi, b_lo, b_hi;          // shared-memory descriptors of the first UMMA
    uint32_t idesc, tmem_d, nk_acc, adv;      // nk | (accumulate-from-start << 8); a advance | b advance << 16 (16-byte units)
};
enum { TC_K_FWD = 0, TC_K_BIAS = 1, TC_K_WGRAD = 2, TC_K_DGRAD = 3, TC_KINDS = 4,
       TC_K_FWD_TA = TC_K_WGRAD };           // forward kernels have no weight grad: the slot holds the A-from-TMEM chain of the TMEM-A variant

struct TcCtx {
    uint8_t* smem; uint64_t* bar; uint32_t tmem; uint32_t phase;
    const TcRec* tab;           // this group's records: tab[kind * TC_ML + layer]
    int g;                      // sub-tile group of this thread inside the CTA
    int r, h;                   // row of the sub-tile (== TMEM lane), column half
    int laneq;                  // 32*(warp%4): the TMEM lane quarter this warp may access
    int wig;                    // warp index inside the group (warp-uniform)
#ifdef WB_TC_TIMING
    int tsn, tsk, tsn2, tsn3;
#endif
};
__device__ __forceinline__ void tc_ctx_init(TcCtx& c, uint8_t* smem, uint64_t* bars, const TcRec* tab, uint32_t tmem, int kernel_id)
{
    const int tig = threadIdx.x & (TC_GROUP - 1);
    c.smem = smem; c.g = threadIdx.x / TC_GROUP; c.bar = bars + c.g; c.tmem = tmem; c.phase = 0;
    c.tab = tab + c.g * (TC_KINDS * TC_ML);
    c.r = tig & (TC_ROWS - 1); c.h = tig / TC_ROWS; c.laneq = ((tig >> 5) & 3) * 32;
    c.wig = __shfl_sync(0xffffffffu, tig >> 5, 0);
#ifdef WB_TC_TIMING
    c.tsn = 0; c.tsk = kernel_id; c.tsn2 = 0; c.tsn3 = 0;
#endif
}

// one record per (group, kind, layer) + the constant tile of the bias UMMA; called by all threads before the first round
__device__ __forceinline__ void tc_build_table(const WbTc& m, TcRec* tab, uint8_t* smem, uint32_t tmem, int groups, bool backward, bool ta = false)
{
    const int nl = m.nl_d + m.nl_c;
    const int e = threadIdx.x;
    if (e < TC_ROWS) {                                           // Ones[128 x 16]: feature 0 = 1, features 1..15 = 0
        uint4 one; one.x = 0x00003C00u; one.y = 0; one.z = 0; one.w = 0;
        *reinterpret_cast<uint4*>(smem + m.ones_off + e * 16) = one;
        *reinterpret_cast<uint4*>(smem + m.ones_off + 2048 + e * 16) = make_uint4(0, 0, 0, 0);
    }
    if (e >= groups * TC_KINDS * nl) return;
    const int l = e % nl, kind = (e / nl) % TC_KINDS, g = e / (nl * TC_KINDS);
    const uint32_t base = tc_smem_u32(smem);
    const int Np = m.Np[l], Kp = m.Kp[l];
    uint64_t da = 0, db = 0; uint32_t id = 0, d = 0, nk = 0, acc = 0, aadv = 0, badv = 0;
    if (kind == TC_K_FWD) {            // D_work[g] (+)= X_l . W_l^T
        da = tc_desc(base + m.sub_off[g] + m.tile_off[l], 2048, 128); db = tc_desc(base + m.w_smem_off + m.w_off[l], Np * 16, 128);
        id = tc_idesc(128, Np, 0, 0); d = tmem + m.work_col[g]; nk = Kp / 16; acc = m.has_bias; aadv = 4096 >> 4; badv = (2 * Np * 16) >> 4;
    } else if (kind == TC_K_BIAS) {    // D_work[g] = Ones . Bias_l^T
        da = tc_desc(base + m.ones_off, 2048, 128); db = tc_desc(base + m.w_smem_off + m.b_off[l], Np * 16, 128);
        id = tc_idesc(128, Np, 0, 0); d = tmem + m.work_col[g]; nk = m.has_bias ? 1 : 0;
    } else if (!backward && kind == TC_K_FWD_TA && ta) {   // D_work (+)= X_l[TMEM] . W_l^T ; a_lo = TMEM address, 8 columns per K step
        da = (uint64_t)(tmem + (uint32_t)m.work_col[1]); db = tc_desc(base + m.w_smem_off + m.w_off[l], Np * 16, 128);
        id = tc_idesc(128, Np, 0, 0); d = tmem + m.work_col[g]; nk = (uint32_t)(Kp / 16); acc = m.has_bias; aadv = 8; badv = (2 * Np * 16) >> 4;
    } else if (!backward) {
        nk = 0;
    } else if (kind == TC_K_WGRAD) {   // acc_l[in, out] += X_l^T . dY_l   (K = 128 samples)
        da = tc_desc(base + m.sub_off[g] + m.tile_off[l], 128, 2048); db = tc_desc(base + m.dy_off[g], 128, 2048);
        id = tc_idesc(128, Np, 1, 1); d = tmem + m.acc_col[l]; nk = 8; acc = 1; aadv = 256 >> 4; badv = 256 >> 4;
    } else {                           // D_work[g] = dY_l . W_l         (K = out features)
        da = tc_desc(base + m.dy_off[g], 2048, 128); db = tc_desc(base + m.w_smem_off + m.w_off[l], 128, Np * 16);
        id = tc_idesc(128, Kp, 0, 1); d = tmem + m.work_col[g]; nk = Np / 16; aadv = 4096 >> 4; badv = 256 >> 4;
    }
    TcRec r = { (uint32_t)da, (uint32_t)(da >> 32), (uint32_t)db, (uint32_t)(db >> 32), id, d, nk | (acc << 8), aadv | (badv << 16) };
    tab[(g * TC_KINDS + kind) * TC_ML + l] = r;
}
template <bool A_IN_TMEM = false>
__device__ __forceinline__ void tc_issue_rec(const uint4 q0, const uint4 q1, long long* ts = nullptr, int* tn = nullptr)
{
    uint64_t da = ((uint64_t)q0.y << 32) | q0.x, db = ((uint64_t)q0.w << 32) | q0.z;
    const int nk = (int)(q1.z & 0xffu);
    const uint32_t acc = q1.z >> 8, aadv = q1.w & 0xffffu, badv = q1.w >> 16;
    for (int kb = 0; kb < nk; ++kb) {
        if (A_IN_TMEM) tc_mma_ts(q1.y, (uint32_t)da, db, q1.x, acc | (uint32_t)(kb > 0));
        else tc_mma(q1.y, da, db, q1.x, acc | (uint32_t)(kb > 0));
        da += aadv; db += badv;
#ifdef WB_TC_TIMING
        if (ts && *tn < 16) ts[(*tn)++] = clock64();
#endif
    }
}

// One round of a sub-tile group: operand tiles written -> group barrier -> the group's two issuer warps launch their UMMA
// chains (warp 0: kind k0a then k0b; warp 1: k1; a negative kind = nothing) and commit to the group's mbarrier -> the group
// waits for all of them.
// Measured on B200 (tools/tc_timing.py), first version of this file: a round cost ~600-1200 cycles from barrier to completion and
// the epilogue of a 64-wide layer another ~1200; the tensor pipe was ~10 % busy.  What this version does about it:
//  (a) issue table + elect.sync in a warp-uniform branch (descriptors in uniform registers, UTCHMMAs back to back; the first
//      version's per-thread branch ran a one-lane waterfall loop of ~200 cycles per UMMA),
//  (b) weight-grad and data-grad chains issued by two different warps,
//  (c) bias added by an init UMMA (Ones x Bias^T) and relu fused into the fp32->fp16x2 conversion: the hidden-layer epilogue is
//      tcgen05.ld + 16 F2FP.RELU + 4 STS.128 instead of ~130 instructions,
//  (d) a row is shared by two threads (column halves),
//  (e) the groups of a CTA (backward) / the CTAs of an SM (forward) have independent barriers and overlap each other.
template <bool TA = false>          // TA: warp 0's second chain (k0b) reads its A operand from tensor memory
__device__ __forceinline__ void tc_round(TcCtx& c, int l, int k0a, int k0b, int k1)
{
    TC_TS(c);
    uint4 qa0 = make_uint4(0, 0, 0, 0), qa1 = qa0, qb0 = qa0, qb1 = qa0;
    if (c.wig < TC_ISSUERS) {                     // table reads do not depend on the barrier
        const int ka = c.wig == 0 ? k0a : k1, kb = c.wig == 0 ? k0b : -1;
        if (ka >= 0) { const uint4* p = reinterpret_cast<const uint4*>(c.tab + ka * TC_ML + l); qa0 = p[0]; qa1 = p[1]; }
        if (kb >= 0) { const uint4* p = reinterpret_cast<const uint4*>(c.tab + kb * TC_ML + l); qb0 = p[0]; qb1 = p[1]; }
    }
    tc_fence_smem_async();
    tc_fence_before();
    tc_group_sync(c.g + 1, TC_GROUP);
    TC_TS(c);
    if (c.wig < TC_ISSUERS) {
        if (tc_elect_one()) {
            tc_fence_after();
            TC_TS2(c, c.tsn2);
#ifdef WB_TC_TIMING
            long long* ts4 = nullptr; int tn4 = 0;
            if (blockIdx.x == 0 && threadIdx.x == 0 && c.tsn2 / 3 < 64) { ts4 = g_tc_ts4[c.tsk][c.tsn2 / 3]; ts4[tn4++] = clock64(); }
            if (((qa1.z | qb1.z) & 0xffu) != 0) { tc_issue_rec(qa0, qa1, ts4, &tn4); tc_issue_rec<TA>(qb0, qb1, ts4, &tn4); TC_TS2(c, c.tsn2); tc_commit(c.bar); }
#else
            if (((qa1.z | qb1.z) & 0xffu) != 0) { tc_issue_rec(qa0, qa1); tc_issue_rec<TA>(qb0, qb1); TC_TS2(c, c.tsn2); tc_commit(c.bar); }
#endif
            else tc_mbar_arrive(c.bar);
            TC_TS2(c, c.tsn2);
        }
        __syncwarp();
    }
    TC_TS(c);
    tc_mbar_wait(c.bar, c.phase);
    c.phase ^= 1u;
    tc_fence_after();
    TC_TS(c);
}

// Decoders of one 128-sample sub-tile, starting from an X0 tile that the group has already written.
// Returns (in registers, both column halves) the density-decoder output df[16] and the colour pre-activations c3[3].
// TA (default forward variant for the F == 2 cat grid): the activation tile lives in tensor memory (m.work_col[1]; lane = row, two halfs per column) and
// feeds the UMMAs as the A operand directly; nothing but the weights is in shared memory.
template <bool TA = false>
__device__ __forceinline__ void tc_decoders(const WbTc& m, TcCtx& c, const TcIn& in, int64_t ray, float df[16], float c3[3])
{
    uint8_t* sub = c.smem + m.sub_off[c.g];
    const int nl = m.nl_d + m.nl_c;
    const uint32_t arow = c.tmem + ((uint32_t)c.laneq << 16) + (uint32_t)(TA ? m.work_col[1] : 0);
    for (int l = 0; l < nl; ++l) {
        tc_round<TA>(c, l, TC_K_BIAS, TA ? TC_K_FWD_TA : TC_K_FWD, -1);   // accumulator = bias + X_l . W_l^T
        const uint32_t trow = c.tmem + ((uint32_t)c.laneq << 16) + m.work_col[c.g];
        const bool last_d = (l == m.nl_d - 1), last_c = (l == nl - 1);
        if (last_d) {
            tc_ld16(trow, df);
            // colour input = [df[1:], embed(ray_d)], zero padded (nerf.py:248-259): the per-ray row already holds the
            // embedding and the zero padding, only the first dout-1 (<= 15) features are per-sample.  16-byte chunk ch of the
            // row is written by column half ch & 1.
            uint8_t* tcol = sub + m.tile_off[l + 1];
            const int nd = m.O[l] - 1, nch = m.Kp[l + 1] / 8;
            const uint4* re = in.ray_embed + ray * nch;
            uint4 q = __ldg(re + c.h);
            __half* hq = reinterpret_cast<__half*>(&q);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                // feature 8*h + j <- df[8*h + j + 1]; select without dynamic register indexing
                const float dv = c.h == 0 ? df[(j + 1) & 15] : df[(j + 9) & 15];
                if (8 * c.h + j < nd) hq[j] = __float2half_rn(dv);
            }
            if (TA) {                                            // chunk ch = 8 features = 4 TMEM columns
                tc_st4(arow + c.h * 4, q);
                for (int ch = 2 + c.h; ch < nch; ch += 2) tc_st4(arow + ch * 4, __ldg(re + ch));
                tc_st_wait();
            } else {
                *reinterpret_cast<uint4*>(tcol + c.h * 2048 + c.r * 16) = q;
                for (int ch = 2 + c.h; ch < nch; ch += 2) *reinterpret_cast<uint4*>(tcol + ch * 2048 + c.r * 16) = __ldg(re + ch);
            }
        } else if (last_c) {
            float v[16]; tc_ld16(trow, v);
            c3[0] = v[0]; c3[1] = v[1]; c3[2] = v[2];
        } else {
            // hidden layer: relu(acc) -> next input tile (F2FP.RELU); column half h owns columns [64k + 32h, 64k + 32h + 32)
            uint8_t* tn = sub + m.tile_off[l + 1];
            const int Np = m.Np[l];
            for (int cc = c.h * 32; cc < Np; cc += 64) {
                float v[32];
                const int nq = (Np - cc >= 32) ? 4 : 2;
                TC_TS3(c);
                if (nq == 4) tc_ld32(trow + cc, v); else tc_ld16(trow + cc, v);
                TC_TS3(c);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (q >= nq) break;
                    uint4 o;
                    o.x = tc_pack2_relu(v[q * 8], v[q * 8 + 1]); o.y = tc_pack2_relu(v[q * 8 + 2], v[q * 8 + 3]);
                    o.z = tc_pack2_relu(v[q * 8 + 4], v[q * 8 + 5]); o.w = tc_pack2_relu(v[q * 8 + 6], v[q * 8 + 7]);
                    if (TA) tc_st4(arow + (cc >> 1) + q * 4, o);         // features cc + 8q .. +7 -> columns (cc + 8q) / 2 ..
                    else *reinterpret_cast<uint4*>(tn + ((cc >> 3) + q) * 2048 + c.r * 16) = o;
                }
                if (TA) tc_st_wait();
                TC_TS3(c);
            }
            // Np[l] == Kp[l+1] (both round_up(hidden,16)); padded outputs are relu(0 + 0) = 0
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// forward kernel: CTA = one group = one 128-sample sub-tile at a time; several CTAs per SM overlap gather / UMMA / epilogue
// ---------------------------------------------------------------------------------------------------------------
// F == 2 'cat' gather straight into the TMEM activation tile (TMEM-A variant): 4 LODs = 8 features = one 16-byte chunk =
// 4 TMEM columns of this thread's lane; the chunk is also what the backward wants saved.
__device__ __forceinline__ void tile_gather_ta(const WbGrid& g, uint32_t arow, int half, float px, float py, float pz,
                                               uint4* __restrict__ save, int64_t S, int64_t s, bool valid)
{
    for (int l0 = 4 * half; l0 < g.L; l0 += 8) {
        float v[8];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int l = l0 + q;
            if (l >= g.L || l >= g.lod_idx) { v[2 * q] = 0.0f; v[2 * q + 1] = 0.0f; continue; }       // hash_grid.py:226-229
            uint32_t idx[8]; float cf[8];
            wb_corner_setup(g, l, px, py, pz, idx, cf);
            const float2* tb = reinterpret_cast<const float2*>(g.table + g.begin[l] * 2);
            float2 c[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) c[j] = __ldg(tb + idx[j]);
            float a0 = c[0].x * cf[0], a1 = c[0].y * cf[0];
#pragma unroll
            for (int j = 1; j < 8; ++j) { a0 = fmaf(c[j].x, cf[j], a0); a1 = fmaf(c[j].y, cf[j], a1); }
            v[2 * q] = a0; v[2 * q + 1] = a1;
        }
        uint4 qv; qv.x = tc_pack2(v[0], v[1]); qv.y = tc_pack2(v[2], v[3]); qv.z = tc_pack2(v[4], v[5]); qv.w = tc_pack2(v[6], v[7]);
        tc_st4(arow + (uint32_t)(l0 >> 2) * 4u, qv);
        if (save != nullptr && valid) save[(int64_t)(l0 >> 2) * S + s] = qv;
    }
    tc_st_wait();
}

template <int MINB, bool TA, bool GX = false>   // MINB: resident CTAs per SM the register allocation is bounded for; TA: activations in tensor
                                                // memory; GX: triplanar / octree feature grid (wb_featx.cuh) instead of the hash grid
__global__ void __launch_bounds__(TC_GROUP, MINB)
wb_shade_fwd_tc_kernel(WbGrid g, WbGridX gx, WbTc m, const uint8_t* __restrict__ blob, TcIn in, float4* __restrict__ shaded)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bars[2];
    __shared__ uint32_t tmem_s;
    __shared__ TcRec itab[TC_KINDS * TC_ML];
    if (threadIdx.x == 0) {
        tc_mbar_init(&bars[0], TC_ISSUERS); tc_mbar_init(&bars[1], 1); tc_mbar_init_fence();
        tc_mbar_expect_tx(&bars[1], (uint32_t)m.blob_bytes);
        tc_bulk_g2s(smem + m.w_smem_off, blob, (uint32_t)m.blob_bytes, &bars[1]);      // TMA: parameters -> shared memory
    }
    if (threadIdx.x < 32) tc_tmem_alloc(&tmem_s, (uint32_t)m.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    tc_build_table(m, itab, smem, tmem_s, 1, false, TA);
    __syncthreads();
    tc_mbar_wait(&bars[1], 0);
    TcCtx c; tc_ctx_init(c, smem, bars, itab, tmem_s, 0);
    uint8_t* t0 = smem + m.sub_off[0] + m.tile_off[0];
    const int nch0 = m.Kp[0] / 8;
    const int64_t ntiles = (in.S + TC_ROWS - 1) / TC_ROWS;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        int64_t s = tile * TC_ROWS + c.r;
        const bool valid = s < in.S;
        if (!valid) s = in.S - 1;
        const int64_t ray = __ldg(in.rec_ray + s);
        const float t = __ldg(in.rec_t + s);
        const float px = wb_addcmul(__ldg(in.origins + 3 * ray), __ldg(in.dirs + 3 * ray), t);
        const float py = wb_addcmul(__ldg(in.origins + 3 * ray + 1), __ldg(in.dirs + 3 * ray + 1), t);
        const float pz = wb_addcmul(__ldg(in.origins + 3 * ray + 2), __ldg(in.dirs + 3 * ray + 2), t);
        // density-decoder input row: grid features (+ position embedding), zero padded to Kp; the two threads of a row split the LODs
        if (TA) {
            tile_gather_ta(g, c.tmem + ((uint32_t)c.laneq << 16) + (uint32_t)m.work_col[1], c.h, px, py, pz, in.x0_save, in.S, s, valid);
        } else {
            if (!GX) tile_gather(g, t0, c.r, c.h, px, py, pz);
            else if (c.h == 0) {
                // one thread of the row pair gathers all LODs.  Splitting the LODs over the pair (partial sums through shared memory for 'sum'
                // grids) was measured SLOWER on config 4 (231 -> 280 ms per 800^2 frame): the gather is latency-bound, the extra group
                // barrier and scratch traffic cost more than the halved chain saves
                wb_featx_gather(gx, px, py, pz, [&](int f, float v) { tile_store1(t0, c.r, f, v); });
            }
            if (c.h == 0) {
                tile_embed(t0, c.r, m.feat_dim, m.pos_mode, m.pos_freq, px, py, pz);
                tile_zero(t0, c.r, m.I[0], m.Kp[0]);
            }
            if (in.x0_save) {
                tc_group_sync(1, TC_GROUP);
                if (valid)
                    for (int ch = c.h; ch < nch0; ch += 2) in.x0_save[(int64_t)ch * in.S + s] = *reinterpret_cast<const uint4*>(t0 + ch * 2048 + c.r * 16);
            }
        }
        float df[16], c3[3];
        tc_decoders<TA>(m, c, in, ray, df, c3);
        if (valid && c.h == 0) {
            const float r = 1.0f / (1.0f + expf(-c3[0])), gg = 1.0f / (1.0f + expf(-c3[1])), b = 1.0f / (1.0f + expf(-c3[2]));
            shaded[s] = make_float4(r, gg, b, fmaxf(df[0], 0.0f));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tc_tmem_dealloc(c.tmem, (uint32_t)m.tmem_cols);
}

// set by wb_rf_workspace_holds_ray_rows(): the next backward of this thread finds the per-ray colour-input rows in its workspace already
static thread_local int g_tc_skip_embed = 0;
static thread_local int64_t g_tc_s_begin = 0, g_tc_s_end = 0;      // sample range of the next backward launches (0, 0 = everything); set by wb_tc_shade_bwd's chunked schedule
extern "C" int wb_rf_workspace_holds_ray_rows(int32_t yes) { g_tc_skip_embed = yes ? 1 : 0; return WB_OK; }

static int tc_launch_ray_embed(const WbTc& m, const wb_rays* rays, void* workspace, cudaStream_t st)
{
    const int64_t R = rays->num_rays;
    if (R == 0) return WB_OK;
    wb_ray_embed_kernel<<<(unsigned)((R + 127) / 128), 128, 0, st>>>(m, rays->dirs, R, reinterpret_cast<uint4*>(workspace));
    WB_LAUNCH_CHECK();
    return WB_OK;
}

// Launch shapes: the measured optimum on B200 for the app/nerf configuration (the sweeps are in profiles/README.md)
constexpr int TC_FWD_CTAS = 3;                 // forward CTAs per SM at most (4 measured slower: 4.26 vs 3.19 ms)
constexpr int TC_WIDE_CHUNKS = 4;              // sample chunks of the wide-decoder backward schedule (wb_tc_shade_bwd)
constexpr int64_t TC_WIDE_MIN_S = 1 << 20;     // below this many samples the chunked schedule is not worth its launches
constexpr int TC_SCATTER_LPB = 16;             // LODs per CTA row of the table scatter
constexpr int TC_SCATTER_CTAS = 16;            // table-scatter CTAs per SM

int wb_tc_shade_fwd(const wb_nef_desc* nef, const float* blob, const wb_rays* rays, const float* rec_t, const int32_t* rec_ray,
                    int64_t S, float* shaded, void* feat_save, void* workspace, cudaStream_t st)
{
    WbGrid g; int rc = wb_make_grid(nef, &g); if (rc) return rc;
    WbGridX gx; rc = wb_make_gridx(nef, false, &gx); if (rc) return rc;
    // Activations in tensor memory, A operand read from TMEM (wb_tc.cuh tc_mma_ts): measured 2.86 ms on the 1024^2 frame against
    // 3.10 ms for the shared-memory tile, same results.  Applies to the specialised F == 2 'cat' gather without position embedding,
    // whose rows are whole 16-byte chunks; every other grid keeps the shared-memory tile.
    const bool ta = nef->grid_kind == 0 && nef->feature_dim == 2 && nef->multiscale == 0 && nef->pos_mode == 0 &&
                    (nef->num_lods * nef->feature_dim) % 16 == 0;
    WbTc m; rc = wb_tc_make(nef, false, &m, ta); if (rc) return rc;
    if (ta) {   // no activation tile in shared memory: the parameter blob and the bias tile move to the front
        const int tile = m.w_smem_off;
        m.w_smem_off -= tile; m.ones_off -= tile; m.smem_bytes -= tile;
    }
    WB_CHECK_ARG(workspace != nullptr, "precision 1 needs the workspace (wb_rf_workspace_bytes)");
    rc = tc_launch_ray_embed(m, rays, workspace, st); if (rc) return rc;
    TcIn in = { rays->origins, rays->dirs, rec_t, rec_ray, S, reinterpret_cast<const uint4*>(workspace), reinterpret_cast<uint4*>(feat_save), nullptr };
    // CTAs per SM: each is one sub-tile group; more groups in flight hide the gather and round latencies (measured sweep in
    // profiles/README.md).  The register bound of the instantiation must match, or the hardware silently runs fewer.
    // The generic grids keep more state per thread.  Triplanar (12 planes x 4 texel loads in flight): 3 CTAs per SM at 80 registers beat 2
    // at 128 despite 144 B of spills (config 4 forward 105 -> 88 ms measured); the octree gather (up to 32 accumulators) stays at 2.
    int per_sm = (227 * 1024) / (m.smem_bytes + 4096);
    per_sm = max(2, min(min(per_sm, 512 / m.tmem_cols), gx.kind == 2 ? 2 : TC_FWD_CTAS));
    // [CTAs per SM - 2][shared-memory tile, TMEM-A, feature grid]
    using FwdKernel = decltype(&wb_shade_fwd_tc_kernel<2, false>);
    static const FwdKernel kerns[2][3] = { { wb_shade_fwd_tc_kernel<2, false>, wb_shade_fwd_tc_kernel<2, true>, wb_shade_fwd_tc_kernel<2, false, true> },
                                           { wb_shade_fwd_tc_kernel<3, false>, wb_shade_fwd_tc_kernel<3, true>, wb_shade_fwd_tc_kernel<3, false, true> } };
    const int variant = gx.kind != 0 ? 2 : ta ? 1 : 0;
    const FwdKernel kern = kerns[per_sm - 2][variant];
    {   // function attributes are driver calls that can wait behind other driver work (e.g. an NVML poll): set them once, not per launch
        static int64_t done_for[2][3] = { { -1, -1, -1 }, { -1, -1, -1 } };
        if (done_for[per_sm - 2][variant] != WB_ATTR_KEY(m.smem_bytes)) {
            WB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, m.smem_bytes));
            WB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout,
                                         min(100, (per_sm * (m.smem_bytes + 4096) * 100) / (228 * 1024) + 1)));
            done_for[per_sm - 2][variant] = WB_ATTR_KEY(m.smem_bytes);
        }
    }
    const int64_t ntiles = (S + TC_ROWS - 1) / TC_ROWS;
    int64_t grid = (int64_t)wb_num_sms() * per_sm; if (grid > ntiles) grid = ntiles;
    kern<<<(unsigned)grid, TC_GROUP, m.smem_bytes, st>>>(g, gx, m, reinterpret_cast<const uint8_t*>(blob), in, reinterpret_cast<float4*>(shaded));
    WB_LAUNCH_CHECK();
    return WB_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// decoder backward kernel: CTA = TC_BWD_GROUPS groups (one per SM: TMEM holds the weight-grad accumulators), each group walks
// its own sequence of 128-sample sub-tiles with its own barriers, so the groups drift out of phase and overlap
// ---------------------------------------------------------------------------------------------------------------
struct TcGrads { float* gdens; float* gcol; const float* scale; __half* dfeat; int planes, width; };

__global__ void __launch_bounds__(TC_BWD_GROUPS * TC_GROUP, 1)
wb_mlp_bwd_tc_kernel(WbTc m, const uint8_t* __restrict__ blob, TcIn in, const float4* __restrict__ g_shaded, TcGrads G)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bars[TC_BWD_GROUPS + 1];
    __shared__ uint32_t tmem_s;
    __shared__ TcRec itab[TC_BWD_GROUPS * TC_KINDS * TC_ML];
    const int nl = m.nl_d + m.nl_c;
    if (threadIdx.x == 0) {
        for (int i = 0; i < TC_BWD_GROUPS; ++i) tc_mbar_init(&bars[i], TC_ISSUERS);
        tc_mbar_init(&bars[TC_BWD_GROUPS], 1); tc_mbar_init_fence();
        tc_mbar_expect_tx(&bars[TC_BWD_GROUPS], (uint32_t)m.blob_bytes);
        tc_bulk_g2s(smem + m.w_smem_off, blob, (uint32_t)m.blob_bytes, &bars[TC_BWD_GROUPS]);
    }
    if (threadIdx.x < 32) tc_tmem_alloc(&tmem_s, (uint32_t)m.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    tc_build_table(m, itab, smem, tmem_s, TC_BWD_GROUPS, true);
    TcCtx c; tc_ctx_init(c, smem, bars, itab, tmem_s, 1);
    uint8_t* sub = smem + m.sub_off[c.g];
    // constant-one slab behind every input tile: feature 0 = 1, features 1..7 = 0  (bias gradient row of the weight grad)
    for (int l = c.h; l < nl; l += 2) {
        uint4 one; one.x = 0x00003C00u; one.y = 0; one.z = 0; one.w = 0;           // fp16 1.0 in the low half
        *reinterpret_cast<uint4*>(sub + m.tile_off[l] + (m.Kp[l] / 8) * 2048 + c.r * 16) = one;
    }
    if (threadIdx.x < 128) {                                       // zero the resident weight-grad accumulators (all 128 lanes)
        const uint32_t tr = c.tmem + ((uint32_t)c.laneq << 16);
        for (int l = 0; l < nl; ++l)
            for (int cc = 0; cc < m.Np[l]; cc += 16) tc_st16_zero(tr + m.acc_col[l] + cc);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    tc_mbar_wait(&bars[TC_BWD_GROUPS], 0);
    const float scale = __ldg(G.scale), inv_scale = 1.0f / scale;
    uint8_t* dyt = smem + m.dy_off[c.g];
    uint8_t* t0 = sub + m.tile_off[0];
    const int nch0 = m.Kp[0] / 8;
    const int64_t ntiles = (in.S + TC_ROWS - 1) / TC_ROWS;
    const float z8[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
    for (int64_t tile = (int64_t)blockIdx.x * TC_BWD_GROUPS + c.g; tile < ntiles; tile += (int64_t)gridDim.x * TC_BWD_GROUPS) {
        int64_t s = tile * TC_ROWS + c.r;
        const bool valid = s < in.S;
        if (!valid) s = in.S - 1;
        const int64_t ray = __ldg(in.rec_ray + s);
        for (int ch = c.h; ch < nch0; ch += 2)                     // saved density-decoder input row (coalesced 16 B per lane)
            *reinterpret_cast<uint4*>(t0 + ch * 2048 + c.r * 16) = __ldg(in.x0_saved + (int64_t)ch * in.S + s);
        float df[16], c3[3];
        tc_decoders(m, c, in, ray, df, c3);
        float4 go = valid ? __ldg(g_shaded + s) : make_float4(0, 0, 0, 0);
        // ---- colour decoder, last layer: dY = dL/d(pre-sigmoid), zero padded ----
        {
            if (c.h == 0) {
                const float r = 1.0f / (1.0f + expf(-c3[0])), gg = 1.0f / (1.0f + expf(-c3[1])), b = 1.0f / (1.0f + expf(-c3[2]));
                float v[8] = { go.x * r * (1.0f - r) * scale, go.y * gg * (1.0f - gg) * scale, go.z * b * (1.0f - b) * scale, 0, 0, 0, 0, 0 };
                tile_store8(dyt, c.r, 0, v);
            }
            for (int sl = 1 + c.h; sl < m.Np[nl - 1] / 8; sl += 2) tile_store8(dyt, c.r, sl, z8);
        }
        const uint32_t trow = c.tmem + ((uint32_t)c.laneq << 16) + m.work_col[c.g];
        for (int l = nl - 1; l >= 0; --l) {
            tc_round(c, l, TC_K_WGRAD, -1, TC_K_DGRAD);
            // D_work row = dL/d(input of layer l), Kp[l] wide
            if (l == m.nl_d) {
                // first colour layer: inputs [df[1:dout], embed(ray_d)]; only the first dout-1 carry gradient (nerf.py:259)
                float v[16]; tc_ld16(trow, v);
                const int dout = m.O[m.nl_d - 1];
                float gdf[16];
                gdf[0] = (df[0] > 0.0f) ? go.w * scale : 0.0f;   // relu' of density (nerf.py:263)
#pragma unroll
                for (int j = 1; j < 16; ++j) gdf[j] = (j < dout) ? v[j - 1] : 0.0f;
                if (c.h == 0) tile_store8(dyt, c.r, 0, gdf); else tile_store8(dyt, c.r, 1, gdf + 8);
                for (int sl = 2 + c.h; sl < m.Np[l - 1] / 8; sl += 2) tile_store8(dyt, c.r, sl, z8);
            } else if (l == 0) {
                // dL/d(grid features) -> fp16 planes [plane][S][width] (still loss-scaled); tcgen05.ld is warp-collective
                const int W = G.width, nfe = G.planes * W;
                for (int f0 = c.h * 16; f0 < nfe; f0 += 32) {
                    float v[16]; tc_ld16(trow + f0, v);
                    if (!valid) continue;
                    if (W == 2) {
#pragma unroll
                        for (int qq = 0; qq < 8; ++qq) {
                            const int pl = (f0 >> 1) + qq;
                            if (pl < G.planes) reinterpret_cast<__half2*>(G.dfeat)[(int64_t)pl * in.S + s] = __floats2half2_rn(v[2 * qq], v[2 * qq + 1]);
                        }
                    } else {
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) {
                            const int fe = f0 + jj;
                            if (fe < nfe) G.dfeat[((int64_t)(fe / W) * in.S + s) * W + (fe % W)] = __float2half_rn(v[jj]);
                        }
                    }
                }
            } else {
                // hidden layer input: apply relu' from the retained activation tile, write the next dY (Np[l-1] == Kp[l])
                const uint8_t* xt = sub + m.tile_off[l];
                const int Kp = m.Kp[l];
                for (int cc = c.h * 32; cc < Kp; cc += 64) {
                    float v[32];
                    const int nq = (Kp - cc >= 32) ? 4 : 2;
                    if (nq == 4) tc_ld32(trow + cc, v); else tc_ld16(trow + cc, v);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        if (q >= nq) break;
                        // relu'(x) as a 16-bit lane mask of the retained fp16 activation (>= 0 by construction)
                        const uint4 a = *reinterpret_cast<const uint4*>(xt + ((cc >> 3) + q) * 2048 + c.r * 16);
                        const __half2 z2 = __float2half2_rn(0.0f);
                        uint4 o;
                        o.x = tc_pack2(v[q * 8], v[q * 8 + 1]) & __hgt2_mask(*reinterpret_cast<const __half2*>(&a.x), z2);
                        o.y = tc_pack2(v[q * 8 + 2], v[q * 8 + 3]) & __hgt2_mask(*reinterpret_cast<const __half2*>(&a.y), z2);
                        o.z = tc_pack2(v[q * 8 + 4], v[q * 8 + 5]) & __hgt2_mask(*reinterpret_cast<const __half2*>(&a.z), z2);
                        o.w = tc_pack2(v[q * 8 + 6], v[q * 8 + 7]) & __hgt2_mask(*reinterpret_cast<const __half2*>(&a.w), z2);
                        *reinterpret_cast<uint4*>(dyt + ((cc >> 3) + q) * 2048 + c.r * 16) = o;
                    }
                }
            }
        }
    }
    // ---- flush weight / bias gradient accumulators (TMEM rows = input feature, row Kp = bias) ----
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (threadIdx.x < 128) {
        const int row = threadIdx.x;
        const uint32_t tr = c.tmem + ((uint32_t)c.laneq << 16);
        for (int l = 0; l < nl; ++l) {
            float* gbase = l < m.nl_d ? G.gdens : G.gcol;
            const int I = m.I[l], O = m.O[l];
            // all 32 lanes of a warp must execute tcgen05.ld: decide per warp, predicate the stores per lane
            const int wrow0 = row & ~31;
            if (wrow0 > m.Kp[l]) continue;
            for (int cc = 0; cc < m.Np[l]; cc += 16) {
                float v[16]; tc_ld16(tr + m.acc_col[l] + cc, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int o = cc + j;
                    if (o >= O) continue;
                    const float val = v[j] * inv_scale;
                    if (row < I) { if (val != 0.0f) atomicAdd(gbase + m.src_w[l] + o * I + row, val); }
                    else if (row == m.Kp[l] && m.src_b[l] >= 0) atomicAdd(gbase + m.src_b[l] + o, val);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tc_tmem_dealloc(c.tmem, (uint32_t)m.tmem_cols);
}

// ---------------------------------------------------------------------------------------------------------------
// table scatter: dL/dfeat planes -> hash table (hashgrid_interpolate_cuda.cu:151-160), with warp-level run merging
// ---------------------------------------------------------------------------------------------------------------
template <int F>   // F == 2: the run sums travel through the warp scan as loss-scaled fp16 pairs (one shuffle per corner) and the corner
                   // entries come from wb_corner_indices (one multiply per axis); F == 0: any g.F, 8 x wb_hash_idx and fp32 run sums
__global__ void __launch_bounds__(256)
wb_table_scatter_kernel(WbGrid g, TcIn in, const __half* __restrict__ dfeat, int planes, int levels, int lpb,
                        const float* __restrict__ scale_p, float* __restrict__ gtable, int pair_v4)
{
    const int l_begin = blockIdx.y * lpb, l_end = min(levels, l_begin + lpb);     // this CTA's LODs; the sample position is built once for all of them
    const int lane = threadIdx.x & 31;
    const float scale = __ldg(scale_p), inv_scale = 1.0f / scale;
    const int Fr = F > 0 ? F : g.F;
    const int64_t s_end = in.s_end ? in.s_end : in.S;
    const int64_t nwork = in.s_begin + ((s_end - in.s_begin + 31) & ~(int64_t)31);            // whole warps
    for (int64_t s = in.s_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < nwork; s += (int64_t)gridDim.x * blockDim.x) {
        const bool valid = s < s_end;
        float px = 0.0f, py = 0.0f, pz = 0.0f;
        if (valid) {
            const int64_t ray = __ldg(in.rec_ray + s);
            const float t = __ldg(in.rec_t + s);
            px = wb_addcmul(__ldg(in.origins + 3 * ray), __ldg(in.dirs + 3 * ray), t);
            py = wb_addcmul(__ldg(in.origins + 3 * ray + 1), __ldg(in.dirs + 3 * ray + 1), t);
            pz = wb_addcmul(__ldg(in.origins + 3 * ray + 2), __ldg(in.dirs + 3 * ray + 2), t);
        }
        __half2 gnext = __float2half2_rn(0.0f);                  // F == 2: the next LOD's gradient is fetched one LOD ahead
        if (F == 2 && valid && l_begin < l_end)
            gnext = reinterpret_cast<const __half2*>(dfeat)[(int64_t)(g.multiscale == 0 ? l_begin : 0) * in.S + s];
        for (int l = l_begin; l < l_end; ++l) {
            const int pl = g.multiscale == 0 ? l : 0;
            float* tb = gtable + g.begin[l] * Fr;
            const bool pair_ok = pair_v4 && ((reinterpret_cast<uintptr_t>(tb) & 15u) == 0);       // level base 16-byte aligned
            uint32_t idx[8]; float cf[8]; uint64_t key = ~0ull - (uint64_t)lane;    // invalid lanes never merge
            float gv[F > 0 ? F : 8];
#pragma unroll
            for (int f = 0; f < (F > 0 ? F : 8); ++f) gv[f] = 0.0f;
            if (valid) {
                int ix, iy, iz; float wx, wy, wz, jx, jy, jz;
                wb_cell(px, g.hres[l], g.hi[l], ix, wx, jx); wb_cell(py, g.hres[l], g.hi[l], iy, wy, jy); wb_cell(pz, g.hres[l], g.hi[l], iz, wz, jz);
                key = (uint64_t)ix | ((uint64_t)iy << 20) | ((uint64_t)iz << 40);
                const float xy00 = jx * jy, xy01 = jx * wy, xy10 = wx * jy, xy11 = wx * wy;
                cf[0] = xy00 * jz; cf[1] = xy00 * wz; cf[2] = xy01 * jz; cf[3] = xy01 * wz;
                cf[4] = xy10 * jz; cf[5] = xy10 * wz; cf[6] = xy11 * jz; cf[7] = xy11 * wz;
                if (F == 2) wb_corner_indices(g, l, ix, iy, iz, idx);
                else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) idx[j] = wb_hash_idx(ix + ((j & 4) >> 2), iy + ((j & 2) >> 1), iz + (j & 1), g.res[l], g.Tmask, g.dense[l]);
                }
                if (F == 2) {
                    const float2 gg = __half22float2(gnext);
                    gv[0] = gg.x * inv_scale; gv[1] = gg.y * inv_scale;
                    if (l + 1 < l_end) gnext = reinterpret_cast<const __half2*>(dfeat)[(int64_t)(g.multiscale == 0 ? l + 1 : 0) * in.S + s];
                } else {
                    for (int f = 0; f < Fr; ++f) gv[f] = __half2float(dfeat[((int64_t)pl * in.S + s) * Fr + f]) * inv_scale;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) { idx[j] = 0; cf[j] = 0.0f; }
            }
            // runs of consecutive lanes with the same cell
            const uint64_t kprev = __shfl_up_sync(0xffffffffu, key, 1);
            const bool head = (lane == 0) || (kprev != key);
            const uint32_t heads = __ballot_sync(0xffffffffu, head);
            const int run_head = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
            const int dist = lane - run_head;
            const bool tail = (lane == 31) || ((heads >> (lane + 1)) & 1u);
            int maxd = dist;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) maxd = max(maxd, __shfl_xor_sync(0xffffffffu, maxd, o));
            if (F == 2) {
                float v0[8], v1[8];
                if (maxd > 0) {
                    // gradients arrive as fp16 anyway: scan the (still loss-scaled) products as half2, unscale after the scan
                    const float s0 = gv[0] * scale, s1 = gv[1] * scale;
                    __half2 h[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) h[j] = __floats2half2_rn(s0 * cf[j], s1 * cf[j]);
                    for (int o = 1; o <= maxd; o <<= 1) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const __half2 a = __shfl_up_sync(0xffffffffu, h[j], o);
                            if (dist >= o) h[j] = __hadd2(h[j], a);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) { const float2 f = __half22float2(h[j]); v0[j] = f.x * inv_scale; v1[j] = f.y * inv_scale; }
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) { v0[j] = gv[0] * cf[j]; v1[j] = gv[1] * cf[j]; }
                    for (int o = 1; o <= maxd; o <<= 1) {               // segmented inclusive scan (warp-uniform trip count)
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float a = __shfl_up_sync(0xffffffffu, v0[j], o), b = __shfl_up_sync(0xffffffffu, v1[j], o);
                            if (dist >= o) { v0[j] += a; v1[j] += b; }
                        }
                    }
                }
                if (tail && valid) {
                    // corners j and j + 4 are x-neighbours at the same (y, z).  When their entries differ only in bit 0 (dense level with
                    // an even index; hashed level with an even x, because (x | 1) ^ A == (x ^ A) ^ 1) the two 8-byte updates are one
                    // aligned 16-byte red.global.add.v4.f32 (measured: -6 % kernel time).
                    float2* t2 = reinterpret_cast<float2*>(tb);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t i0 = idx[j], i1 = idx[j + 4];
                        const bool nz0 = (v0[j] != 0.0f || v1[j] != 0.0f), nz1 = (v0[j + 4] != 0.0f || v1[j + 4] != 0.0f);
                        if (pair_ok && ((i0 ^ i1) == 1u)) {
                            if (nz0 || nz1) {
                                const float4 val = (i0 & 1u) ? make_float4(v0[j + 4], v1[j + 4], v0[j], v1[j]) : make_float4(v0[j], v1[j], v0[j + 4], v1[j + 4]);
                                atomicAdd(reinterpret_cast<float4*>(t2 + (i0 & ~1u)), val);
                            }
                        } else {
                            if (nz0) atomicAdd(t2 + i0, make_float2(v0[j], v1[j]));
                            if (nz1) atomicAdd(t2 + i1, make_float2(v0[j + 4], v1[j + 4]));
                        }
                    }
                }
            } else {
                for (int f = 0; f < Fr; ++f) {
                    float v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = gv[f] * cf[j];
                    for (int o = 1; o <= maxd; o <<= 1) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) { const float a = __shfl_up_sync(0xffffffffu, v[j], o); if (dist >= o) v[j] += a; }
                    }
                    if (tail && valid) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) if (v[j] != 0.0f) atomicAdd(tb + (int64_t)idx[j] * Fr + f, v[j]);
                    }
                }
            }
        }
    }
}

// dL/dfeat planes -> triplanar planes / octree feature levels (kinds 1, 2): one thread per sample, lanes = consecutive samples.
// Triplanar: consecutive samples of a ray stay in the same texel cell for several steps on the coarse planes (8 / 4 / 2 / 1 samples per
// cell on the four LODs of config 4), and the plane reductions are the wall of that configuration (6.3e10 per 800^2 frame at the L2
// reduction rate): runs of lanes with the same (LOD, plane, cell) are summed with a segmented warp scan -- 4 texel weights x C channels
// per lane -- and only the last lane of a run issues the reductions, as the hash-grid scatter does for its cells.
__global__ void __launch_bounds__(256)
wb_featx_scatter_kernel(WbGridX gx, TcIn in, const __half* __restrict__ dfeat, int width, const float* __restrict__ scale_p)
{
    const float inv_scale = 1.0f / __ldg(scale_p);
    const int lane = threadIdx.x & 31;
    const int64_t nwork = (in.S + 31) & ~(int64_t)31;            // whole warps
    for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < nwork; s += (int64_t)gridDim.x * blockDim.x) {
        const bool valid = s < in.S;
        float px = 0.0f, py = 0.0f, pz = 0.0f;
        if (valid) {
            const int64_t ray = __ldg(in.rec_ray + s);
            const float t = __ldg(in.rec_t + s);
            px = wb_addcmul(__ldg(in.origins + 3 * ray), __ldg(in.dirs + 3 * ray), t);
            py = wb_addcmul(__ldg(in.origins + 3 * ray + 1), __ldg(in.dirs + 3 * ray + 1), t);
            pz = wb_addcmul(__ldg(in.origins + 3 * ray + 2), __ldg(in.dirs + 3 * ray + 2), t);
        }
        auto grad = [&](int f) {                                  // feature f lives in plane f / width at column f % width
            return __half2float(dfeat[((int64_t)(f / width) * in.S + s) * width + (f % width)]) * inv_scale;
        };
        if (gx.kind != 1 || gx.C > 4) {                           // octree grid (or wide triplanar channels): no merging
            if (valid) wb_featx_scatter(gx, px, py, pz, grad);
            continue;
        }
        const int C = gx.C;
        float gsum[3][4];                                         // 'sum' grids: every LOD receives the same dL/dfeat -> loaded once per sample
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
            for (int c = 0; c < 4; ++c) gsum[p][c] = (gx.sum && valid && c < C) ? grad(p * C + c) : 0.0f;
        for (int l = 0; l < gx.nl; ++l) {
            const int size = gx.res[l] + 1; const int64_t hw = (int64_t)size * size;
#pragma unroll
            for (int p = 0; p < 3; ++p) {
                WbBilinear b = wb_tp_setup(px, py, pz, p, size);
                float v[4][4];                                    // [texel nw, ne, sw, se][channel]
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float g = gx.sum ? gsum[p][c] : ((valid && c < C) ? grad((l * 3 + p) * C + c) : 0.0f);
                    v[0][c] = g * b.nw; v[1][c] = g * b.ne; v[2][c] = g * b.sw; v[3][c] = g * b.se;
                }
                const int key = valid ? b.o00 : -1 - lane;        // invalid lanes never merge
                const int kprev = __shfl_up_sync(0xffffffffu, key, 1);
                const bool head = (lane == 0) || (kprev != key);
                const uint32_t heads = __ballot_sync(0xffffffffu, head);
                const int run_head = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
                const int dist = lane - run_head;
                const bool tail = (lane == 31) || ((heads >> (lane + 1)) & 1u);
                const int maxd = __reduce_max_sync(0xffffffffu, dist);
                for (int o = 1; o <= maxd; o <<= 1) {             // segmented inclusive scan (warp-uniform trip count)
#pragma unroll
                    for (int t4 = 0; t4 < 4; ++t4)
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const float a = __shfl_up_sync(0xffffffffu, v[t4][c], o);
                            if (dist >= o) v[t4][c] += a;
                        }
                }
                if (tail && valid && gx.chlast) {                 // C == 4, channel-last gradients: one 16-byte reduction per texel
                    float4* t4 = reinterpret_cast<float4*>(gx.gptr[l * 3 + p]);
                    auto nz = [](const float* q) { return q[0] != 0.0f || q[1] != 0.0f || q[2] != 0.0f || q[3] != 0.0f; };
                    if (nz(v[0])) atomicAdd(t4 + b.o00, make_float4(v[0][0], v[0][1], v[0][2], v[0][3]));
                    if (b.bx1 && nz(v[1])) atomicAdd(t4 + b.o01, make_float4(v[1][0], v[1][1], v[1][2], v[1][3]));
                    if (b.by1 && nz(v[2])) atomicAdd(t4 + b.o10, make_float4(v[2][0], v[2][1], v[2][2], v[2][3]));
                    if (b.bx1 && b.by1 && nz(v[3])) atomicAdd(t4 + b.o11, make_float4(v[3][0], v[3][1], v[3][2], v[3][3]));
                } else if (tail && valid) {
                    float* pl = gx.gptr[l * 3 + p];
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        if (c >= C) break;
                        float* ch = pl + c * hw;
                        if (v[0][c] != 0.0f) atomicAdd(ch + b.o00, v[0][c]);
                        if (b.bx1 && v[1][c] != 0.0f) atomicAdd(ch + b.o01, v[1][c]);
                        if (b.by1 && v[2][c] != 0.0f) atomicAdd(ch + b.o10, v[2][c]);
                        if (b.bx1 && b.by1 && v[3][c] != 0.0f) atomicAdd(ch + b.o11, v[3][c]);
                    }
                }
            }
        }
    }
}

#include "wb_shade_tc_bwd3.cuh"          // three groups / one wide group: the app/nerf decoder shape; the kernel above serves the shapes it refuses

// decoder backward only: dL/d(shaded) -> weight gradients + dL/dfeat planes in the workspace
// grad_table != NULL asks for the table scatter to be fused into the decoder backward; *fused_out reports whether it was (it is for the
// app/nerf shape: F == 2 'cat' hash grid, three-group kernel) -- otherwise the caller runs wb_tc_table_scatter afterwards
int wb_tc_decoder_bwd_ex(const wb_nef_desc* nef, const float* blob, const wb_rays* rays, const float* rec_t, const int32_t* rec_ray,
                         int64_t S, const float* g_shaded, const float* scale, const void* feat_saved, void* workspace,
                         float* grad_dens, float* grad_col, float* grad_table, int* fused_out, cudaStream_t st);
int wb_tc_decoder_bwd(const wb_nef_desc* nef, const float* blob, const wb_rays* rays, const float* rec_t, const int32_t* rec_ray,
                      int64_t S, const float* g_shaded, const float* scale, const void* feat_saved, void* workspace,
                      float* grad_dens, float* grad_col, cudaStream_t st)
{
    return wb_tc_decoder_bwd_ex(nef, blob, rays, rec_t, rec_ray, S, g_shaded, scale, feat_saved, workspace, grad_dens, grad_col, nullptr, nullptr, st);
}
int wb_tc_decoder_bwd_ex(const wb_nef_desc* nef, const float* blob, const wb_rays* rays, const float* rec_t, const int32_t* rec_ray,
                         int64_t S, const float* g_shaded, const float* scale, const void* feat_saved, void* workspace,
                         float* grad_dens, float* grad_col, float* grad_table, int* fused_out, cudaStream_t st)
{
    if (fused_out) *fused_out = 0;
    WbTc m; int rc = wb_tc_make(nef, true, &m); if (rc) return rc;
    WB_CHECK_ARG(scale != nullptr, "precision 1 needs the device loss-scale pointer");
    WB_CHECK_ARG(feat_saved != nullptr && workspace != nullptr, "precision 1 backward needs the saved features and the workspace");
    if (g_tc_skip_embed) g_tc_skip_embed = 0;          // the forward's workspace (same rays) is being reused: the rows are there
    else { rc = tc_launch_ray_embed(m, rays, workspace, st); if (rc) return rc; }
    int planes, width; tc_dfeat_shape(nef, &planes, &width);
    const int64_t R = rays->num_rays;
    __half* dfeat = reinterpret_cast<__half*>(reinterpret_cast<uint8_t*>(workspace) + tc_align256(R * m.Kp[m.nl_d] * 2));
    TcIn in = { rays->origins, rays->dirs, rec_t, rec_ray, S, reinterpret_cast<const uint4*>(workspace), nullptr, reinterpret_cast<const uint4*>(feat_saved),
                g_tc_s_begin, g_tc_s_end };
    const int64_t S_launch = (g_tc_s_end ? g_tc_s_end : S) - g_tc_s_begin;
    TcGrads G = { grad_dens, grad_col, scale, dfeat, planes, width };
    TcB3Plan plan;
    if (tc_b3_plan(m, &plan)) {      // wb_shade_tc_bwd3.cuh: three sub-tile groups per SM (3.69 ms measured against 4.53 ms for the two-group
        WbGrid g; memset(&g, 0, sizeof(g));    // kernel below), or one 128-wide group (hidden_dim = 128)
        // one wide group per SM: the fused scatter has only 8 warps to issue from and measured slower than the stand-alone scatter kernel
        // (16.0 vs 13.7 ms at hidden_dim 128 on the 1024^2 frame), so only the three-group kernel fuses it
        const bool fuse = grad_table != nullptr && nef->grid_kind == 0 && nef->feature_dim == 2 && nef->multiscale == 0 && planes <= 16 &&
                          plan.groups == 3;
        if (fuse) { rc = wb_make_grid(nef, &g); if (rc) return rc; }
        // [one wide group, three groups, three groups + fused scatter]
        using Bwd3Kernel = decltype(&wb_mlp_bwd3_tc_kernel<false, 3>);
        static const Bwd3Kernel kerns3[3] = { wb_mlp_bwd3_tc_kernel<false, 1>, wb_mlp_bwd3_tc_kernel<false, 3>, wb_mlp_bwd3_tc_kernel<true, 3> };
        const int variant = plan.groups == 1 ? 0 : fuse ? 2 : 1;
        const Bwd3Kernel kern3 = kerns3[variant];
        static int64_t done3[3] = { -1, -1, -1 };
        if (done3[variant] != WB_ATTR_KEY(plan.smem_bytes)) {
            WB_CUDA(cudaFuncSetAttribute(kern3, cudaFuncAttributeMaxDynamicSharedMemorySize, plan.smem_bytes));
            done3[variant] = WB_ATTR_KEY(plan.smem_bytes);
        }
        const int64_t nctas3 = ((S_launch + TC_ROWS - 1) / TC_ROWS + plan.groups - 1) / plan.groups;
        int64_t grid3 = (int64_t)wb_num_sms(); if (grid3 > nctas3) grid3 = nctas3;
        kern3<<<(unsigned)grid3, plan.groups * TC_GROUP, plan.smem_bytes, st>>>(m, plan, reinterpret_cast<const uint8_t*>(blob), in,
                                                                          reinterpret_cast<const float4*>(g_shaded), G, g, grad_table);
        WB_LAUNCH_CHECK();
        if (fuse && fused_out) *fused_out = 1;
        return WB_OK;
    }
    WB_CHECK_ARG(m.fits2, "tensor-core path: decoder backward does not fit in shared memory (use precision 0)");
    {
        static int64_t done_for = -1;
        if (done_for != WB_ATTR_KEY(m.smem_bytes)) {
            WB_CUDA(cudaFuncSetAttribute(wb_mlp_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, m.smem_bytes));
            done_for = WB_ATTR_KEY(m.smem_bytes);
        }
    }
    const int64_t nctas = ((S + TC_ROWS - 1) / TC_ROWS + TC_BWD_GROUPS - 1) / TC_BWD_GROUPS;
    int64_t grid = (int64_t)wb_num_sms(); if (grid > nctas) grid = nctas;         // 1 CTA / SM: TMEM holds the weight-grad accumulators
    wb_mlp_bwd_tc_kernel<<<(unsigned)grid, TC_BWD_GROUPS * TC_GROUP, m.smem_bytes, st>>>(m, reinterpret_cast<const uint8_t*>(blob), in,
                                                                           reinterpret_cast<const float4*>(g_shaded), G);
    WB_LAUNCH_CHECK();
    return WB_OK;
}
// table scatter only: dL/dfeat planes (written by wb_tc_decoder_bwd into the same workspace) -> grad_table
int wb_tc_table_scatter(const wb_nef_desc* nef, const wb_rays* rays, const float* rec_t, const int32_t* rec_ray, int64_t S,
                        const float* scale, void* workspace, float* grad_table, cudaStream_t st)
{
    WbGrid g; int rc = wb_make_grid(nef, &g); if (rc) return rc;
    WbGridX gx; rc = wb_make_gridx(nef, true, &gx); if (rc) return rc;
    WbTc m; rc = wb_tc_make(nef, true, &m); if (rc) return rc;
    WB_CHECK_ARG(scale != nullptr && workspace != nullptr && (grad_table != nullptr || gx.kind != 0), "null pointer");
    int planes, width; tc_dfeat_shape(nef, &planes, &width);
    const int64_t R = rays->num_rays;
    const __half* dfeat = reinterpret_cast<const __half*>(reinterpret_cast<const uint8_t*>(workspace) + tc_align256(R * m.Kp[m.nl_d] * 2));
    TcIn in = { rays->origins, rays->dirs, rec_t, rec_ray, S, nullptr, nullptr, nullptr, gx.kind != 0 ? 0 : g_tc_s_begin, gx.kind != 0 ? 0 : g_tc_s_end };
    const int64_t S_launch = gx.kind != 0 ? S : (g_tc_s_end ? g_tc_s_end : S) - g_tc_s_begin;
    if (gx.kind != 0) {
        int64_t bx = (S + 255) / 256; const int64_t cap = (int64_t)wb_num_sms() * 16; if (bx > cap) bx = cap;
        wb_featx_scatter_kernel<<<(unsigned)bx, 256, 0, st>>>(gx, in, dfeat, width, scale);
        WB_LAUNCH_CHECK();
        return WB_OK;
    }
    const int levels = g.multiscale == 0 ? planes : g.L;
    if (levels > 0) {
        // LODs per CTA row: the sample position / record loads are shared by `lpb` LODs (measured sweep in profiles/README.md)
        const int lpb = max(1, min(levels, TC_SCATTER_LPB));
        int64_t bx = (S_launch + 255) / 256; const int64_t cap = (int64_t)wb_num_sms() * TC_SCATTER_CTAS; if (bx > cap) bx = cap;
        dim3 grid2((unsigned)bx, (unsigned)((levels + lpb - 1) / lpb));
        auto kern = g.F == 2 ? wb_table_scatter_kernel<2> : wb_table_scatter_kernel<0>;
        kern<<<grid2, 256, 0, st>>>(g, in, dfeat, planes, levels, lpb, scale, grad_table, g.F == 2);
        WB_LAUNCH_CHECK();
    }
    return WB_OK;
}

// Wide decoders (one 256-thread group per SM, half the register file and all the other warp slots idle): the sample range is cut
// into chunks; the decoder backward of chunk c+1 runs on the caller's stream while the table scatter of chunk c (an issue-bound SIMT
// kernel with 48 registers per thread and no shared memory: two of its CTAs fit beside a decoder CTA) runs on a side stream.
struct TcSide { cudaStream_t stream; cudaEvent_t ev[TC_WIDE_CHUNKS + 1]; bool ok; };
static TcSide* tc_side_stream()
{
    static TcSide side[64];
    int dev = 0; if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    TcSide& s = side[dev];
    if (!s.ok) {
        if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
        for (int i = 0; i <= TC_WIDE_CHUNKS; ++i) if (cudaEventCreateWithFlags(&s.ev[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
        s.ok = true;
    }
    return &s;
}

int wb_tc_shade_bwd(const wb_nef_desc* nef, const float* blob, const wb_rays* rays, const float* rec_t, const int32_t* rec_ray,
                    int64_t S, const float* g_shaded, const float* scale, const void* feat_saved, void* workspace,
                    float* grad_table, float* grad_dens, float* grad_col, cudaStream_t st)
{
    {
        WbTc m; TcB3Plan plan;
        TcSide* side = nullptr;
        if (S >= TC_WIDE_MIN_S && nef->grid_kind == 0 && grad_table && wb_tc_make(nef, true, &m) == WB_OK && !m.fits2 &&
            tc_b3_plan(m, &plan) && plan.groups == 1 && (side = tc_side_stream()) != nullptr) {
            const int64_t per = ((S + TC_WIDE_CHUNKS - 1) / TC_WIDE_CHUNKS + TC_ROWS - 1) / TC_ROWS * TC_ROWS;
            int rc = WB_OK, c = 0;
            for (int64_t s0 = 0; s0 < S && rc == WB_OK; s0 += per, ++c) {
                g_tc_s_begin = s0; g_tc_s_end = s0 + per < S ? s0 + per : S;
                if (c > 0) g_tc_skip_embed = 1;                       // the per-ray rows were written by the first chunk's launch
                rc = wb_tc_decoder_bwd_ex(nef, blob, rays, rec_t, rec_ray, S, g_shaded, scale, feat_saved, workspace, grad_dens, grad_col, nullptr, nullptr, st);
                if (rc == WB_OK && (cudaEventRecord(side->ev[c], st) != cudaSuccess || cudaStreamWaitEvent(side->stream, side->ev[c], 0) != cudaSuccess)) rc = WB_ERR_CUDA;
                if (rc == WB_OK) rc = wb_tc_table_scatter(nef, rays, rec_t, rec_ray, S, scale, workspace, grad_table, side->stream);
            }
            g_tc_s_begin = 0; g_tc_s_end = 0;
            // the caller's stream continues after the last scatter (also on an error path: never leave the side stream unjoined)
            if (cudaEventRecord(side->ev[TC_WIDE_CHUNKS], side->stream) != cudaSuccess || cudaStreamWaitEvent(st, side->ev[TC_WIDE_CHUNKS], 0) != cudaSuccess) { if (rc == WB_OK) rc = WB_ERR_CUDA; }
            return rc;
        }
    }
    int fused = 0;
    int rc = wb_tc_decoder_bwd_ex(nef, blob, rays, rec_t, rec_ray, S, g_shaded, scale, feat_saved, workspace, grad_dens, grad_col, grad_table, &fused, st);
    if (rc || fused) return rc;
    return wb_tc_table_scatter(nef, rays, rec_t, rec_ray, S, scale, workspace, grad_table, st);
}
