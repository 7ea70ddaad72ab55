// wb_shade_tc_bwd3.cuh -- decoder backward with THREE sub-tile groups per SM, included by wb_shade_tc.cu.  Designed from the
// measured round costs (profiles/README.md, backlog item (d)); validated on B200 in round 2 (same gradients as the two-group
// kernel, 4.53 -> 3.69 ms on the 1024^2 frame) and used for every decoder shape tc_b3_plan accepts; the two-group kernel
// (wb_mlp_bwd_tc_kernel) serves the shapes it refuses.
//
// The two-group kernel retains all five activation tiles of a sub-tile (78 KB) + a dY tile (16 KB), so only two sub-tiles fit
// in shared memory and only two latency chains are in flight per SM.  This variant keeps three uniform buffers P, Q, R
// (one 64-wide tile + its constant-one slab each) and a small buffer E per group and pays one extra round:
//
//   tile start : X0 -> P                                    (saved features)
//   r0  F0     : P  -> relu -> X1 -> Q
//   r1  F1     : Q  -> df (registers);  X2 = [df[1:], view] -> R
//   r2  F2     : R  -> relu -> X3 -> P
//   r3  F3     : P  -> relu -> X4 -> Q
//   r4  F4     : Q  -> c3 (registers);  dY4 -> E
//   r5  B4     : wgrad(X4@Q, dY4@E), dgrad -> mask with X4@Q -> dY3 IN PLACE over X4 -> Q
//   r6  B3     : wgrad(X3@P, dY3@Q), dgrad -> mask with X3@P -> dY2 in place -> P
//   r7  B2     : wgrad(X2@R, dY2@P), dgrad -> dY1 (16 wide) -> E;  X0 reloaded -> R
//   r8  F0'    : R  -> relu -> X1 -> Q                       (the extra round)
//   r9  B1     : wgrad(X1@Q, dY1@E), dgrad -> mask with X1@Q -> dY0 in place -> Q
//   r10 B0     : wgrad(X0@R, dY0@Q), dgrad -> dL/dfeat planes (global)
//
// In-place dY: a thread reads the relu-mask elements of its own row chunk before it overwrites that chunk; the UMMAs that read the
// tile have completed (the group waited on them).  Constant-one slabs: P and Q always carry it at slab maxw/8 (never overwritten: the
// tiles living there are maxw wide, X0 in P carries its own at Kp0/8 and is rewritten at every tile start); R carries it at
// Kp2/8 (X2) or Kp0/8 (X0), rewritten whenever the tile is placed.
// Restricted to the app/nerf decoder depth (2 density layers, 3 colour layers), every width <= 64.
#pragma once

constexpr int TC_B3_ROUNDS = 11;

// ---- per-CTA issue table: [group][round][chain]  (chain 0, 1: warp 0 in this order; chain 2: warp 1) ----
template <int NG>
__device__ __forceinline__ void tc_b3_build_table(const WbTc& m, const TcB3Plan& p, TcRec* tab, uint8_t* smem, uint32_t tmem)
{
    constexpr int WC = NG == 3 ? 64 : 128;                        // working-accumulator columns per group
    const int e = threadIdx.x;
    if (e < TC_ROWS) {                                           // Ones[128 x 16] of the bias UMMA
        uint4 one; one.x = 0x00003C00u; one.y = 0; one.z = 0; one.w = 0;
        *reinterpret_cast<uint4*>(smem + p.ones_off + e * 16) = one;
        *reinterpret_cast<uint4*>(smem + p.ones_off + 2048 + e * 16) = make_uint4(0, 0, 0, 0);
    }
    if (e >= NG * TC_B3_ROUNDS * 3) return;
    const int ch = e % 3, rd = (e / 3) % TC_B3_ROUNDS, g = e / (3 * TC_B3_ROUNDS);
    const uint32_t base = tc_smem_u32(smem), gb = base + g * p.GB;
    const uint32_t bP = gb + p.P, bQ = gb + p.Q, bR = gb + p.R, bE = gb + p.E;
    const uint32_t wbase = base + p.blob_off;
    const uint32_t work = tmem + g * WC;                          // D_work[g]: WC columns per group, accumulators behind them
    // round -> (layer, forward?, X buffer, dY buffer)
    const int  lay[TC_B3_ROUNDS] = { 0, 1, 2, 3, 4, 4, 3, 2, 0, 1, 0 };
    const bool fwd[TC_B3_ROUNDS] = { true, true, true, true, true, false, false, false, true, false, false };
    const uint32_t X[TC_B3_ROUNDS] = { bP, bQ, bR, bP, bQ, bQ, bP, bR, bR, bQ, bR };
    const uint32_t Y[TC_B3_ROUNDS] = { 0, 0, 0, 0, 0, bE, bQ, bP, 0, bE, bQ };
    const int l = lay[rd], Np = m.Np[l], Kp = m.Kp[l];
    uint64_t da = 0, db = 0; uint32_t id = 0, d = 0, nk = 0, acc = 0, aadv = 0, badv = 0;
    if (fwd[rd]) {
        if (ch == 0) {            // bias: D_work = Ones . Bias_l^T
            da = tc_desc(base + p.ones_off, 2048, 128); db = tc_desc(wbase + m.b_off[l], Np * 16, 128);
            id = tc_idesc(128, Np, 0, 0); d = work; nk = m.has_bias ? 1 : 0;
        } else if (ch == 1) {     // D_work (+)= X_l . W_l^T
            da = tc_desc(X[rd], 2048, 128); db = tc_desc(wbase + m.w_off[l], Np * 16, 128);
            id = tc_idesc(128, Np, 0, 0); d = work; nk = Kp / 16; acc = m.has_bias; aadv = 4096 >> 4; badv = (2 * Np * 16) >> 4;
        }
    } else {
        if (ch == 0 && p.kind[l] != 2) {   // acc_l[in, out] += X_l^T . dY_l   (K = 128 samples); kind 0: row Kp_l = bias gradient (constant-one slab)
            da = tc_desc(X[rd], 128, 2048); db = tc_desc(Y[rd], 128, 2048);
            id = tc_idesc(128, Np, 1, 1); d = tmem + p.acc_col[l]; nk = 8; acc = 1; aadv = 256 >> 4; badv = 256 >> 4;
        } else if (ch == 0) {              // kind 2: acc_l^T[out, in | 1] += dY_l^T . [X_l | 1]: Kp_l + 16 columns instead of Np_l, column Kp_l = bias gradient
            da = tc_desc(Y[rd], 128, 2048); db = tc_desc(X[rd], 128, 2048);
            id = tc_idesc(128, Kp + 16, 1, 1); d = tmem + p.acc_col[l]; nk = 8; acc = 1; aadv = 256 >> 4; badv = 256 >> 4;
        } else if (ch == 1 && p.kind[l] == 1) {   // kind 1 (X_l is 128 wide: no row left for the bias): bias_l[out, 0] += dY_l^T . Ones, Ones = the tile's constant-one slab
            da = tc_desc(Y[rd], 128, 2048); db = tc_desc(X[rd] + (uint32_t)(Kp / 8) * 2048u, 128, 2048);
            id = tc_idesc(128, 16, 1, 1); d = tmem + p.bias_col[l]; nk = m.has_bias ? 8 : 0; acc = 1; aadv = 256 >> 4; badv = 256 >> 4;
        } else if (ch == 2) {     // D_work = dY_l . W_l             (K = out features)
            da = tc_desc(Y[rd], 2048, 128); db = tc_desc(wbase + m.w_off[l], 128, Np * 16);
            id = tc_idesc(128, Kp, 0, 1); d = work; nk = Np / 16; aadv = 4096 >> 4; badv = 256 >> 4;
        }
    }
    TcRec r = { (uint32_t)da, (uint32_t)(da >> 32), (uint32_t)db, (uint32_t)(db >> 32), id, d, nk | (acc << 8), aadv | (badv << 16) };
    tab[(g * TC_B3_ROUNDS + rd) * 3 + ch] = r;
}

__device__ __forceinline__ void tc_b3_round(TcCtx& c, const TcRec* r3)
{
    uint4 qa0 = make_uint4(0, 0, 0, 0), qa1 = qa0, qb0 = qa0, qb1 = qa0;
    if (c.wig == 0) {
        const uint4* pa = reinterpret_cast<const uint4*>(r3); const uint4* pb = reinterpret_cast<const uint4*>(r3 + 1);
        qa0 = pa[0]; qa1 = pa[1]; qb0 = pb[0]; qb1 = pb[1];
    } else if (c.wig == 1) {
        const uint4* pa = reinterpret_cast<const uint4*>(r3 + 2);
        qa0 = pa[0]; qa1 = pa[1];
    }
    tc_fence_smem_async();
    tc_fence_before();
    tc_group_sync(c.g + 1, TC_GROUP);
    if (c.wig < TC_ISSUERS) {
        if (tc_elect_one()) {
            tc_fence_after();
            if (((qa1.z | qb1.z) & 0xffu) != 0) { tc_issue_rec(qa0, qa1); tc_issue_rec(qb0, qb1); tc_commit(c.bar); }
            else tc_mbar_arrive(c.bar);
        }
        __syncwarp();
    }
    tc_mbar_wait(c.bar, c.phase);
    c.phase ^= 1u;
    tc_fence_after();
}

// relu(D_work[:, 0:Np)) -> fp16 tile `dst` (this thread: its row, its column half)
__device__ __forceinline__ void tc_b3_relu_to_tile(const TcCtx& c, uint32_t trow, int Np, uint8_t* dst)
{
    // 16 columns at a time: this kernel runs 768 threads per SM, i.e. at most 85 registers per thread
    for (int c0 = c.h * 32; c0 < Np; c0 += 64) {
        for (int cc = c0; cc < min(c0 + 32, Np); cc += 16) {
            float v[16]; tc_ld16(trow + cc, v);
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                uint4 o;
                o.x = tc_pack2_relu(v[q * 8], v[q * 8 + 1]); o.y = tc_pack2_relu(v[q * 8 + 2], v[q * 8 + 3]);
                o.z = tc_pack2_relu(v[q * 8 + 4], v[q * 8 + 5]); o.w = tc_pack2_relu(v[q * 8 + 6], v[q * 8 + 7]);
                *reinterpret_cast<uint4*>(dst + ((cc >> 3) + q) * 2048 + c.r * 16) = o;
            }
        }
    }
}
// dY = D_work[:, 0:Kp) masked by relu'(X) written IN PLACE over the activation tile `tile`
__device__ __forceinline__ void tc_b3_mask_in_place(const TcCtx& c, uint32_t trow, int Kp, uint8_t* tile)
{
    for (int c0 = c.h * 32; c0 < Kp; c0 += 64) {
        for (int cc = c0; cc < min(c0 + 32, Kp); cc += 16) {
            float v[16]; tc_ld16(trow + cc, v);
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                uint4* slot = reinterpret_cast<uint4*>(tile + ((cc >> 3) + q) * 2048 + c.r * 16);
                const uint4 a = *slot;
                const __half2 z2 = __float2half2_rn(0.0f);
                uint4 o;
                o.x = tc_pack2(v[q * 8], v[q * 8 + 1]) & __hgt2_mask(*reinterpret_cast<const __half2*>(&a.x), z2);
                o.y = tc_pack2(v[q * 8 + 2], v[q * 8 + 3]) & __hgt2_mask(*reinterpret_cast<const __half2*>(&a.y), z2);
                o.z = tc_pack2(v[q * 8 + 4], v[q * 8 + 5]) & __hgt2_mask(*reinterpret_cast<const __half2*>(&a.z), z2);
                o.w = tc_pack2(v[q * 8 + 6], v[q * 8 + 7]) & __hgt2_mask(*reinterpret_cast<const __half2*>(&a.w), z2);
                *slot = o;
            }
        }
    }
}
__device__ __forceinline__ void tc_b3_one_slab(uint8_t* tile, int slab, int r)
{
    uint4 one; one.x = 0x00003C00u; one.y = 0; one.z = 0; one.w = 0;           // fp16 1.0 in feature 0 of the slab
    *reinterpret_cast<uint4*>(tile + slab * 2048 + r * 16) = one;
}

// One LOD of the hash-table scatter for the 32 consecutive samples of a warp (F == 2): the arithmetic of wb_table_scatter_kernel
// <2> (hashgrid_interpolate_cuda.cu:151-160 + run merging + paired 16-byte reductions), callable from the decoder
// backward's last epilogue so that dL/dfeat never leaves the SM.  s0, s1: this sample's (still loss-scaled) gradient of the LOD's two
// features.  Warp-collective: every lane of the warp calls it with the same `l`.
__device__ __forceinline__ void tc_scatter_level_f2(const WbGrid& g, int l, float px, float py, float pz, bool valid, float s0, float s1,
                                                    float inv_scale, int lane, float* __restrict__ gtable)
{
    float* tb = gtable + g.begin[l] * 2;
    const bool pair_ok = (reinterpret_cast<uintptr_t>(tb) & 15u) == 0;
    uint32_t idx[8]; float cf[8]; uint64_t key = ~0ull - (uint64_t)lane;    // invalid lanes never merge
    if (valid) {
        int ix, iy, iz; float wx, wy, wz, jx, jy, jz;
        wb_cell(px, g.hres[l], g.hi[l], ix, wx, jx); wb_cell(py, g.hres[l], g.hi[l], iy, wy, jy); wb_cell(pz, g.hres[l], g.hi[l], iz, wz, jz);
        key = (uint64_t)ix | ((uint64_t)iy << 20) | ((uint64_t)iz << 40);
        const float xy00 = jx * jy, xy01 = jx * wy, xy10 = wx * jy, xy11 = wx * wy;
        cf[0] = xy00 * jz; cf[1] = xy00 * wz; cf[2] = xy01 * jz; cf[3] = xy01 * wz;
        cf[4] = xy10 * jz; cf[5] = xy10 * wz; cf[6] = xy11 * jz; cf[7] = xy11 * wz;
        wb_corner_indices(g, l, ix, iy, iz, idx);
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) { idx[j] = 0; cf[j] = 0.0f; }
    }
    const uint64_t kprev = __shfl_up_sync(0xffffffffu, key, 1);
    const bool head = (lane == 0) || (kprev != key);
    const uint32_t heads = __ballot_sync(0xffffffffu, head);
    const int run_head = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
    const int dist = lane - run_head;
    const bool tail = (lane == 31) || ((heads >> (lane + 1)) & 1u);
    const int maxd = __reduce_max_sync(0xffffffffu, dist);
    float v0[8], v1[8];
    if (maxd > 0) {     // run sums as loss-scaled fp16 pairs (one shuffle per corner and scan step), unscaled after the scan
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
        const float g0 = s0 * inv_scale, g1 = s1 * inv_scale;
#pragma unroll
        for (int j = 0; j < 8; ++j) { v0[j] = g0 * cf[j]; v1[j] = g1 * cf[j]; }
    }
    if (tail && valid) {
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
}

// FUSE: the hash-table scatter of a sub-tile's dL/dfeat runs in its last epilogue (F == 2 'cat' hash grids, three groups): the planes
//   never exist, 7.12 ms on the 1024^2 frame against 3.70 + 3.72 = 7.46 ms for this kernel writing fp16 planes and wb_table_scatter_kernel
//   as a second launch.  The win is only the planes' 124 B/sample of traffic and one launch -- the three groups of a CTA run in lockstep
//   (they convoy on the tensor pipe), so all 24 warps scatter at the same time and the scatter phase is as issue / reduction-bound as the
//   stand-alone kernel was.  Two other placements were measured slower and removed (profiles/README.md): the scatter as a critical section
//   of the CTA, which forces the groups' reduction phases apart (7.60 ms), and LOD q of sub-tile i scattered inside round q of sub-tile
//   i+1 (7.34 ms; a round's wait is barrier / commit / wake-up latency, not UMMA execution time, so there is little to hide behind).
template <bool FUSE, int NG = TC_B3_GROUPS>    // NG: sub-tile groups per CTA: 3 (every width <= 64) or 1 (widths up to 128: hidden_dim = 128)
__global__ void __launch_bounds__(NG * TC_GROUP, 1)
wb_mlp_bwd3_tc_kernel(WbTc m, TcB3Plan p, const uint8_t* __restrict__ blob, TcIn in, const float4* __restrict__ g_shaded, TcGrads G, WbGrid g, float* __restrict__ gtable)
{
    constexpr int WC = NG == 3 ? 64 : 128;
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t bars[NG + 1];
    __shared__ uint32_t tmem_s;
    __shared__ TcRec tab[NG * TC_B3_ROUNDS * 3];
    if (threadIdx.x == 0) {
        for (int i = 0; i < NG; ++i) tc_mbar_init(&bars[i], TC_ISSUERS);
        tc_mbar_init(&bars[NG], 1); tc_mbar_init_fence();
        tc_mbar_expect_tx(&bars[NG], (uint32_t)m.blob_bytes);
        tc_bulk_g2s(smem + p.blob_off, blob, (uint32_t)m.blob_bytes, &bars[NG]);
    }
    if (threadIdx.x < 32) tc_tmem_alloc(&tmem_s, 512u);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    tc_b3_build_table<NG>(m, p, tab, smem, tmem_s);
    TcCtx c; tc_ctx_init(c, smem, bars, nullptr, tmem_s, 1);
    uint8_t* gbase = smem + c.g * p.GB;
    uint8_t* bP = gbase + p.P; uint8_t* bQ = gbase + p.Q; uint8_t* bR = gbase + p.R; uint8_t* bE = gbase + p.E;
    const TcRec* rec = tab + c.g * TC_B3_ROUNDS * 3;
    const int maxslab = (p.Q - p.P) / 2048 - 1;                  // slab of the constant-one column of a maxw-wide tile
    if (c.h == 0) { tc_b3_one_slab(bP, maxslab, c.r); tc_b3_one_slab(bQ, maxslab, c.r); }
    if (threadIdx.x < 128) {                                     // zero the resident weight-grad accumulators
        const uint32_t tr = c.tmem + ((uint32_t)c.laneq << 16);
        for (int cc = p.acc_begin; cc < p.acc_end; cc += 16) tc_st16_zero(tr + cc);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    tc_mbar_wait(&bars[NG], 0);
    const float scale = __ldg(G.scale), inv_scale = 1.0f / scale;
    const int nch0 = m.Kp[0] / 8, nchc = m.Kp[2] / 8;
    const int64_t s_end = in.s_end ? in.s_end : in.S;             // this launch's sample range (in.S stays the stride of the saved rows / planes)
    const int64_t tile0 = in.s_begin / TC_ROWS, ntiles = (s_end + TC_ROWS - 1) / TC_ROWS;
    const uint32_t trow = c.tmem + ((uint32_t)c.laneq << 16) + (uint32_t)(c.g * WC);
    const float z8[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
    const int lane_ = threadIdx.x & 31;
    for (int64_t tile = tile0 + (int64_t)blockIdx.x * NG + c.g; tile < ntiles; tile += (int64_t)gridDim.x * NG) {
        int64_t s = tile * TC_ROWS + c.r;
        const bool valid = s < s_end;
        if (!valid) s = s_end - 1;
        const int64_t ray = __ldg(in.rec_ray + s);
        // X0 -> P
        for (int ch = c.h; ch < nch0; ch += 2)
            *reinterpret_cast<uint4*>(bP + ch * 2048 + c.r * 16) = __ldg(in.x0_saved + (int64_t)ch * in.S + s);
        if (c.h == 0) tc_b3_one_slab(bP, nch0, c.r);
        // r0: F0 -> X1 -> Q
        tc_b3_round(c, rec + 0 * 3);
        tc_b3_relu_to_tile(c, trow, m.Np[0], bQ);
        // r1: F1 -> df; X2 -> R
        tc_b3_round(c, rec + 1 * 3);
        float df0;
        {
            float df[16];
            tc_ld16(trow, df);
            df0 = df[0];
            const int nd = m.O[1] - 1;
            const uint4* re = in.ray_embed + ray * nchc;
            uint4 q = __ldg(re + c.h);
            __half* hq = reinterpret_cast<__half*>(&q);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float dv = c.h == 0 ? df[(j + 1) & 15] : df[(j + 9) & 15];
                if (8 * c.h + j < nd) hq[j] = __float2half_rn(dv);
            }
            *reinterpret_cast<uint4*>(bR + c.h * 2048 + c.r * 16) = q;
            for (int ch = 2 + c.h; ch < nchc; ch += 2) *reinterpret_cast<uint4*>(bR + ch * 2048 + c.r * 16) = __ldg(re + ch);
            if (c.h == 0) tc_b3_one_slab(bR, nchc, c.r);
        }
        // r2: F2 -> X3 -> P ; r3: F3 -> X4 -> Q
        tc_b3_round(c, rec + 2 * 3);
        tc_b3_relu_to_tile(c, trow, m.Np[2], bP);
        tc_b3_round(c, rec + 3 * 3);
        tc_b3_relu_to_tile(c, trow, m.Np[3], bQ);
        // r4: F4 -> c3 ; dY4 -> E
        tc_b3_round(c, rec + 4 * 3);
        const float4 go = valid ? __ldg(g_shaded + s) : make_float4(0, 0, 0, 0);
        {
            float v[16]; tc_ld16(trow, v);
            if (c.h == 0) {
                const float r = 1.0f / (1.0f + expf(-v[0])), gg = 1.0f / (1.0f + expf(-v[1])), b = 1.0f / (1.0f + expf(-v[2]));
                float dy[8] = { go.x * r * (1.0f - r) * scale, go.y * gg * (1.0f - gg) * scale, go.z * b * (1.0f - b) * scale, 0, 0, 0, 0, 0 };
                tile_store8(bE, c.r, 0, dy);
            }
            for (int sl = 1 + c.h; sl < m.Np[4] / 8; sl += 2) tile_store8(bE, c.r, sl, z8);
        }
        // r5: B4 -> dY3 in place over X4 (Q) ; r6: B3 -> dY2 in place over X3 (P)
        tc_b3_round(c, rec + 5 * 3);
        tc_b3_mask_in_place(c, trow, m.Kp[4], bQ);
        tc_b3_round(c, rec + 6 * 3);
        tc_b3_mask_in_place(c, trow, m.Kp[3], bP);
        // r7: B2 -> dY1 -> E ; X0 -> R
        tc_b3_round(c, rec + 7 * 3);
        {
            float v[16]; tc_ld16(trow, v);
            const int dout = m.O[1];
            float gdf[16];
            gdf[0] = (df0 > 0.0f) ? go.w * scale : 0.0f;         // relu' of density (nerf.py:263)
#pragma unroll
            for (int j = 1; j < 16; ++j) gdf[j] = (j < dout) ? v[j - 1] : 0.0f;
            if (c.h == 0) tile_store8(bE, c.r, 0, gdf); else tile_store8(bE, c.r, 1, gdf + 8);
            for (int sl = 2 + c.h; sl < m.Np[1] / 8; sl += 2) tile_store8(bE, c.r, sl, z8);
            for (int ch = c.h; ch < nch0; ch += 2)
                *reinterpret_cast<uint4*>(bR + ch * 2048 + c.r * 16) = __ldg(in.x0_saved + (int64_t)ch * in.S + s);
            if (c.h == 0) tc_b3_one_slab(bR, nch0, c.r);
        }
        // r8: F0' -> X1 -> Q
        tc_b3_round(c, rec + 8 * 3);
        tc_b3_relu_to_tile(c, trow, m.Np[0], bQ);
        // r9: B1 -> dY0 in place over X1 (Q)
        tc_b3_round(c, rec + 9 * 3);
        tc_b3_mask_in_place(c, trow, m.Kp[1], bQ);
        // r10: B0 -> dL/dfeat: scattered into the hash table right here (FUSE) or written as fp16 planes for wb_table_scatter_kernel
        float px = 0.0f, py = 0.0f, pz = 0.0f;
        if (FUSE) {                                               // sample position (octree_as.py:283); the loads overlap the round
            const float t = __ldg(in.rec_t + s);
            px = wb_addcmul(__ldg(in.origins + 3 * ray), __ldg(in.dirs + 3 * ray), t);
            py = wb_addcmul(__ldg(in.origins + 3 * ray + 1), __ldg(in.dirs + 3 * ray + 1), t);
            pz = wb_addcmul(__ldg(in.origins + 3 * ray + 2), __ldg(in.dirs + 3 * ray + 2), t);
        }
        tc_b3_round(c, rec + 10 * 3);
        if (FUSE) {
            // column half h holds features [16h, 16h+16) = LODs 8h .. 8h+7; a warp = 32 consecutive samples of one half
            float v[16]; tc_ld16(trow + c.h * 16, v);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int l = c.h * 8 + q;
                if (l < G.planes) tc_scatter_level_f2(g, l, px, py, pz, valid, v[2 * q], v[2 * q + 1], inv_scale, lane_, gtable);
            }
        } else {
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
        }
    }
    // ---- flush weight / bias gradient accumulators ----
    // kind 0: TMEM rows = input feature, row Kp = bias;  kind 1: the same rows, bias in column 0 of its own 16-column accumulator (row = output);
    // kind 2: TMEM rows = output feature, columns = input features, column Kp = bias
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (threadIdx.x < 128) {
        const int row = threadIdx.x;
        const uint32_t tr = c.tmem + ((uint32_t)c.laneq << 16);
        for (int l = 0; l < 5; ++l) {
            float* gbase2 = l < m.nl_d ? G.gdens : G.gcol;
            const int I = m.I[l], O = m.O[l];
            const int wrow0 = row & ~31;
            if (p.kind[l] == 2) {
                if (wrow0 >= m.Np[l]) continue;
                for (int cc = 0; cc < m.Kp[l] + 16; cc += 16) {
                    float v[16]; tc_ld16(tr + p.acc_col[l] + cc, v);
                    if (row >= O) continue;
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const int i = cc + j;
                        const float val = v[j] * inv_scale;
                        if (i < I) { if (val != 0.0f) atomicAdd(gbase2 + m.src_w[l] + row * I + i, val); }
                        else if (i == m.Kp[l] && m.src_b[l] >= 0) atomicAdd(gbase2 + m.src_b[l] + row, val);
                    }
                }
                continue;
            }
            if (p.kind[l] == 1 && m.src_b[l] >= 0 && wrow0 < m.Np[l]) {
                float v[16]; tc_ld16(tr + p.bias_col[l], v);
                if (row < O) atomicAdd(gbase2 + m.src_b[l] + row, v[0] * inv_scale);
            }
            if (wrow0 > m.Kp[l]) continue;
            for (int cc = 0; cc < m.Np[l]; cc += 16) {
                float v[16]; tc_ld16(tr + p.acc_col[l] + cc, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int o = cc + j;
                    if (o >= O) continue;
                    const float val = v[j] * inv_scale;
                    if (row < I) { if (val != 0.0f) atomicAdd(gbase2 + m.src_w[l] + o * I + row, val); }
                    else if (p.kind[l] == 0 && row == m.Kp[l] && m.src_b[l] >= 0) atomicAdd(gbase2 + m.src_b[l] + o, val);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tc_tmem_dealloc(c.tmem, 512u);
}
