// K2 (tensor-core, full precision) -- fused SV edge convolution of the fp SV-DGCNN models (cfg3) with the dense part of
// linear1 on tcgen05.  Same layer as edge_fast.cu's edge_fp_fast_kernel (include/svnet_b200.h: svnet_svblock_edge_fwd;
// reference models/utils/sv_util.py:90-132 + models/sv_layers.py:29-31,111-129,172-196), re-planned like edge_tc.cu:
//
//   y[e][o] = Wa (s_j - s_i) + Wb s_i + Wq q_e            q_e[3 ds + m] = sum_x v_e[x][ds] z_e[x][m],  v_e = [v_j - v_i | v_i]
//
//   * the q part (K = 6 Cv = 60 / 126) is the per-edge work: 655 k edges x 126 x 128 MACs at conv4 were 10 k FMA
//     warp-instructions per point on the CUDA cores.  Here every lane computes the three q values of its (edge, vector
//     channel) in fp32 and splits each EXACTLY into three bf16 planes hi + mid + lo (8 + 8 + 8 mantissa bits) that go
//     straight into the UMMA B operand (K-major canonical layout, no swizzle); Wq is split the same way at pack time (A
//     operand, resident in shared memory); six plane products (h*l, l*h, m*m, h*m, m*h, h*h: everything down to
//     2^-16 |a||w|... of each product, i.e. fp32-grade) accumulate in fp32 in tensor memory: D[128 channels][160 edges];
//   * the s part never enters the tile: Ya = Wa s and Yb = Wb s are one per-point table (svnet_linear_rows, as for the
//     CUDA-core kernel); the epilogue (lane = output channel) adds Ya_j per edge with one coalesced load, takes
//     max / min over the k columns of a point and applies (+ Yb_i - Ya_i) -> BN -> LeakyReLU once per (point, channel);
//   * frames, q channels and the vector branch read the ONE per-point float4 table [P | Q | T | U | v] of edge_tc.cu
//     (one tcgen05 vector linear over the layer input, full-precision weights: three weight planes);
//   * K positions: [diff half: 3 ds + m, ds < Cv | pad to KH][centre half: 3 (ds - Cv) + m | pad], KH = 3 Cv rounded up to 16.
//     conv2 / conv3 (KH = 32): one phase of 64 positions.  conv4 (KH = 64): two phases through ONE 64-position operand
//     buffer (the weights, 96 KB, and a 128-position tile, 125 KB, do not fit together): diff half -> MMAs -> [vector
//     branch while they run] -> centre half (no gathers: v_i only) -> MMAs -> epilogue.
//
// One persistent CTA per SM, 16 warps x 10 edges = 160 edge rows per tile (8 points at k = 20); numerics: fp32-grade,
// tolerance-level like every fp linear of this package (the reference's sgemm order is not reproducible either).
#include "common.cuh"
#include "edge_vector.cuh"
#include "edge_tc_common.cuh"
#include <stdlib.h>

namespace {

constexpr int FTMEM_COLS = 256;

// Tile shapes.  Cout <= 64 (conv2 / conv3): 8 warps x 20 edges, two CTAs per SM (as edge_tc.cu) -- the weight planes keep
// only 64 rows per k-block (the UMMA still multiplies 128 rows: rows 64..127 alias the next k-block, their accumulator lanes
// are never read), which is what lets two tiles fit one SM's shared memory.  Cout = 128 (conv4): the planes alone are
// 96 KB, one CTA per SM with 16 warps x 10 edges.
template <int CS, int CV, int COUT, int CVO, int KE>
struct FTC {
    static constexpr bool SMALL = COUT <= 64;
    static constexpr int EPW = SMALL ? 20 : 10;     // edges per warp
    static constexpr int NWARP = SMALL ? 8 : 16, BT = 10;
    static constexpr int CTAS_PER_SM = SMALL ? 2 : 1;
    static constexpr int AROWS = SMALL ? 64 : 128;  // weight rows kept per k-block
    static constexpr int ROWS = NWARP * EPW, ROWS_PAD = ROWS + 3;
    static constexpr int WPP = KE / EPW;            // warps per point
    static constexpr int NP = NWARP / WPP;          // points per tile
    static constexpr int KH = (3 * CV + 15) / 16 * 16;
    static constexpr int KTOT = 2 * KH;
    static constexpr int NPH = KTOT <= 64 ? 1 : 2;  // phases through the operand buffer
    static constexpr int KPH = KTOT / NPH;          // K positions per phase
    static constexpr int KBA = AROWS * 16;          // bytes per 8-position k-block of a weight plane
    static constexpr int KBB = ROWS_PAD * 16;       // ... of an activation plane
    static constexpr int APL = (KTOT / 8) * KBA;    // bytes per weight plane
    static constexpr int BPL = (KPH / 8) * KBB;     // bytes per activation plane
    static constexpr int A_BYTES = 3 * APL, B_BYTES = 3 * BPL;
    static constexpr int WARP_FLOATS = EPW * 12;    // frames [e][m][4]
    static constexpr int NC = 2 * CVO + 6 + CV;     // float4 columns of the per-point table: P | Q | T | U | v
    static constexpr int TQ0 = CVO, TT0 = 2 * CVO, TU0 = 2 * CVO + 3, TV0 = 2 * CVO + 6;
    static constexpr int VPART = (WPP > 1) ? NWARP * 3 * CVO : 0;
    static constexpr size_t SMEM = (size_t)A_BYTES + B_BYTES + sizeof(float) * (NWARP * WARP_FLOATS + VPART) + 16;
    static_assert(KE % EPW == 0 && NWARP % WPP == 0 && NP * KE == ROWS && ROWS <= FTMEM_COLS && ROWS % 16 == 0, "tile shape");
    static_assert(COUT % 32 == 0 && COUT <= AROWS && NP % (NWARP / 4) == 0 && KPH % 16 == 0 && EPW % 10 == 0, "shape");
    static_assert(CTAS_PER_SM * (SMEM + 1024) <= 227 * 1024, "shared memory");
};

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// K position of q channel (ds, m); KH = positions per half
__host__ __device__ inline int ftc_pos(int ds, int m, int CV, int KH) { return (ds < CV ? 0 : KH) + 3 * (ds < CV ? ds : ds - CV) + m; }

// exact three-way bf16 split of an fp32 value: hi | mid | lo as 16-bit patterns
__device__ __forceinline__ void split3(float a, uint32_t& h, uint32_t& m, uint32_t& l)
{
    const uint32_t hb = __float_as_uint(a) & 0xFFFF0000u;
    const float r1 = a - __uint_as_float(hb);
    const uint32_t mb = __float_as_uint(r1) & 0xFFFF0000u;
    const float r2 = r1 - __uint_as_float(mb);
    h = hb >> 16; m = mb >> 16; l = __float_as_uint(r2) >> 16;
}

// ---- weights: fp32 W1 [COUT][2Cs + 6Cv] (the q columns start at 2Cs) -> three bf16 planes in the canonical K-major
// operand layout [plane][k-block][128 rows][8], K positions by ftc_pos, zero rows / positions for padding
__global__ void edge_fp_tc_pack_w_kernel(const float* __restrict__ W1, int ldw, int CS, int CV, int COUT, int KH, int AROWS,
                                         unsigned char* __restrict__ out)
{
    const int KTOT = 2 * KH, NKB = KTOT / 8;
    const int APL = NKB * AROWS * 16;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < NKB * AROWS; i += gridDim.x * blockDim.x) {
        const int row = i % AROWS, kb = i / AROWS;
        uint32_t w[3][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}};
        for (int e = 0; e < 8; ++e) {
            const int pos = kb * 8 + e;
            const int half = pos >= KH ? 1 : 0, pp = pos - half * KH;
            float v = 0.0f;
            if (row < COUT && pp < 3 * CV) {
                const int ds = half * CV + pp / 3, m = pp % 3;
                v = __ldg(W1 + (long)row * ldw + 2 * CS + 3 * ds + m);
            }
            uint32_t h, md, l;
            split3(v, h, md, l);
            w[0][e >> 1] |= h << (16 * (e & 1));
            w[1][e >> 1] |= md << (16 * (e & 1));
            w[2][e >> 1] |= l << (16 * (e & 1));
        }
        for (int pl = 0; pl < 3; ++pl)
            *reinterpret_cast<uint4*>(out + (size_t)pl * APL + (size_t)kb * AROWS * 16 + (size_t)row * 16) =
                make_uint4(w[pl][0], w[pl][1], w[pl][2], w[pl][3]);
    }
}

// ---- one q section: vector channels ds in [DS0, DS0 + NDS) (inside one half) of every edge of the warp; GE = 32 / NDS
// edges per pass; PH0 = first K position of the phase the section is written in
template <typename S, int CV, int DS0, int NDS, int PH0>
struct QSecF {
    static constexpr int GE = 32 / NDS;
    static constexpr int PASSES = (S::EPW + GE - 1) / GE;
    static constexpr bool DIFF = DS0 < CV;
    static constexpr int PB = DIFF ? (PASSES < S::BT ? PASSES : S::BT) : 1;
    int esub, dcol;
    bool lane_on;
    float4 vi;
    uint32_t bst[3];           // shared addresses of this lane's three values in operand row 0 of the warp, plane 0
    const float4* vcol;

    __device__ __forceinline__ void init(int lane, uint32_t brow0)
    {
        esub = lane / NDS;
        const int ds = DS0 + lane % NDS;
        lane_on = lane < GE * NDS && ds < (DIFF ? CV : 2 * CV);
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            const int pos = ftc_pos(lane_on ? ds : DS0, m, CV, S::KH) - PH0;
            bst[m] = brow0 + (uint32_t)((pos >> 3) * S::KBB + (pos & 7) * 2);
        }
        dcol = S::TV0 + (lane_on ? (DIFF ? ds : ds - CV) : 0);
    }
    __device__ __forceinline__ void centre(const float4* tabc, const float4* trow)
    {
        vcol = tabc + dcol;
        vi = __ldg(trow + dcol);
    }
    __device__ __forceinline__ void run(int my_j, uint32_t zb) const
    {
#pragma unroll 1
        for (int p0 = 0; p0 < PASSES; p0 += PB) {
            float4 nb[PB];
            if (DIFF) {
#pragma unroll
                for (int i = 0; i < PB; ++i) {
                    const int e = (p0 + i) * GE + esub;
                    const unsigned j = (unsigned)__shfl_sync(SV_FULL, my_j, (lane_on && e < S::EPW) ? e : 0);
                    nb[i] = __ldg(vcol + (size_t)j * S::NC);
                }
            }
#pragma unroll
            for (int i = 0; i < PB; ++i) {
                const int e = (p0 + i) * GE + esub;
                const bool on = lane_on && e < S::EPW;
                const int es = on ? e : 0;
                float ve[3];
                if (DIFF) {
                    ve[0] = __fsub_rn(nb[i].x, vi.x); ve[1] = __fsub_rn(nb[i].y, vi.y); ve[2] = __fsub_rn(nb[i].z, vi.z);
                } else {
                    ve[0] = vi.x; ve[1] = vi.y; ve[2] = vi.z;
                }
#pragma unroll
                for (int m = 0; m < 3; ++m) {
                    const float4 z = lds128(zb + (uint32_t)(es * 48 + m * 16));        // frame column m
                    float q = __fmul_rn(ve[0], z.x);
                    q = __fmaf_rn(ve[1], z.y, q);
                    q = __fmaf_rn(ve[2], z.z, q);
                    uint32_t h, md, l;
                    split3(q, h, md, l);
                    if (on) {
                        const uint32_t a = bst[m] + (uint32_t)(es * 16);
                        sts16(a, h);
                        sts16(a + S::BPL, md);
                        sts16(a + 2 * S::BPL, l);
                    }
                }
            }
        }
    }
};

template <int CS, int CV, int COUT, int CVO, int KE>
__global__ void __launch_bounds__(FTC<CS, CV, COUT, CVO, KE>::NWARP * 32, FTC<CS, CV, COUT, CVO, KE>::CTAS_PER_SM)
edge_fp_tc_kernel(svnet_edge_params p, const unsigned char* __restrict__ W1tc, const float4* __restrict__ tab4, int ntiles)
{
    using S = FTC<CS, CV, COUT, CVO, KE>;
    constexpr int NWARP = S::NWARP, ROWS = S::ROWS;
    extern __shared__ __align__(1024) unsigned char smraw[];
    unsigned char* As = smraw;
    unsigned char* Bs = As + S::A_BYTES;
    float* wsm = reinterpret_cast<float*>(Bs + S::B_BYTES);
    float* vpart = wsm + NWARP * S::WARP_FLOATS;
    uint64_t* bar = reinterpret_cast<uint64_t*>(vpart + S::VPART);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);

    const int tid = threadIdx.x, lane = tid & 31, warp = sv_warp_id();
    const long total = (long)p.B * p.N;

    // ---- one-time setup: weight planes resident, operand buffer zeroed (pads stay zero), barrier, tensor memory ----
    for (int i = tid; i < S::A_BYTES / 16; i += NWARP * 32)
        reinterpret_cast<uint4*>(As)[i] = __ldg(reinterpret_cast<const uint4*>(W1tc) + i);
    for (int i = tid; i < S::B_BYTES / 16; i += NWARP * 32) reinterpret_cast<uint4*>(Bs)[i] = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(FTMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    // ---- per-lane constants ----
    const uint32_t zb = smem_u32(wsm + warp * S::WARP_FLOATS);     // frames [EPW][3 m][4]
    const int pt_in_tile = warp / S::WPP, e0 = (warp % S::WPP) * S::EPW;
    const uint32_t brow0 = smem_u32(Bs) + (uint32_t)(warp * S::EPW) * 16u;     // first operand row of this warp
    // q sections: the diff half and the centre half; halves wider than 32 channels never occur (Cv <= 24)
    static_assert(CV <= 32, "two sections per half");
    // a half wider than 16 channels is walked as 16 + rest channels (32 / 30 of 32 lanes busy instead of Cv of 32)
    constexpr int NA = CV > 16 ? 16 : CV, NB2 = CV - NA;
    constexpr int PHC = S::NPH == 1 ? 0 : S::KH;
    QSecF<S, CV, 0, NA, 0> qd;
    QSecF<S, CV, NA, (NB2 > 0 ? NB2 : 1), 0> qd2;
    QSecF<S, CV, CV, NA, PHC> qc;
    QSecF<S, CV, CV + NA, (NB2 > 0 ? NB2 : 1), PHC> qc2;
    qd.init(lane, brow0);
    qc.init(lane, brow0);
    if (NB2 > 0) { qd2.init(lane, brow0); qc2.init(lane, brow0); }
    // epilogue role: TMEM lane quarter = output channels, column group = points
    const int q4 = warp & 3, grp = warp >> 2;
    const int oc = q4 * 32 + lane;
    const bool epi_on = q4 * 32 < COUT;
    float a1 = 0.0f, c1 = 0.0f;
    if (epi_on) { a1 = __ldg(p.bn1_a + oc); c1 = __ldg(p.bn1_c + oc); }
    const int m_lane = lane % 3, e_lane = lane / 3;                // frame tasks: 10 edges x 3 columns

    VBranch<S, CVO> vb;
    vb.init(p, lane);
    int next_j = 0;
    {
        const long r = (long)blockIdx.x * S::NP + pt_in_tile;
        if (blockIdx.x < ntiles && r < total && lane < S::EPW) next_j = __ldg(p.idx + r * KE + e0 + lane);
    }
    // D fp32, A / B bf16, both K-major, N = 160 edge rows, M = 128 channels
    constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(ROWS >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    // plane products, small terms first: (weight plane, activation plane) = h*l, l*h, m*m, h*m, m*h, h*h
    uint32_t phase = 0;
    auto issue_mmas = [&](int ph) {
        if (warp == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            if (lane == 0) {
                const uint32_t a0 = smem_u32(As) + (uint32_t)(ph * (S::KPH / 8) * S::KBA), b0 = smem_u32(Bs);
                constexpr int WPL[6] = {0, 2, 1, 0, 1, 0}, APLN[6] = {2, 0, 1, 1, 0, 0};
                bool first = ph == 0;
#pragma unroll
                for (int pr = 0; pr < 6; ++pr) {
#pragma unroll
                    for (int ks = 0; ks < S::KPH / 16; ++ks) {
                        const uint64_t adesc = make_desc(a0 + (uint32_t)(WPL[pr] * S::APL + 2 * ks * S::KBA), S::KBA, 128);
                        const uint64_t bdesc = make_desc(b0 + (uint32_t)(APLN[pr] * S::BPL + 2 * ks * S::KBB), S::KBB, 128);
                        umma_bf16(tmem_base, adesc, bdesc, idesc, first ? 0u : 1u);
                        first = false;
                    }
                }
                umma_commit(bar);
            }
            __syncwarp();
        }
    };
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long r = (long)tile * S::NP + pt_in_tile;
        const bool valid = r < total;
        const int my_j = next_j;
        {
            const long rn = r + (long)gridDim.x * S::NP;
            next_j = (tile + gridDim.x < ntiles && rn < total && lane < S::EPW) ? __ldg(p.idx + rn * KE + e0 + lane) : 0;
        }
        int b = 0;
        const float4* tabc = tab4;
        const float4* trow = tab4;
        if (valid) {
            b = (int)(r / p.N);
            const long cbase = (long)b * p.N;
            tabc = tab4 + cbase * S::NC;
            trow = tab4 + r * S::NC;
            // ---- frames z_e[x][m] = T_j + (U_i - T_i), stored [e][m][x (4)] ----
            const float4 ti = __ldg(trow + S::TT0 + m_lane), ui = __ldg(trow + S::TU0 + m_lane);
            float4 tj[S::EPW / 10];
#pragma unroll
            for (int rd = 0; rd < S::EPW / 10; ++rd) {
                const int e = rd * 10 + e_lane;
                const unsigned jf = (unsigned)__shfl_sync(SV_FULL, my_j, e < S::EPW ? e : 0);
                tj[rd] = __ldg(tabc + (size_t)jf * S::NC + S::TT0 + m_lane);
            }
            qd.centre(tabc, trow);
            qc.centre(tabc, trow);
            if (NB2 > 0) { qd2.centre(tabc, trow); qc2.centre(tabc, trow); }
            if (lane < 30) {
#pragma unroll
                for (int rd = 0; rd < S::EPW / 10; ++rd)
                    sts128(zb + (uint32_t)((rd * 10 + e_lane) * 48 + m_lane * 16),
                           make_float4(tj[rd].x + (ui.x - ti.x), tj[rd].y + (ui.y - ti.y), tj[rd].z + (ui.z - ti.z), 0.0f));
            }
            __syncwarp();
            // ---- q sections of the first phase ----
            qd.run(my_j, zb);
            if (NB2 > 0) qd2.run(my_j, zb);
            if (S::NPH == 1) { qc.run(my_j, zb); if (NB2 > 0) qc2.run(my_j, zb); }
        }
        // first vector-branch gathers go out before the barrier
        if (valid) vb.prefetch(p, b, tabc, trow, my_j, lane);
        // ---- operand complete: generic-proxy writes -> tensor-core reads ----
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
        __syncthreads();
        issue_mmas(0);
        // ---- vector branch while the tensor core works ----
        if (valid) vb.run(p, r, b, tabc, trow, my_j, KE, lane, S::WPP == 1 ? nullptr : vpart + warp * 3 * CVO);
        if (S::WPP > 1) {
            __syncthreads();
            if (valid && e0 == 0) vector_branch_combine<CVO, S::WPP>(p, r, b, vpart + warp * 3 * CVO, 3 * CVO, KE, lane);
        }
        if (S::NPH == 2) {
            // ---- second phase: the centre half through the same operand buffer, once the first MMAs have read it ----
            mbar_wait(bar, phase);
            phase ^= 1u;
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            if (valid) { qc.run(my_j, zb); if (NB2 > 0) qc2.run(my_j, zb); }
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
            __syncthreads();
            issue_mmas(1);
        }
        // ---- epilogue: + Ya_j per edge, max / min over the k columns of each point, one float chain per (point, channel) ----
        mbar_wait(bar, phase);
        phase ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        if (epi_on) {
            constexpr int PPW = S::NP / (NWARP / 4);                // points per epilogue warp
#pragma unroll 1
            for (int pp = 0; pp < PPW; ++pp) {
                const int pt = grp * PPW + pp;
                const long rr = (long)tile * S::NP + pt;
                if (rr >= total) continue;                           // warp-uniform
                const long cb2 = (rr / p.N) * (long)p.N;
                const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(pt * KE);
                const float* yrow = p.Yab + rr * 2 * COUT;
                const float ci = __ldg(yrow + COUT + oc) - __ldg(yrow + oc);      // Yb_i - Ya_i
                const float* ya0 = p.Yab + cb2 * 2 * COUT + oc;
                float dmax = -INFINITY, dmin = INFINITY;
#pragma unroll
                for (int c0 = 0; c0 < KE; c0 += 20) {
                    const int jj = (lane < 20) ? __ldg(p.idx + rr * KE + c0 + lane) : 0;
                    float ya[20];
#pragma unroll
                    for (int i = 0; i < 20; ++i) {
                        const unsigned j = (unsigned)__shfl_sync(SV_FULL, jj, i);
                        ya[i] = __ldg(ya0 + (size_t)j * (2 * COUT));
                    }
                    uint32_t v16[16], v4[4];
                    tmem_ld16(taddr + c0, v16);
                    tmem_ld4(taddr + c0 + 16, v4);
                    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const float t = __uint_as_float(v16[i]) + ya[i];
                        dmax = fmaxf(dmax, t);
                        dmin = fminf(dmin, t);
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float t = __uint_as_float(v4[i]) + ya[16 + i];
                        dmax = fmaxf(dmax, t);
                        dmin = fminf(dmin, t);
                    }
                }
                float y0 = __fadd_rn(__fmul_rn(dmax + ci, a1), c1);
                float y1 = __fadd_rn(__fmul_rn(dmin + ci, a1), c1);
                y0 = y0 > 0.0f ? y0 : __fmul_rn(0.2f, y0);
                y1 = y1 > 0.0f ? y1 : __fmul_rn(0.2f, y1);
                p.out.s[rr * p.out.lds + oc] = fmaxf(y0, y1);
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    }
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(FTMEM_COLS));
}

int ftc_sm_count()
{
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

template <int CS, int CV, int COUT, int CVO, int KE>
int launch_ftc(const svnet_edge_params* p, cudaStream_t st)
{
    using S = FTC<CS, CV, COUT, CVO, KE>;
    const long total = (long)p->B * p->N;
    const int ntiles = sv_cdiv(total, S::NP);
    const int slots = S::CTAS_PER_SM * ftc_sm_count();
    const int grid = ntiles < slots ? ntiles : slots;
    SV_CUDA(cudaFuncSetAttribute(edge_fp_tc_kernel<CS, CV, COUT, CVO, KE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::SMEM));
    edge_fp_tc_kernel<CS, CV, COUT, CVO, KE><<<grid, S::NWARP * 32, S::SMEM, st>>>(*p, p->W1tc, reinterpret_cast<const float4*>(p->tab4), ntiles);
    SV_CHECK_LAUNCH("svnet_svblock_edge_fwd(tcgen05, fp)");
    return SVNET_OK;
}

// The instantiated (shape, k) pairs: the three fp edge layers of SV_DGCNN_CLS at k = 20 and of SV_DGCNN_PSEG at k = 20 / 40.
// svnet_edge_fp_tc_weight_bytes goes through ftc_covered, which reads this list; svnet_edge_fp_tc_dispatch has one FCASE per
// entry and no other, so a covered layer always finds its kernel.
struct ftc_case { int cs, cv, co, cvo, k; };
const ftc_case kFCases[] = {{32, 10, 32, 10, 20}, {32, 10, 64, 21, 20}, {64, 21, 128, 42, 20},
                            {32, 16, 32, 16, 20}, {32, 16, 64, 24, 20}, {64, 24, 128, 40, 20},
                            {32, 16, 32, 16, 40}, {32, 16, 64, 24, 40}, {64, 24, 128, 40, 40}};

bool ftc_covered(int cs, int cv, int co, int cvo, int k)
{
    const char* off = getenv("SVNET_EDGE_FP_TC");
    if (off && off[0] == '0') return false;
    const char* tc = getenv("SVNET_TCGEN05");          // the per-point table comes from the tcgen05 vector linear
    if (tc && tc[0] == '0') return false;
    const char* fp = getenv("SVNET_VLINEAR_FP_TC");    // ... with full-precision weights: its three-plane path
    if (fp && fp[0] == '0') return false;
    const char* gen = getenv("SVNET_EDGE_GENERIC");    // the generic kernel reads the P | Q table, not the float4 one
    if (gen && gen[0] == '1') return false;
    for (const ftc_case& s : kFCases)
        if (s.cs == cs && s.cv == cv && s.co == co && s.cvo == cvo && s.k == k) return true;
    return false;
}

}  // namespace

extern "C" size_t svnet_edge_fp_tc_weight_bytes(int Cs, int Cv, int Cout, int Cvo, int k)
{
    if (!ftc_covered(Cs, Cv, Cout, Cvo, k)) return 0;
    const int KH = (3 * Cv + 15) / 16 * 16;
    return (size_t)3 * (2 * KH / 8) * (Cout <= 64 ? 64 : 128) * 16 + 1024;      // + the rows the last k-block's 128-row read overhangs
}

extern "C" int svnet_edge_fp_tc_pack_w(const float* W1, int ldw, int Cs, int Cv, int Cout, unsigned char* out, void* stream)
{
    SV_REQUIRE(W1 && out, "svnet_edge_fp_tc_pack_w: null pointer");
    SV_REQUIRE(Cs >= 1 && Cv >= 1 && Cv <= 32 && Cout >= 1 && Cout <= 128, "svnet_edge_fp_tc_pack_w: shape not covered");
    SV_REQUIRE(ldw >= 2 * Cs + 6 * Cv, "svnet_edge_fp_tc_pack_w: ldw too small");
    const int KH = (3 * Cv + 15) / 16 * 16;
    const int arows = Cout <= 64 ? 64 : 128;
    SV_CUDA(cudaMemsetAsync(out + (size_t)3 * (2 * KH / 8) * arows * 16, 0, 1024, sv_stream(stream)));
    edge_fp_tc_pack_w_kernel<<<sv_cdiv((long)(2 * KH / 8) * arows, 256), 256, 0, sv_stream(stream)>>>(W1, ldw, Cs, Cv, Cout, KH, arows, out);
    SV_CHECK_LAUNCH("svnet_edge_fp_tc_pack_w");
    return SVNET_OK;
}

// Returns 1 if the tensor-core kernel handled the layer, 0 if the caller must use another kernel, < 0 on error.
int svnet_edge_fp_tc_dispatch(const svnet_edge_params* p, cudaStream_t st)
{
    if (p->binary || !p->W1tc || !p->tab4 || !p->Yab) return 0;
    const int cs = p->in.Cs, cv = p->in.Cv, co = p->Cout, cvo = p->Cvo, k = p->k;
    if (!ftc_covered(cs, cv, co, cvo, k)) return 0;
    if ((reinterpret_cast<uintptr_t>(p->W1tc) & 15) || (reinterpret_cast<uintptr_t>(p->tab4) & 15)) return 0;
    int rc = 0;
#define FCASE(A, Bv, C, D, KE) \
    if (cs == A && cv == Bv && co == C && cvo == D && k == KE) { rc = launch_ftc<A, Bv, C, D, KE>(p, st); return rc == SVNET_OK ? 1 : rc; }
    FCASE(32, 10, 32, 10, 20)
    FCASE(32, 10, 64, 21, 20)
    FCASE(64, 21, 128, 42, 20)
    FCASE(32, 16, 32, 16, 20)
    FCASE(32, 16, 64, 24, 20)
    FCASE(64, 24, 128, 40, 20)
    FCASE(32, 16, 32, 16, 40)
    FCASE(32, 16, 64, 24, 40)
    FCASE(64, 24, 128, 40, 40)
#undef FCASE
    return 0;
}
