// K2 -- fused SV edge convolution for layers 2..4:
//   get_graph_feature_sv + SVBlock + svpool in one pass, no edge tensor in HBM.
// Reference: models/utils/sv_util.py:90-132, models/sv_layers.py:29-53,86-129,172-196,
//            models/sv_dgcnn_cls.py:55-65.
//
// One warp per centre point i.  The warp
//   A. stages the centre row and, three neighbours at a time, the gathered rows in shared memory;
//      computes the 3x3 frames z = v_e Wz^T (27 lanes = 3 edges x 9 entries, sequential fmaf chain
//      over channels == oracle order), then u = [s_j - s_i | s_i | q] lane-per-channel and
//      packs sign(u + beta) with __ballot_sync into 32-bit words plus a non-zero mask plane
//      (torch.sign(0) == 0) -- binary model; or stores q as floats -- fp model.
//   B. binary: XNOR/popcount linear1, lanes = output channels, accumulating EB edges at a time;
//      y = scale * (nvalid - 2*popc((a ^ w) & m)); BN affine; LeakyReLU; running max over edges.
//      fp: y = (Ya_j - Ya_i) + Yb_i + W1q q with the per-point tables Ya/Yb.
//   C. vector branch from the per-point tables P = v W2a^T, Q = v W2b^T:
//      w = (P_j - P_i) + Q_i; VectorBN; gate; mean over edges.
#include "common.cuh"
#include <stdlib.h>

int svnet_edge_fast_dispatch(const svnet_edge_params* p, cudaStream_t st);
int svnet_edge_tc_dispatch(const svnet_edge_params* p, cudaStream_t st);
int svnet_edge_fp_tc_dispatch(const svnet_edge_params* p, cudaStream_t st);

namespace {

constexpr int WARPS = 8;
constexpr int EB = 10;   // edges accumulated per pass in phase B
constexpr int EG = 3;    // edges staged per group in phase A

struct Smem {
    // shared by the CTA
    float* Wz;      // [3][Cve]
    float* beta;    // [K]
    uint32_t* W1b;  // [Kw][Cout]
    float* scale1;  // [Cout]
    float* a1;
    float* c1;
    float* a2;      // [Cvo]
    float* c2;
    float* zscale;  // [3]
    // per warp
    float* ctr;     // [F]
    float* nb;      // [EG][F]
    float* zb;      // [EG][9]
    uint32_t* A;    // [Kw][kp]
    uint32_t* M;    // [Kw][kp]
    int* nvalid;    // [kp]
    int* nidx;      // [kp]
    float* q;       // fp: [EB][3*Cve]
};

struct Dims {
    int Cs, Cv, Cve, F, K, Kw, kp, Cout, Cvo, k;
    size_t shared_floats, warp_floats;
};

__host__ __device__ inline Dims make_dims(int Cs, int Cv, int k, int Cout, int Cvo, bool binary)
{
    Dims d;
    d.Cs = Cs; d.Cv = Cv; d.Cve = 2 * Cv; d.F = Cs + 3 * Cv; d.K = 2 * Cs + 6 * Cv; d.Kw = (d.K + 31) / 32;
    d.k = k; d.kp = ((k + EB - 1) / EB) * EB; d.Cout = Cout; d.Cvo = Cvo;
    d.shared_floats = (size_t)3 * d.Cve + d.K + (binary ? (size_t)d.Kw * Cout : 0) + 3 * (size_t)Cout + 2 * (size_t)Cvo + 4;
    d.warp_floats = (size_t)d.F * (1 + EG) + EG * 9 + 3 +
                    (binary ? (size_t)2 * d.Kw * d.kp + d.kp : (size_t)EB * 3 * d.Cve) + d.kp;
    return d;
}

__device__ inline Smem carve(float* base, const Dims& d, bool binary, int warp)
{
    Smem s;
    float* p = base;
    s.Wz = p; p += 3 * d.Cve;
    s.beta = p; p += d.K;
    s.W1b = reinterpret_cast<uint32_t*>(p); p += binary ? (size_t)d.Kw * d.Cout : 0;
    s.scale1 = p; p += d.Cout;
    s.a1 = p; p += d.Cout;
    s.c1 = p; p += d.Cout;
    s.a2 = p; p += d.Cvo;
    s.c2 = p; p += d.Cvo;
    s.zscale = p; p += 4;
    p += (size_t)warp * d.warp_floats;
    s.ctr = p; p += d.F;
    s.nb = p; p += (size_t)EG * d.F;
    s.zb = p; p += EG * 9 + 3;
    if (binary) {
        s.A = reinterpret_cast<uint32_t*>(p); p += (size_t)d.Kw * d.kp;
        s.M = reinterpret_cast<uint32_t*>(p); p += (size_t)d.Kw * d.kp;
        s.nvalid = reinterpret_cast<int*>(p); p += d.kp;
        s.q = nullptr;
    } else {
        s.A = s.M = nullptr; s.nvalid = nullptr;
        s.q = p; p += (size_t)EB * 3 * d.Cve;
    }
    s.nidx = reinterpret_cast<int*>(p);
    return s;
}

__device__ __forceinline__ void load_row(float* dst, const svnet_view& in, long r, int lane)
{
    for (int c = lane; c < in.Cs; c += 32) dst[c] = __ldg(in.s + r * in.lds + c);
#pragma unroll
    for (int x = 0; x < 3; ++x)
        for (int c = lane; c < in.Cv; c += 32) dst[in.Cs + x * in.Cv + c] = __ldg(in.v + r * in.ldv + x * in.xs + c);
}

// z frames for up to EG staged edges: lane -> (g, x, m)
__device__ __forceinline__ void compute_z(const Smem& s, const Dims& d, int lane, bool use_zscale)
{
    if (lane < EG * 9) {
        const int g = lane / 9, xm = lane - g * 9, x = xm / 3, m = xm - x * 3;
        const float* nv = s.nb + (size_t)g * d.F + d.Cs + x * d.Cv;
        const float* cv = s.ctr + d.Cs + x * d.Cv;
        const float* wz = s.Wz + m * d.Cve;
        float acc = 0.0f;
#pragma unroll 8
        for (int c = 0; c < d.Cv; ++c) acc = __fmaf_rn(__fsub_rn(nv[c], cv[c]), wz[c], acc);
#pragma unroll 8
        for (int c = 0; c < d.Cv; ++c) acc = __fmaf_rn(cv[c], wz[d.Cv + c], acc);
        if (use_zscale) acc = __fmul_rn(acc, s.zscale[m]);
        s.zb[lane] = acc;
    }
}

// q[d][m] of staged edge g for flattened index t = d*3 + m  (sv_layers.py:117-125)
__device__ __forceinline__ float compute_q(const Smem& s, const Dims& d, int g, int t)
{
    const int dd = t / 3, m = t - dd * 3;
    const float* z = s.zb + g * 9;
    float ve[3];
    if (dd < d.Cv) {
        const float* nv = s.nb + (size_t)g * d.F + d.Cs + dd;
        const float* cv = s.ctr + d.Cs + dd;
#pragma unroll
        for (int x = 0; x < 3; ++x) ve[x] = __fsub_rn(nv[x * d.Cv], cv[x * d.Cv]);
    } else {
        const float* cv = s.ctr + d.Cs + (dd - d.Cv);
#pragma unroll
        for (int x = 0; x < 3; ++x) ve[x] = cv[x * d.Cv];
    }
    float q = __fmul_rn(ve[0], z[m]);
    q = __fmaf_rn(ve[1], z[3 + m], q);
    q = __fmaf_rn(ve[2], z[6 + m], q);
    return q;
}

template <bool BIN, int OPT>
__global__ void __launch_bounds__(WARPS * 32, 3) svblock_edge_kernel(svnet_edge_params p)
{
    extern __shared__ __align__(16) float smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const Dims d = make_dims(p.in.Cs, p.in.Cv, p.k, p.Cout, p.Cvo, BIN);
    const Smem s = carve(smem_raw, d, BIN, warp);

    // ---- CTA-shared parameters ----
    for (int i = threadIdx.x; i < 3 * d.Cve; i += blockDim.x) s.Wz[i] = p.Wz[i];
    if (BIN) {
        for (int i = threadIdx.x; i < d.K; i += blockDim.x) s.beta[i] = p.beta[i];
        for (int i = threadIdx.x; i < d.Kw * d.Cout; i += blockDim.x) s.W1b[i] = p.W1b[i];
        for (int i = threadIdx.x; i < d.Cout; i += blockDim.x) s.scale1[i] = p.scale1[i];
    }
    for (int i = threadIdx.x; i < d.Cout; i += blockDim.x) { s.a1[i] = p.bn1_a[i]; s.c1[i] = p.bn1_c[i]; }
    for (int i = threadIdx.x; i < d.Cvo; i += blockDim.x) { s.a2[i] = p.bn2_a[i]; s.c2[i] = p.bn2_c[i]; }
    if (threadIdx.x < 3) s.zscale[threadIdx.x] = p.zscale ? p.zscale[threadIdx.x] : 1.0f;
    __syncthreads();

    const long r = (long)blockIdx.x * WARPS + warp;
    if (r >= (long)p.B * p.N) return;
    const int b = (int)(r / p.N);
    const long cbase = (long)b * p.N;
    const bool use_zscale = p.zscale != nullptr;

    load_row(s.ctr, p.in, r, lane);
    for (int e = lane; e < d.kp; e += 32) s.nidx[e] = e < p.k ? p.idx[r * p.k + e] : 0;
    if (BIN) {
        for (int i = lane; i < d.Kw * d.kp; i += 32) { s.A[i] = 0u; s.M[i] = 0u; }
        for (int e = lane; e < d.kp; e += 32) s.nvalid[e] = 0;
    }
    __syncwarp();

    float smax[OPT];
#pragma unroll
    for (int oo = 0; oo < OPT; ++oo) smax[oo] = -INFINITY;

    if (BIN) {
        // ================= phase A (binary): sign words for all k edges =================
        for (int e0 = 0; e0 < p.k; e0 += EG) {
            const int ng = min(EG, p.k - e0);
            for (int g = 0; g < ng; ++g) load_row(s.nb + (size_t)g * d.F, p.in, cbase + s.nidx[e0 + g], lane);
            for (int g = ng; g < EG; ++g) for (int c = lane; c < d.F; c += 32) s.nb[(size_t)g * d.F + c] = 0.0f;
            __syncwarp();
            compute_z(s, d, lane, use_zscale);
            __syncwarp();
            for (int g = 0; g < ng; ++g) {
                const int e = e0 + g;
                const float* nrow = s.nb + (size_t)g * d.F;
                int nval = 0;
#pragma unroll 4
                for (int wd = 0; wd < d.Kw; ++wd) {
                    const int kk = wd * 32 + lane;
                    float u = 0.0f;
                    if (kk < d.Cs) u = __fsub_rn(nrow[kk], s.ctr[kk]);
                    else if (kk < 2 * d.Cs) u = s.ctr[kk - d.Cs];
                    else if (kk < d.K) u = compute_q(s, d, g, kk - 2 * d.Cs);
                    const float t = (kk < d.K) ? __fadd_rn(u, s.beta[kk]) : 0.0f;
                    const unsigned pos = __ballot_sync(SV_FULL, t > 0.0f);
                    const unsigned nz = __ballot_sync(SV_FULL, t != 0.0f);
                    nval += __popc(nz);
                    if (lane == 0) {
                        s.A[wd * d.kp + e] = pos;
                        s.M[wd * d.kp + e] = nz;
                        if (p.dbg_bits) p.dbg_bits[(r * p.k + e) * d.Kw + wd] = pos;
                        if (p.dbg_mask) p.dbg_mask[(r * p.k + e) * d.Kw + wd] = nz;
                    }
                }
                if (lane == 0) s.nvalid[e] = nval;
            }
            __syncwarp();
        }
        // ================= phase B (binary): XNOR/popcount linear1 + BN + leaky + max =================
        for (int eb = 0; eb < p.k; eb += EB) {
            int acc[EB][OPT];
#pragma unroll
            for (int e = 0; e < EB; ++e)
#pragma unroll
                for (int oo = 0; oo < OPT; ++oo) acc[e][oo] = 0;
            for (int wd = 0; wd < d.Kw; ++wd) {
                uint32_t wv[OPT];
#pragma unroll
                for (int oo = 0; oo < OPT; ++oo) {
                    const int o = lane + 32 * oo;
                    wv[oo] = (o < d.Cout) ? s.W1b[wd * d.Cout + o] : 0u;
                }
                const uint32_t* Ap = s.A + wd * d.kp + eb;
                const uint32_t* Mp = s.M + wd * d.kp + eb;
#pragma unroll
                for (int e = 0; e < EB; ++e) {
                    const uint32_t a = Ap[e], m = Mp[e];
#pragma unroll
                    for (int oo = 0; oo < OPT; ++oo) acc[e][oo] += __popc((a ^ wv[oo]) & m);
                }
            }
#pragma unroll
            for (int oo = 0; oo < OPT; ++oo) {
                const int o = lane + 32 * oo;
                if (o < d.Cout) {
                    const float sc = s.scale1[o], a1 = s.a1[o], c1 = s.c1[o];
#pragma unroll
                    for (int e = 0; e < EB; ++e) {
                        if (eb + e < p.k) {
                            const int dot = s.nvalid[eb + e] - 2 * acc[e][oo];
                            float y = __fmul_rn((float)dot, sc);
                            y = __fadd_rn(__fmul_rn(y, a1), c1);
                            y = y > 0.0f ? y : __fmul_rn(0.2f, y);
                            smax[oo] = fmaxf(smax[oo], y);
                        }
                    }
                }
            }
        }
    } else {
        // ================= fp: per block of EB edges, q floats then dense linear1 =================
        const int KQ = 3 * d.Cve;
        for (int eb = 0; eb < p.k; eb += EB) {
            const int ne = min(EB, p.k - eb);
            for (int e0 = 0; e0 < ne; e0 += EG) {
                const int ng = min(EG, ne - e0);
                for (int g = 0; g < ng; ++g) load_row(s.nb + (size_t)g * d.F, p.in, cbase + s.nidx[eb + e0 + g], lane);
                for (int g = ng; g < EG; ++g) for (int c = lane; c < d.F; c += 32) s.nb[(size_t)g * d.F + c] = 0.0f;
                __syncwarp();
                compute_z(s, d, lane, use_zscale);
                __syncwarp();
                for (int g = 0; g < ng; ++g)
                    for (int t = lane; t < KQ; t += 32) s.q[(size_t)(e0 + g) * KQ + t] = compute_q(s, d, g, t);
                __syncwarp();
            }
            for (int e = ne; e < EB; ++e) for (int t = lane; t < KQ; t += 32) s.q[(size_t)e * KQ + t] = 0.0f;
            __syncwarp();
            float acc[EB][OPT];
#pragma unroll
            for (int oo = 0; oo < OPT; ++oo) {
                const int o = lane + 32 * oo;
                const float ya_i = (o < d.Cout) ? __ldg(p.Yab + r * 2 * d.Cout + o) : 0.0f;
                const float yb_i = (o < d.Cout) ? __ldg(p.Yab + r * 2 * d.Cout + d.Cout + o) : 0.0f;
#pragma unroll
                for (int e = 0; e < EB; ++e) {
                    const long j = cbase + s.nidx[eb + e];
                    const float ya_j = (o < d.Cout) ? __ldg(p.Yab + j * 2 * d.Cout + o) : 0.0f;
                    acc[e][oo] = (ya_j - ya_i) + yb_i;
                }
            }
            for (int t = 0; t < KQ; ++t) {
                float wv[OPT];
#pragma unroll
                for (int oo = 0; oo < OPT; ++oo) {
                    const int o = lane + 32 * oo;
                    wv[oo] = (o < d.Cout) ? __ldg(p.W1q_t + (size_t)t * d.Cout + o) : 0.0f;
                }
#pragma unroll
                for (int e = 0; e < EB; ++e) {
                    const float qv = s.q[(size_t)e * KQ + t];
#pragma unroll
                    for (int oo = 0; oo < OPT; ++oo) acc[e][oo] = fmaf(qv, wv[oo], acc[e][oo]);
                }
            }
#pragma unroll
            for (int oo = 0; oo < OPT; ++oo) {
                const int o = lane + 32 * oo;
                if (o < d.Cout) {
                    const float a1 = s.a1[o], c1 = s.c1[o];
#pragma unroll
                    for (int e = 0; e < EB; ++e) {
                        if (e < ne) {
                            float y = __fadd_rn(__fmul_rn(acc[e][oo], a1), c1);
                            y = y > 0.0f ? y : __fmul_rn(0.2f, y);
                            smax[oo] = fmaxf(smax[oo], y);
                        }
                    }
                }
            }
            __syncwarp();
        }
    }
#pragma unroll
    for (int oo = 0; oo < OPT; ++oo) {
        const int o = lane + 32 * oo;
        if (o < d.Cout) p.out.s[r * p.out.lds + o] = smax[oo];
    }

    // ================= phase C: vector branch =================
    const int ldp = 2 * d.Cvo;
    const float inv_k = 1.0f / (float)p.k;
    for (int c = lane; c < d.Cvo; c += 32) {
        const float* pi = p.PQ + r * 3 * ldp + c;
        const float p_i[3] = {__ldg(pi), __ldg(pi + ldp), __ldg(pi + 2 * ldp)};
        const float q_i[3] = {__ldg(pi + d.Cvo), __ldg(pi + ldp + d.Cvo), __ldg(pi + 2 * ldp + d.Cvo)};
        const float a2 = s.a2[c], c2 = s.c2[c];
        float sum[3] = {0.0f, 0.0f, 0.0f};
#pragma unroll 4
        for (int e = 0; e < p.k; ++e) {
            const float* pj = p.PQ + (cbase + s.nidx[e]) * 3 * ldp + c;
            float w[3];
#pragma unroll
            for (int x = 0; x < 3; ++x) w[x] = (__ldg(pj + x * ldp) - p_i[x]) + q_i[x];
            const float n = sqrtf(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]) + 1e-6f;
            const float t = (n * a2 + c2) / n;
#pragma unroll
            for (int x = 0; x < 3; ++x) sum[x] += w[x] * t;
        }
        const float g = p.gate[(long)b * d.Cvo + c] * inv_k;
#pragma unroll
        for (int x = 0; x < 3; ++x) p.out.v[r * p.out.ldv + x * p.out.xs + c] = sum[x] * g;
    }
}

template <bool BIN>
int launch_edge(const svnet_edge_params* p, cudaStream_t st)
{
    const Dims d = make_dims(p->in.Cs, p->in.Cv, p->k, p->Cout, p->Cvo, BIN);
    const size_t smem = sizeof(float) * (d.shared_floats + WARPS * d.warp_floats);
    SV_REQUIRE(smem <= 220 * 1024, "svnet_svblock_edge_fwd: shared memory %zu B too large (Cs=%d Cv=%d k=%d Cout=%d)", smem,
               d.Cs, d.Cv, d.k, d.Cout);
    const int grid = sv_cdiv((long)p->B * p->N, WARPS);
    const int opt = (p->Cout + 31) / 32;
#define LAUNCH(O)                                                                                               \
    do {                                                                                                        \
        SV_CUDA(cudaFuncSetAttribute(svblock_edge_kernel<BIN, O>, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                     (int)smem));                                                               \
        svblock_edge_kernel<BIN, O><<<grid, WARPS * 32, smem, st>>>(*p);                                        \
    } while (0)
    if (opt == 1) LAUNCH(1);
    else if (opt == 2) LAUNCH(2);
    else if (opt <= 4) LAUNCH(4);
    else { SV_REQUIRE(false, "svnet_svblock_edge_fwd: Cout=%d > 128 unsupported", p->Cout); }
#undef LAUNCH
    SV_CHECK_LAUNCH("svnet_svblock_edge_fwd");
    return SVNET_OK;
}

}  // namespace

extern "C" int svnet_svblock_edge_fwd(const svnet_edge_params* p, void* stream)
{
    SV_REQUIRE(p, "svnet_svblock_edge_fwd: null params");
    SV_REQUIRE(p->in.s && p->in.v && p->idx && p->Wz && p->bn1_a && p->bn1_c && (p->PQ || (p->tab4 && p->W1tc)) && p->bn2_a &&
                   p->bn2_c && p->gate && p->out.s && p->out.v,
               "svnet_svblock_edge_fwd: null pointer");
    SV_REQUIRE(p->in.Cs >= 1 && p->in.Cv >= 1 && p->B >= 0 && p->N >= 1 && p->k >= 1 && p->Cout >= 1 && p->Cvo >= 1,
               "svnet_svblock_edge_fwd: bad shape");
    if ((long)p->B * p->N == 0) return SVNET_OK;
    if (p->binary) {
        SV_REQUIRE(p->beta && p->W1b && p->scale1, "svnet_svblock_edge_fwd: binary layer needs beta/W1b/scale1");
        // shapes of the SV-DGCNN models have compile-time specialisations (edge_fast.cu, edge_tc.cu);
        // SVNET_EDGE_GENERIC=1 forces the generic kernel below (tests/test_gpu_edge_fp64.py runs it next to the
        // specialised ones against a float64 restatement of the layer)
        const char* force = getenv("SVNET_EDGE_GENERIC");
        if (!(force && force[0] == '1')) {
            // tensor-core kernel when the caller supplied its packed weights and table scratch (edge_tc.cu)
            int h = svnet_edge_tc_dispatch(p, sv_stream(stream));
            if (h < 0) return h;
            if (h == 1) return SVNET_OK;
            SV_REQUIRE(p->PQ, "svnet_svblock_edge_fwd: layer not covered by the tensor-core kernel and no PQ table given");
            h = svnet_edge_fast_dispatch(p, sv_stream(stream));
            if (h < 0) return h;
            if (h == 1) return SVNET_OK;
        }
        SV_REQUIRE(p->PQ, "svnet_svblock_edge_fwd: the generic kernel needs the PQ table");
        return launch_edge<true>(p, sv_stream(stream));
    }
    SV_REQUIRE(p->Yab, "svnet_svblock_edge_fwd: fp layer needs Yab");
    {
        const char* force = getenv("SVNET_EDGE_GENERIC");
        if (!(force && force[0] == '1')) {
            // tensor-core kernel when the caller supplied the packed weight planes and the float4 table (edge_fp_tc.cu)
            int h = svnet_edge_fp_tc_dispatch(p, sv_stream(stream));
            if (h < 0) return h;
            if (h == 1) return SVNET_OK;
        }
    }
    SV_REQUIRE(p->W1q_t && p->PQ, "svnet_svblock_edge_fwd: fp layer not covered by the tensor-core kernel needs W1q_t and PQ");
    {
        const char* force = getenv("SVNET_EDGE_GENERIC");
        if (!(force && force[0] == '1')) {
            const int h = svnet_edge_fast_dispatch(p, sv_stream(stream));
            if (h < 0) return h;
            if (h == 1) return SVNET_OK;
        }
    }
    return launch_edge<false>(p, sv_stream(stream));
}
