// Generic fp32 linear over (grouped) rows on the CUDA cores, with the epilogues the SV layers need.
// C[m][n] = epi(sum_k A[m][k] * W[n][k]); the k loop is one sequential fmaf chain per output, which
// is the oracle's order, so fp layers that go through here are bit-reproducible.
// Used for: per-point tables of the fused edge kernel (P|Q, Ya|Yb), fp linear1 on rows, the vector
// branch of per-row SVBlocks (VectorBN + gate epilogue, groups of 3 rows), heads, conv7/conv11.
// Reference: models/sv_layers.py:29-53 (Linear), :86-102 (VectorBN), :192-194.
#include "common.cuh"

int svnet_signlinear_tc_dispatch(const svnet_gemm_params* p, cudaStream_t st);
int svnet_vlinear_tcgen05_dispatch(const svnet_gemm_params* p, cudaStream_t st);
size_t svnet_linear_tc3_workspace(const svnet_gemm_params* p);
int svnet_linear_tc3_dispatch(const svnet_gemm_params* p, void* workspace, size_t workspace_bytes, cudaStream_t st);

namespace {

constexpr int BN_ = 64, BK = 16;

__device__ __forceinline__ int swz(int kk, int m) { return m ^ ((kk & 7) << 2); }

template <int TM>
__global__ void __launch_bounds__(256) linear_rows_kernel(svnet_gemm_params p)
{
    constexpr int BM = 16 * TM;
    constexpr int BMP = 64;  // padded row count (>= BM, multiple of 32 so that the swizzle stays in range)
    __shared__ __align__(16) float As[BK][BMP];
    __shared__ __align__(16) float Ws[BK][BN_];
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const long m0 = (long)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN_;
    float acc[TM][4];
#pragma unroll
    for (int a = 0; a < TM; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][c] = 0.0f;

    for (int k0 = 0; k0 < p.K; k0 += BK) {
        __syncthreads();
        for (int i = tid; i < BM * BK; i += 256) {
            const int mm = i >> 4, kk = i & 15;
            const long m = m0 + mm;
            const int k = k0 + kk;
            float v = 0.0f;
            if (m < p.M && k < p.K) {
                long off;
                if (p.G == 1) off = m * p.lda_g;
                else if (p.G == 3) { const unsigned g = (unsigned)m / 3u; off = (long)g * p.lda_g + (long)((unsigned)m - 3u * g) * p.lda_x; }
                else off = (m / p.G) * p.lda_g + (m % p.G) * (long)p.lda_x;
                v = __ldg(p.A + off + k);
            }
            As[kk][swz(kk, mm)] = v;
        }
        for (int i = tid; i < BN_ * BK; i += 256) {
            const int nn = i >> 4, kk = i & 15;
            const int n = n0 + nn, k = k0 + kk;
            float v = 0.0f;
            if (n < p.N && k < p.K) {
                v = __ldg(p.W + (long)n * p.ldw + k);
                if (p.sign_w) v = (v > 0.0f) ? 1.0f : ((v < 0.0f) ? -1.0f : 0.0f);
            }
            Ws[kk][swz(kk, nn)] = v;
        }
        __syncthreads();
        const int kn = min(BK, p.K - k0);
        for (int kk = 0; kk < kn; ++kk) {
            const float4 w4 = *reinterpret_cast<const float4*>(&Ws[kk][swz(kk, tx * 4)]);
            const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
            for (int a = 0; a < TM; ++a) {
                const float av = As[kk][swz(kk, ty * TM + a)];
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[a][c] = __fmaf_rn(av, wv[c], acc[a][c]);
            }
        }
    }

    if (p.vbn) {
        // TM == 3: rows ty*3 .. ty*3+2 are x = 0,1,2 of one group
        const long m = m0 + ty * TM;
        if (m >= p.M) return;
        const long grp = m / 3;
        const long cloud = grp / p.groups_per_cloud;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int n = n0 + tx * 4 + c;
            if (n >= p.N) continue;
            float w[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) w[a] = p.colscale ? __fmul_rn(acc[a % TM][c], p.colscale[n]) : acc[a % TM][c];
            const float nrm = __fadd_rn(
                __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(w[0], w[0]), __fmul_rn(w[1], w[1])), __fmul_rn(w[2], w[2]))),
                1e-6f);
            const float nb = __fadd_rn(__fmul_rn(nrm, p.bn_a[n]), p.bn_c[n]);
            const float g = p.gate ? p.gate[cloud * p.N + n] : 1.0f;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                float t = __fmul_rn(__fdiv_rn(w[a], nrm), nb);
                if (p.gate) t = __fmul_rn(t, g);
                p.C[grp * p.ldc_g + a * (long)p.ldc_x + n] = t;
            }
        }
        return;
    }
#pragma unroll
    for (int a = 0; a < TM; ++a) {
        const long m = m0 + ty * TM + a;
        if (m >= p.M) continue;
        long coff;
        if (p.G == 1) coff = m * p.ldc_g;
        else if (p.G == 3) { const unsigned g = (unsigned)m / 3u; coff = (long)g * p.ldc_g + (long)((unsigned)m - 3u * g) * p.ldc_x; }
        else coff = (m / p.G) * p.ldc_g + (m % p.G) * (long)p.ldc_x;
        float* crow = p.C + coff;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int n = n0 + tx * 4 + c;
            if (n >= p.N) continue;
            float v = acc[a][c];
            if (p.colscale) v = __fmul_rn(v, p.colscale[n]);
            if (p.bias) v = __fadd_rn(v, p.bias[n]);
            if (p.bn_a) v = __fadd_rn(__fmul_rn(v, p.bn_a[n]), p.bn_c[n]);
            crow[n] = sv_act(v, p.act);
        }
    }
}

}  // namespace

extern "C" size_t svnet_linear_workspace_bytes(const svnet_gemm_params* p) { return svnet_linear_tc3_workspace(p); }

extern "C" int svnet_linear_rows(const svnet_gemm_params* p, void* stream)
{
    return svnet_linear_rows_ws(p, nullptr, 0, stream);
}

extern "C" int svnet_linear_rows_ws(const svnet_gemm_params* p, void* workspace, size_t workspace_bytes, void* stream)
{
    SV_REQUIRE(p, "svnet_linear_rows: null params");
    SV_REQUIRE(p->A && p->W && p->C, "svnet_linear_rows: null pointer");
    SV_REQUIRE(p->M >= 0 && p->N >= 1 && p->K >= 1 && p->G >= 1 && p->ldw >= p->K, "svnet_linear_rows: bad shape");
    SV_REQUIRE(p->M < (1L << 31), "svnet_linear_rows: M too large");
    SV_REQUIRE((p->bn_a == nullptr) == (p->bn_c == nullptr), "svnet_linear_rows: bn_a/bn_c must come together");
    if (p->vbn) {
        SV_REQUIRE(p->G == 3 && p->M % 3 == 0 && p->bn_a, "svnet_linear_rows: vbn needs G == 3, M %% 3 == 0 and bn");
        SV_REQUIRE(!p->gate || p->groups_per_cloud >= 1, "svnet_linear_rows: groups_per_cloud");
    }
    if (p->M == 0) return SVNET_OK;
    cudaStream_t st = sv_stream(stream);
    if (workspace) {   // plain fp32 linear over many rows: three-plane bf16 tcgen05 kernel (gemm_tc3.cu)
        const int h = svnet_linear_tc3_dispatch(p, workspace, workspace_bytes, st);
        if (h < 0) return h;
        if (h == 1) return SVNET_OK;
    }
    {   // binary-weight vector linear + VectorBN: tcgen05 / TMEM kernel (gemm_tcgen05.cu)
        const int h = svnet_vlinear_tcgen05_dispatch(p, st);
        if (h < 0) return h;
        if (h == 1) return SVNET_OK;
    }
    SV_REQUIRE(!p->c4, "svnet_linear_rows: the c4 table layout needs the tcgen05 vector-linear path (G == 3, K <= 96, N <= 256, "
                       "no bias / BN / activation; full-precision weights also need SVNET_TCGEN05 and SVNET_VLINEAR_FP_TC not 0)");
    {   // binary-weight vector linears: exact-split bf16 mma.sync kernel (gemm_tc.cu)
        const int h = svnet_signlinear_tc_dispatch(p, st);
        if (h < 0) return h;
        if (h == 1) return SVNET_OK;
    }
    if (p->vbn) {
        dim3 grid(sv_cdiv(p->M, 48), sv_cdiv(p->N, BN_));
        linear_rows_kernel<3><<<grid, 256, 0, st>>>(*p);
    } else {
        dim3 grid(sv_cdiv(p->M, 64), sv_cdiv(p->N, BN_));
        linear_rows_kernel<4><<<grid, 256, 0, st>>>(*p);
    }
    SV_CHECK_LAUNCH("svnet_linear_rows");
    return SVNET_OK;
}
