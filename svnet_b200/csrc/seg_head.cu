// K5 -- part-segmentation head as ONE C-ABI call (reference models/sv_dgcnn_partseg.py:112-126; SURVEY 8(b)
// `svnet_seg_head_fwd`):
//     conv8 ([per-cloud channels | svfuse1(s_cat, v_cat)] -> C8) -> conv9 -> conv10 (binarised Conv1d + BN + LeakyReLU,
//     sv_layers.py:64-78) -> conv11 (fp Conv1d C10 -> parts) -> logits written in the reference's (B, parts, N) order.
// The call sequences this library's own kernels on the caller's stream with caller-owned scratch:
//   * the per-cloud-constant leading channels of conv8 (`repeat(1, 1, num_points)`, sv_dgcnn_partseg.py:118) are reduced
//     once per cloud to integer dot products (sign-pack + XNOR/popcount, rows = B) and added per point;
//   * conv8's per-point sign words come straight from (s_cat, v_cat) (svfuse1's float table is never written) -- or
//     from the caller, who can compute them early on another stream (svnet_rows_prep) and pass them in;
//   * conv8 / conv9 / conv10: binarised linears on the tcgen05 tensor cores where covered (csrc/binlinear_tc.cu; bit-identical
//     to the popcount kernel), each followed by the sign-pack of its activation;
//   * conv11: three-plane tcgen05 GEMM (csrc/gemm_tc3.cu) into a row-major scratch, then one tiled transpose.
// Bit-identical to the same layers called one by one through svnet_rows_prep / svnet_binlinear_rows_ws /
// svnet_linear_rows_ws (tests/test_gpu_parity.py::test_seg_head_call_equals_layerwise).
//
// svnet_seg_head_fp_fwd: the same head of the full-precision model.  svfuse1's rows u = [s | v2s(v)] go to the workspace;
// conv8's per-cloud part W8[:, :Kc] glob[b] is one linear over the B clouds, added per point in the epilogue of the per-point
// linear (K = Cs + 3Cv instead of Kc + Cs + 3Cv); conv9 .. conv11 as the module's fp Conv1d layers.  Every linear goes through
// svnet_linear_rows_ws: the three-plane tcgen05 kernel (csrc/gemm_tc3.cu) where it covers (K, N), the CUDA-core chain otherwise
// (conv11 with fewer than 32 parts); the per-point conv8, which carries the per-cloud term, needs the tcgen05 kernel.
#include "common.cuh"

int svnet_linear_tc3_rowadd(const svnet_gemm_params* p, const float* rowadd, long rows_per_add, long ld_add, void* workspace,
                            size_t workspace_bytes, cudaStream_t st);

namespace {

// (R = B*N, P) row-major -> (B, P, N)
__global__ void __launch_bounds__(256) seg_transpose_kernel(const float* __restrict__ in, int P, long N, float* __restrict__ out)
{
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    const long n0 = (long)blockIdx.x * 32;
    const int p0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
    for (int i = ty; i < 32; i += 8) {
        const long n = n0 + i;
        const int p = p0 + tx;
        tile[i][tx] = (n < N && p < P) ? __ldg(in + ((long)b * N + n) * P + p) : 0.0f;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int p = p0 + i;
        const long n = n0 + tx;
        if (p < P && n < N) out[((long)b * P + p) * N + n] = tile[tx][i];
    }
}

inline size_t a256(size_t x) { return (x + 255) & ~(size_t)255; }

struct seg_plan {
    size_t cb, cm, cn, cdot, bits, mask, nvalid, hA, hB, blws, lws, total;
    size_t blws_bytes, lws_bytes;
};

svnet_gemm_params conv11_params(const svnet_seg_head_params* p, const float* h10, float* out_rm)
{
    svnet_gemm_params g = {};
    g.A = h10; g.lda_g = p->C10; g.lda_x = 0; g.G = 1;
    g.W = p->W11; g.ldw = p->C10;
    g.M = (long)p->B * p->N; g.N = p->parts; g.K = p->C10;
    g.C = out_rm; g.ldc_g = p->parts; g.ldc_x = 0;
    return g;
}

bool make_plan(const svnet_seg_head_params* p, seg_plan* pl)
{
    const long R = (long)p->B * p->N;
    const int Kp = p->sv.Cs + 3 * p->sv.Cv;
    const int Kcw = (p->Kc + 31) / 32;
    int wmax = (Kp + 31) / 32;
    wmax = wmax > (p->C8 + 31) / 32 ? wmax : (p->C8 + 31) / 32;
    wmax = wmax > (p->C9 + 31) / 32 ? wmax : (p->C9 + 31) / 32;
    const int hAc = p->C8 > p->C10 ? p->C8 : p->C10;
    const int hBc = p->C9 > p->parts ? p->C9 : p->parts;
    size_t o = 0;
    pl->cb = o; o += a256((size_t)p->B * Kcw * 4);
    pl->cm = o; o += a256((size_t)p->B * Kcw * 4);
    pl->cn = o; o += a256((size_t)p->B * 4);
    pl->cdot = o; o += a256((size_t)p->B * p->C8 * 4);
    pl->bits = o; o += a256((size_t)R * wmax * 4);
    pl->mask = o; o += a256((size_t)R * wmax * 4);
    pl->nvalid = o; o += a256((size_t)R * 4);
    pl->hA = o; o += a256((size_t)R * hAc * 4);
    pl->hB = o; o += a256((size_t)R * hBc * 4);
    size_t b = svnet_binlinear_workspace_bytes(R, Kp, p->C8);
    const size_t b9 = svnet_binlinear_workspace_bytes(R, p->C8, p->C9), b10 = svnet_binlinear_workspace_bytes(R, p->C9, p->C10);
    b = b > b9 ? b : b9;
    b = b > b10 ? b : b10;
    pl->blws_bytes = b;
    pl->blws = o; o += a256(b);
    const svnet_gemm_params g = conv11_params(p, nullptr, nullptr);
    pl->lws_bytes = svnet_linear_workspace_bytes(&g);
    pl->lws = o; o += a256(pl->lws_bytes);
    pl->total = o;
    return true;
}

}  // namespace

extern "C" size_t svnet_seg_head_workspace_bytes(const svnet_seg_head_params* p)
{
    if (!p || p->B < 1 || p->N < 1) return 0;
    seg_plan pl;
    make_plan(p, &pl);
    return pl.total;
}

extern "C" int svnet_seg_head_fwd_nz(const svnet_seg_head_params* p, const uint32_t* W8c_nz, const uint32_t* W8p_nz,
                                     const uint32_t* W9_nz, const uint32_t* W10_nz, void* workspace, size_t workspace_bytes,
                                     void* stream)
{
    SV_REQUIRE(p && p->logits && p->glob && p->beta8 && p->W8c && p->W8p && p->beta9 && p->W9 && p->beta10 && p->W10 && p->W11,
               "svnet_seg_head_fwd: null pointer");
    SV_REQUIRE(p->B >= 0 && p->N >= 1 && p->Kc >= 1 && p->C8 >= 1 && p->C9 >= 1 && p->C10 >= 1 && p->parts >= 1,
               "svnet_seg_head_fwd: bad shape");
    SV_REQUIRE(p->bits8 || (p->sv.s && p->sv.v && p->Wz1), "svnet_seg_head_fwd: needs (s_cat, v_cat, Wz1) or conv8's sign words");
    SV_REQUIRE(!p->bits8 || (p->mask8 && p->nvalid8), "svnet_seg_head_fwd: bits8 needs mask8 and nvalid8");
    if (p->B == 0) return SVNET_OK;
    seg_plan pl;
    make_plan(p, &pl);
    SV_REQUIRE(workspace && workspace_bytes >= pl.total && !(reinterpret_cast<uintptr_t>(workspace) & 15),
               "svnet_seg_head_fwd: workspace too small (svnet_seg_head_workspace_bytes) or misaligned");
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    const long R = (long)p->B * p->N;
    const int Kp = p->sv.Cs + 3 * p->sv.Cv;
    uint32_t* cb = reinterpret_cast<uint32_t*>(ws + pl.cb);
    uint32_t* cm = reinterpret_cast<uint32_t*>(ws + pl.cm);
    int32_t* cn = reinterpret_cast<int32_t*>(ws + pl.cn);
    int32_t* cdot = reinterpret_cast<int32_t*>(ws + pl.cdot);
    uint32_t* bits = reinterpret_cast<uint32_t*>(ws + pl.bits);
    uint32_t* mask = reinterpret_cast<uint32_t*>(ws + pl.mask);
    int32_t* nvalid = reinterpret_cast<int32_t*>(ws + pl.nvalid);
    float* hA = reinterpret_cast<float*>(ws + pl.hA);
    float* hB = reinterpret_cast<float*>(ws + pl.hB);
    void* blws = pl.blws_bytes ? ws + pl.blws : nullptr;
    void* lws = pl.lws_bytes ? ws + pl.lws : nullptr;
    int rc;
    // ---- per-cloud-constant channels of conv8: sign-pack, integer dot products per cloud ----
    svnet_view gv = {};
    gv.s = p->glob; gv.lds = p->ldg; gv.Cs = p->Kc;
    rc = svnet_rows_prep(&gv, p->B, nullptr, nullptr, nullptr, p->beta8, nullptr, 0, nullptr, cb, cm, cn, stream);
    if (rc != SVNET_OK) return rc;
    rc = svnet_binlinear_rows_nz(cb, cm, cn, p->B, p->Kc, p->W8c, W8c_nz, p->C8, nullptr, nullptr, nullptr, nullptr, SVNET_ACT_NONE,
                                 nullptr, 1, nullptr, 0, cdot, nullptr, 0, stream);
    if (rc != SVNET_OK) return rc;
    // ---- conv8: per-point sign words of svfuse1(s_cat, v_cat), binarised linear + per-cloud part ----
    const uint32_t* b8 = p->bits8;
    const uint32_t* m8 = p->mask8;
    const int32_t* n8 = p->nvalid8;
    if (!b8) {
        rc = svnet_rows_prep(&p->sv, R, p->Wz1, p->zscale1, nullptr, p->beta8 + p->Kc, nullptr, 0, nullptr, bits, mask, nvalid, stream);
        if (rc != SVNET_OK) return rc;
        b8 = bits; m8 = mask; n8 = nvalid;
    }
    rc = svnet_binlinear_rows_nz(b8, m8, n8, R, Kp, p->W8p, W8p_nz, p->C8, p->scale8, nullptr, p->bn8_a, p->bn8_c, SVNET_ACT_LEAKY, cdot, p->N,
                                 hA, p->C8, nullptr, blws, pl.blws_bytes, stream);
    if (rc != SVNET_OK) return rc;
    // ---- conv9, conv10 ----
    svnet_view hv = {};
    hv.s = hA; hv.lds = p->C8; hv.Cs = p->C8;
    rc = svnet_rows_prep(&hv, R, nullptr, nullptr, nullptr, p->beta9, nullptr, 0, nullptr, bits, mask, nvalid, stream);
    if (rc != SVNET_OK) return rc;
    rc = svnet_binlinear_rows_nz(bits, mask, nvalid, R, p->C8, p->W9, W9_nz, p->C9, p->scale9, nullptr, p->bn9_a, p->bn9_c, SVNET_ACT_LEAKY,
                                 nullptr, 1, hB, p->C9, nullptr, blws, pl.blws_bytes, stream);
    if (rc != SVNET_OK) return rc;
    hv.s = hB; hv.lds = p->C9; hv.Cs = p->C9;
    rc = svnet_rows_prep(&hv, R, nullptr, nullptr, nullptr, p->beta10, nullptr, 0, nullptr, bits, mask, nvalid, stream);
    if (rc != SVNET_OK) return rc;
    rc = svnet_binlinear_rows_nz(bits, mask, nvalid, R, p->C9, p->W10, W10_nz, p->C10, p->scale10, nullptr, p->bn10_a, p->bn10_c,
                                 SVNET_ACT_LEAKY, nullptr, 1, hA, p->C10, nullptr, blws, pl.blws_bytes, stream);
    if (rc != SVNET_OK) return rc;
    // ---- conv11 (full precision) and the (B, N, parts) -> (B, parts, N) transpose ----
    const svnet_gemm_params g = conv11_params(p, hA, hB);
    rc = svnet_linear_rows_ws(&g, lws, pl.lws_bytes, stream);
    if (rc != SVNET_OK) return rc;
    seg_transpose_kernel<<<dim3(sv_cdiv(p->N, 32), sv_cdiv(p->parts, 32), p->B), 256, 0, sv_stream(stream)>>>(hB, p->parts, p->N, p->logits);
    SV_CHECK_LAUNCH("svnet_seg_head_fwd(transpose)");
    return SVNET_OK;
}

extern "C" int svnet_seg_head_fwd(const svnet_seg_head_params* p, void* workspace, size_t workspace_bytes, void* stream)
{
    return svnet_seg_head_fwd_nz(p, nullptr, nullptr, nullptr, nullptr, workspace, workspace_bytes, stream);
}

// ---- full-precision head ----------------------------------------------------------------------------------------------
namespace {

struct seg_fp_plan {
    size_t u, cterm, hA, hB, lws, total, lws_bytes;
};

svnet_gemm_params fp_linear(const float* A, long lda, long M, int K, const float* W, int ldw, int N, const float* bn_a,
                            const float* bn_c, int act, float* C, long ldc)
{
    svnet_gemm_params g = {};
    g.A = A; g.lda_g = lda; g.lda_x = 0; g.G = 1;
    g.W = W; g.ldw = ldw; g.M = M; g.N = N; g.K = K;
    g.bn_a = bn_a; g.bn_c = bn_c; g.act = act;
    g.C = C; g.ldc_g = ldc; g.ldc_x = 0; g.groups_per_cloud = 1;
    return g;
}

// the five linears of the head, in call order: per-cloud term, conv8 (per point), conv9, conv10, conv11
void fp_linears(const svnet_seg_head_fp_params* p, const float* u, float* cterm, float* hA, float* hB, svnet_gemm_params g[5])
{
    const long R = (long)p->B * p->N;
    const int Kp = p->sv.Cs + 3 * p->sv.Cv, K8 = p->Kc + Kp;
    g[0] = fp_linear(p->glob, p->ldg, p->B, p->Kc, p->W8, K8, p->C8, nullptr, nullptr, SVNET_ACT_NONE, cterm, p->C8);
    g[1] = fp_linear(u, Kp, R, Kp, p->W8 ? p->W8 + p->Kc : nullptr, K8, p->C8, p->bn8_a, p->bn8_c, SVNET_ACT_LEAKY, hA, p->C8);
    g[2] = fp_linear(hA, p->C8, R, p->C8, p->W9, p->C8, p->C9, p->bn9_a, p->bn9_c, SVNET_ACT_LEAKY, hB, p->C9);
    g[3] = fp_linear(hB, p->C9, R, p->C9, p->W10, p->C9, p->C10, p->bn10_a, p->bn10_c, SVNET_ACT_LEAKY, hA, p->C10);
    g[4] = fp_linear(hA, p->C10, R, p->C10, p->W11, p->C10, p->parts, nullptr, nullptr, SVNET_ACT_NONE, hB, p->parts);
}

// false: the per-point conv8 (the only linear with the per-cloud addend) is not covered by the tensor-core linear
bool make_fp_plan(const svnet_seg_head_fp_params* p, seg_fp_plan* pl)
{
    const long R = (long)p->B * p->N;
    const int Kp = p->sv.Cs + 3 * p->sv.Cv;
    const int hAc = p->C8 > p->C10 ? p->C8 : p->C10;
    const int hBc = p->C9 > p->parts ? p->C9 : p->parts;
    size_t o = 0;
    pl->u = o; o += a256((size_t)R * Kp * 4);
    pl->cterm = o; o += a256((size_t)p->B * p->C8 * 4);
    pl->hA = o; o += a256((size_t)R * hAc * 4);
    pl->hB = o; o += a256((size_t)R * hBc * 4);
    svnet_gemm_params g[5];
    fp_linears(p, nullptr, nullptr, nullptr, nullptr, g);
    size_t lb = 0;
    for (int i = 0; i < 5; ++i) {
        const size_t b = svnet_linear_workspace_bytes(&g[i]);
        lb = b > lb ? b : lb;
    }
    pl->lws_bytes = lb;
    pl->lws = o; o += a256(lb);
    pl->total = o;
    return svnet_linear_workspace_bytes(&g[1]) > 0;
}

}  // namespace

extern "C" size_t svnet_seg_head_fp_workspace_bytes(const svnet_seg_head_fp_params* p)
{
    if (!p || p->B < 1 || p->N < 1 || p->Kc < 1 || p->C8 < 1 || p->C9 < 1 || p->C10 < 1 || p->parts < 1) return 0;
    seg_fp_plan pl;
    return make_fp_plan(p, &pl) ? pl.total : 0;
}

extern "C" int svnet_seg_head_fp_fwd(const svnet_seg_head_fp_params* p, void* workspace, size_t workspace_bytes, void* stream)
{
    SV_REQUIRE(p && p->logits && p->glob && p->sv.s && p->sv.v && p->Wz1 && p->W8 && p->bn8_a && p->bn8_c && p->W9 && p->bn9_a &&
                   p->bn9_c && p->W10 && p->bn10_a && p->bn10_c && p->W11,
               "svnet_seg_head_fp_fwd: null pointer");
    SV_REQUIRE(p->B >= 0 && p->N >= 1 && p->Kc >= 1 && p->ldg >= p->Kc && p->sv.Cs >= 1 && p->sv.Cv >= 1 && p->C8 >= 1 && p->C9 >= 1 &&
                   p->C10 >= 1 && p->parts >= 1,
               "svnet_seg_head_fp_fwd: bad shape");
    if (p->B == 0) return SVNET_OK;
    seg_fp_plan pl;
    SV_REQUIRE(make_fp_plan(p, &pl), "svnet_seg_head_fp_fwd: conv8's per-point linear is not covered by the tensor-core linear (svnet_linear_workspace_bytes)");
    SV_REQUIRE(workspace && workspace_bytes >= pl.total && !(reinterpret_cast<uintptr_t>(workspace) & 15),
               "svnet_seg_head_fp_fwd: workspace too small (svnet_seg_head_fp_workspace_bytes) or misaligned");
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    cudaStream_t st = sv_stream(stream);
    const int Kp = p->sv.Cs + 3 * p->sv.Cv;
    float* u = reinterpret_cast<float*>(ws + pl.u);
    float* cterm = reinterpret_cast<float*>(ws + pl.cterm);
    float* hA = reinterpret_cast<float*>(ws + pl.hA);
    float* hB = reinterpret_cast<float*>(ws + pl.hB);
    void* lws = ws + pl.lws;
    // svfuse1: u = [s | v2s(v)] per point
    int rc = svnet_rows_prep(&p->sv, (long)p->B * p->N, p->Wz1, nullptr, nullptr, nullptr, u, Kp, nullptr, nullptr, nullptr, nullptr, stream);
    if (rc != SVNET_OK) return rc;
    svnet_gemm_params g[5];
    fp_linears(p, u, cterm, hA, hB, g);
    for (int i = 0; i < 5; ++i) {
        if (i == 1) {
            // conv8 adds the per-cloud term g[0] wrote (row r of the point table belongs to cloud r / N)
            rc = svnet_linear_tc3_rowadd(&g[i], cterm, p->N, p->C8, lws, pl.lws_bytes, st);
            if (rc < 0) return rc;
            SV_REQUIRE(rc == 1, "svnet_seg_head_fp_fwd: conv8's tensor-core linear not taken");
        } else {
            // as the layer-by-layer path: the tensor-core linear where its workspace query covers the layer
            const size_t b = svnet_linear_workspace_bytes(&g[i]);
            rc = svnet_linear_rows_ws(&g[i], b ? lws : nullptr, b, stream);
            if (rc != SVNET_OK) return rc;
        }
    }
    seg_transpose_kernel<<<dim3(sv_cdiv(p->N, 32), sv_cdiv(p->parts, 32), p->B), 256, 0, st>>>(hB, p->parts, p->N, p->logits);
    SV_CHECK_LAUNCH("svnet_seg_head_fp_fwd(transpose)");
    return SVNET_OK;
}
