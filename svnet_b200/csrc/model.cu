// Whole-model C entry (SURVEY 8(b): svnet_model_create / _forward / _destroy): the SV-DGCNN classifier, binary or full precision,
// (reference models/sv_dgcnn_cls.py:22-82) from a checkpoint's state_dict tensors to logits, without Python in the loop.
//   create  : copies the tensors it needs, packs them once (sign bit-planes, folded BatchNorm affines, fp8 operand bytes of
//             the tensor-core edge kernel, per-point table weights) -- the handle owns everything it uses afterwards;
//   forward : sequences this library's own entry points with caller-owned scratch (svnet_model_workspace_bytes): no
//             allocation, no host synchronisation -- capturable into a CUDA graph.  Launch structure as the Python path's: a
//             batch of >= 32 768 points runs as two to four sub-batches (>= 16 384 points each) on the handle's streams, and inside each the chains that
//             do not depend on the kNN graph or the gate (per-point tables, conv5's scalar branch) run on an auxiliary
//             stream; everything forks from and joins the caller's stream through events (SVNET_MODEL_ONE_STREAM=1: no split);
//             layer 1      svnet_knn_ws -> svnet_gate_xyz -> svnet_edge_xyz_fwd                    (sv_dgcnn_cls.py:48-53)
//             layers 2..4  svnet_linear_rows (float4 table) -> svnet_knn_ws -> svnet_gate_edge -> svnet_svblock_edge_fwd (:55-65)
//             conv5        svnet_gate_rows -> svnet_rows_prep -> svnet_binlinear_pool_ws -> svnet_linear_rows (vector branch) (:67-68)
//             svfuse+pool  svnet_svfuse_pool                                                      (:69-74)
//             head         svnet_head_fwd                                                         (:76-80)
//   The same calls, with the same arguments, as svnet_b200/sv_dgcnn_cls.py + fused.py make through ctypes: the logits are
//   bit-identical to the nn.Module path (tests/test_gpu_parity.py::test_model_c_entry_equals_module).
// Covered: k = 20 (binary also 40: the shapes of the tensor-core edge kernels), 64 <= N <= 4096.  The list of calls above is
// the binary model's; the full-precision model takes svnet_linear_rows_ws where the binary one takes the sign-word kernels
// (sv_dgcnn_cls.py in this package shows both).
// The part-segmentation model (svnet_model_forward_seg, binary or full precision, k = 20 or 40) follows below; its
// full-precision head is svnet_seg_head_fp_fwd (conv8's per-cloud part once per cloud).
#include "common.cuh"
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>

struct svnet_model {
    int k, ncls, binary;
    int pseg;                        // 0: SV_DGCNN_CLS, 1: SV_DGCNN_PSEG (ncls = parts)
    std::vector<void*> allocs;
    // init_scalar + five SVBlocks
    float* Winit;
    struct Block {
        int Cs, Cv, Cout, Cvo, H;      // Cs / Cv: per-point input dims (edge layers: half of the block's in_dims)
        float *G1, *G2, *Wz, *zscale, *W1, *beta, *scale1, *bn1_a, *bn1_c, *W2, *scale2, *bn2_a, *bn2_c;
        uint32_t* W1b;
        unsigned char* W1tc;
        float *Wt, *cst, *Wab;        // Wab: [W1a; W1b] (2 Cout x Cs) of a full-precision linear1 (the Ya | Yb table)
        int NC;
    } conv[6];
    float *fuse_Wz, *fuse_zs;
    // head
    uint32_t *h1_bits, *h2_bits;
    float *h1_beta, *h1_scale, *h1_a, *h1_c, *h2_beta, *h2_scale, *h2_a, *h2_c, *h3_W, *h3_b;
    float *h1_W, *h2_W;              // full-precision head
    // part segmentation: svfuse1 / 2 / 3, conv7 (labels), conv8 .. conv11
    float *f1_Wz, *f1_zs, *f2_Wz, *f2_zs, *f3_Wz, *f3_zs, *c7_W, *c7_a, *c7_c;
    struct SegConv { float *beta, *scale, *bn_a, *bn_c; uint32_t *bits, *bits_c; float* W; int Cin, Cout; } c8, c9, c10;   // W: fp
    float* c11_W;
    int C6s, C6v, Kc;
    // launch structure of svnet_model_forward: two sub-batch streams, each with an auxiliary stream for the chains that do
    // not depend on the kNN graph (per-point tables, conv5's scalar branch); events for the forks / joins
    cudaStream_t sub[4], aux[4];
    cudaEvent_t ev[13];
    bool streams_ok;
    int Cf, C5s, C5v, h1, h2;
};

namespace {

__global__ void sign_kernel(const float* __restrict__ in, long n, float* __restrict__ out)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { const float w = in[i]; out[i] = w > 0.0f ? 1.0f : (w < 0.0f ? -1.0f : 0.0f); }
}
__global__ void eye_ones_kernel(float* __restrict__ eye, int n, float* __restrict__ ones)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n * n) eye[i] = (i / n == i % n) ? 1.0f : 0.0f;
    if (i < n) ones[i] = 1.0f;
}
// (B, 3, N) -> (B*N, 3)
__global__ void xyz_rows_kernel(const float* __restrict__ x, int B, int N, float* __restrict__ out)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long)B * N) return;
    const long b = i / N, n = i - b * N;
    const float* p = x + b * 3 * N + n;
    out[3 * i] = p[0]; out[3 * i + 1] = p[N]; out[3 * i + 2] = p[2L * N];
}

struct Loader {
    const svnet_tensor* t;
    int n;
    svnet_model* m;
    cudaStream_t st;
    bool ok = true;
    std::string err;
    const svnet_tensor* find(const std::string& name, long numel)
    {
        for (int i = 0; i < n; ++i)
            if (name == t[i].name) {
                if (t[i].numel != numel || !t[i].data) { fail(name + ": wrong size"); return nullptr; }
                return t + i;
            }
        fail(name + ": missing from the state_dict");
        return nullptr;
    }
    void fail(const std::string& e) { if (ok) { ok = false; err = e; } }
    void* alloc(size_t bytes)
    {
        void* p = nullptr;
        if (cudaMalloc(&p, bytes ? bytes : 16) != cudaSuccess) { fail("cudaMalloc failed"); return nullptr; }
        m->allocs.push_back(p);
        return p;
    }
    float* dup(const std::string& name, long numel)
    {
        const svnet_tensor* s = find(name, numel);
        float* d = static_cast<float*>(alloc(sizeof(float) * numel));
        if (s && d && cudaMemcpyAsync(d, s->data, sizeof(float) * numel, cudaMemcpyDeviceToDevice, st) != cudaSuccess) fail("copy failed");
        return d;
    }
    float* signed_copy(const std::string& name, long numel)
    {
        const svnet_tensor* s = find(name, numel);
        float* d = static_cast<float*>(alloc(sizeof(float) * numel));
        if (s && d) sign_kernel<<<sv_cdiv(numel, 256), 256, 0, st>>>(s->data, numel, d);
        return d;
    }
    void fold(const std::string& bn, int C, float** a, float** c)
    {
        const svnet_tensor *w = find(bn + ".weight", C), *b = find(bn + ".bias", C), *mu = find(bn + ".running_mean", C),
                           *var = find(bn + ".running_var", C);
        *a = static_cast<float*>(alloc(sizeof(float) * C));
        *c = static_cast<float*>(alloc(sizeof(float) * C));
        if (w && b && mu && var && *a && *c && svnet_fold_bn(w->data, b->data, mu->data, var->data, 1e-5f, C, *a, *c, st) != SVNET_OK)
            fail("svnet_fold_bn failed");
    }
    // sign bit-planes [ceil(K/32)][rows]; the zero weights of call i are counted into zc[i] (device; svnet_pack_sign
    // resets its counter)
    int nz = 0;
    uint32_t* bits(const float* W, int rows, int K, int* zc)
    {
        uint32_t* d = static_cast<uint32_t*>(alloc(sizeof(uint32_t) * (size_t)((K + 31) / 32) * rows));
        if (W && d && nz < 16 && svnet_pack_sign(W, rows, K, K, d, zc + nz, st) != SVNET_OK) fail("svnet_pack_sign failed");
        ++nz;
        return d;
    }
};

inline size_t up256(size_t x) { return (x + 255) & ~(size_t)255; }

struct fwd_plan {
    size_t xyz, idx, s_cat, v_cat, gate, table, knn, v5, g, bits, mask, nvalid, blp, fuse, s5, yab, u5, lin, h1, total;
    size_t knn_bytes, blp_bytes, bl_bytes, fuse_bytes, lin_bytes;
    int Cs_cat, Cv_cat;
};

// scratch of the four edge layers; returns the running offset
size_t plan_trunk(const svnet_model* m, int B, int N, fwd_plan* pl)
{
    const long R = (long)B * N;
    int cs = 0, cv = 0, ncmax = 0, cvomax = 0;
    for (int l = 0; l < 4; ++l) { cs += m->conv[l].Cout; cv += m->conv[l].Cvo; }
    for (int l = 1; l < 4; ++l) ncmax = m->conv[l].NC > ncmax ? m->conv[l].NC : ncmax;
    for (int l = 0; l < 6; ++l) cvomax = m->conv[l].Cvo > cvomax ? m->conv[l].Cvo : cvomax;
    pl->Cs_cat = cs; pl->Cv_cat = cv;
    size_t o = 0;
    pl->xyz = o; o += up256(sizeof(float) * 3 * R);
    pl->idx = o; o += up256(sizeof(int32_t) * R * m->k);
    pl->s_cat = o; o += up256(sizeof(float) * R * cs);
    pl->v_cat = o; o += up256(sizeof(float) * R * 3 * cv);
    pl->gate = o; o += up256(sizeof(float) * B * cvomax);
    pl->table = o; o += up256(sizeof(float) * R * ncmax * 4);
    // kNN scratch: the largest of the four layers
    size_t kb = 0;
    {
        svnet_view v = {};
        v.Cs = 3;
        kb = svnet_knn_workspace_bytes(&v, B, N, m->k);
        for (int l = 1; l < 4; ++l) {
            v.Cs = m->conv[l - 1].Cout; v.Cv = m->conv[l - 1].Cvo;
            const size_t b = svnet_knn_workspace_bytes(&v, B, N, m->k);
            kb = b > kb ? b : kb;
        }
    }
    pl->knn_bytes = kb;
    pl->knn = o; o += up256(kb);
    return o;
}

// the largest scratch of the plain fp linear (rows x K -> Nc) and `lb`
size_t max_lin(size_t lb, long rows, int K, int Nc)
{
    svnet_gemm_params q = {};
    q.G = 1; q.M = rows; q.N = Nc; q.K = K;
    const size_t b = svnet_linear_workspace_bytes(&q);
    return b > lb ? b : lb;
}

// full precision, classifier and part segmentation: the Ya | Yb table of the edge layers, conv5's u = [s | v2s(v)] rows and its
// scalar output; returns the running offset, *lb = the largest scratch of those linears (Ya | Yb and conv5, one at a time)
size_t plan_fp_rows(const svnet_model* m, long R, int K5, fwd_plan* pl, size_t o, size_t* lb)
{
    pl->yab = o; o += up256(sizeof(float) * R * 2 * m->conv[3].Cout);
    pl->u5 = o; o += up256(sizeof(float) * R * K5);
    pl->s5 = o; o += up256(sizeof(float) * R * m->C5s);
    size_t b = max_lin(0, R, K5, m->C5s);
    for (int l = 1; l < 4; ++l) b = max_lin(b, R, m->conv[l].Cs, 2 * m->conv[l].Cout);
    *lb = b;
    return o;
}

bool make_fwd_plan(const svnet_model* m, int B, int N, fwd_plan* pl)
{
    const long R = (long)B * N;
    size_t o = plan_trunk(m, B, N, pl);
    const int cs = pl->Cs_cat, cv = pl->Cv_cat;
    const size_t kb = pl->knn_bytes;
    pl->v5 = o; o += up256(sizeof(float) * R * 3 * m->C5v);
    pl->g = o; o += up256(sizeof(float) * B * 2 * m->Cf);
    const int K5 = cs + 3 * cv, Kw = (K5 + 31) / 32;
    pl->bits = o; o += up256(sizeof(uint32_t) * R * Kw);
    pl->mask = o; o += up256(sizeof(uint32_t) * R * Kw);
    pl->nvalid = o; o += up256(sizeof(int32_t) * R);
    if (!m->binary) {
        // full precision: Ya | Yb table of the edge layers, conv5's u = [s | v2s(v)] rows and scalar output, head layer 1
        pl->bits = pl->mask = pl->nvalid = pl->blp = 0;
        pl->blp_bytes = pl->bl_bytes = 0;
        size_t lb;
        o = plan_fp_rows(m, R, K5, pl, o, &lb);
        pl->h1 = o; o += up256(sizeof(float) * B * m->h1);
        lb = max_lin(lb, B, 2 * m->Cf, m->h1);
        pl->lin_bytes = lb;
        pl->lin = o; o += up256(lb);
        pl->fuse_bytes = svnet_svfuse_pool_workspace(B, m->C5v, N);
        pl->fuse = o; o += up256(pl->fuse_bytes);
        pl->total = o;
        return kb > 0;
    }
    pl->lin_bytes = 0;
    pl->blp_bytes = svnet_binlinear_pool_workspace_bytes(R, K5, m->C5s, N);
    pl->bl_bytes = pl->blp_bytes ? 0 : svnet_binlinear_workspace_bytes(R, K5, m->C5s);
    pl->blp = o; o += up256(pl->blp_bytes + pl->bl_bytes);
    // few rows: conv5's scalar output is materialised and pooled (svnet_binlinear_rows_ws + svnet_pool_rows)
    pl->s5 = o; o += pl->blp_bytes ? 0 : up256(sizeof(float) * R * m->C5s);
    pl->fuse_bytes = svnet_svfuse_pool_workspace(B, m->C5v, N);
    pl->fuse = o; o += up256(pl->fuse_bytes);
    pl->total = o;
    return kb > 0;
}

}  // namespace

extern "C" void svnet_model_destroy(svnet_model* m)
{
    if (!m) return;
    if (m->streams_ok) {
        for (int i = 0; i < 4; ++i) { cudaStreamDestroy(m->sub[i]); cudaStreamDestroy(m->aux[i]); }
        for (int i = 0; i < 13; ++i) cudaEventDestroy(m->ev[i]);
    }
    for (void* p : m->allocs) cudaFree(p);
    delete m;
}

extern "C" int svnet_model_create(const char* kind, int k, int binary, int num_class, const svnet_tensor* tensors, int n_tensors,
                                  void* stream, svnet_model** out)
{
    SV_REQUIRE(kind && tensors && out && n_tensors > 0, "svnet_model_create: null pointer");
    const bool pseg = strcmp(kind, "SV_DGCNN_PSEG") == 0;
    SV_REQUIRE(pseg || strcmp(kind, "SV_DGCNN_CLS") == 0,
               "svnet_model_create: kind '%s' not covered (SV_DGCNN_CLS, SV_DGCNN_PSEG; the PointNet models go through the nn.Module API)", kind);
    SV_REQUIRE(binary == 0 || binary == 1, "svnet_model_create: binary must be 0 or 1");
    SV_REQUIRE(k == 20 || (k == 40 && (binary || pseg)),
               "svnet_model_create: k = %d not covered (the tensor-core edge kernels' shapes: 20; binary and part segmentation also 40)", k);
    SV_REQUIRE(num_class >= 1, "svnet_model_create: bad num_class");
    svnet_model* m = new svnet_model();
    m->k = k; m->ncls = num_class; m->binary = binary; m->pseg = pseg ? 1 : 0;
    Loader L{tensors, n_tensors, m, sv_stream(stream)};
    int* zc = static_cast<int*>(L.alloc(16 * sizeof(int)));
    if (zc) cudaMemsetAsync(zc, 0, 16 * sizeof(int), L.st);
    m->Winit = L.dup("init_scalar.linear.weight", 3 * 2);
    // per-point dims entering each block / leaving it (sv_dgcnn_cls.py:29-34)
    // (sv_dgcnn_partseg.py:52-64: channel counts rounded to multiples of 8; conv6 takes conv5's pooled output, one row per cloud)
    const int cls_cs_in[6] = {3, 32, 32, 64, 256, 0}, cls_cv_in[6] = {1, 10, 10, 21, 83, 0};
    const int cls_cs_out[6] = {32, 32, 64, 128, 512, 0}, cls_cv_out[6] = {10, 10, 21, 42, 170, 0};
    const int seg_cs_in[6] = {3, 32, 32, 64, 256, 512}, seg_cv_in[6] = {1, 16, 16, 24, 96, 168};
    const int seg_cs_out[6] = {32, 32, 64, 128, 512, 256}, seg_cv_out[6] = {16, 16, 24, 40, 168, 88};
    const int* cs_in = pseg ? seg_cs_in : cls_cs_in;
    const int* cv_in = pseg ? seg_cv_in : cls_cv_in;
    const int* cs_out = pseg ? seg_cs_out : cls_cs_out;
    const int* cv_out = pseg ? seg_cv_out : cls_cv_out;
    const int nblocks = pseg ? 6 : 5;
    for (int l = 0; l < nblocks && L.ok; ++l) {
        svnet_model::Block& b = m->conv[l];
        const std::string p = "conv" + std::to_string(l + 1) + ".";
        b = svnet_model::Block();
        b.Cs = cs_in[l]; b.Cv = cv_in[l]; b.Cout = cs_out[l]; b.Cvo = cv_out[l]; b.H = b.Cvo / 2;
        // the block's own input dims: layer 1 (6, 2) full precision; edge layers (2Cs, 2Cv); conv5 (Cs, Cv)
        const int bcs = l == 0 ? 6 : (l < 4 ? 2 * b.Cs : b.Cs), bcv = l == 0 ? 2 : (l < 4 ? 2 * b.Cv : b.Cv);      // l >= 4: row blocks
        const int K1 = bcs + 3 * bcv;
        b.G1 = L.dup(p + "gate.0.weight", (long)b.H * bcs);
        b.G2 = L.dup(p + "gate.2.weight", (long)b.Cvo * b.H);
        L.fold(p + "bn1", b.Cout, &b.bn1_a, &b.bn1_c);
        L.fold(p + "bn2.bn", b.Cvo, &b.bn2_a, &b.bn2_c);
        b.W1 = L.dup(p + "linear1.weight", (long)b.Cout * K1);
        b.W2 = L.dup(p + "linear2.weight", (long)b.Cvo * bcv);
        if (l == 0) {
            b.Wz = L.dup(p + "v2s.linear.weight", 3 * bcv);
            continue;
        }
        if (!binary) {
            // full precision: raw weights; edge layers: three bf16 planes of linear1's q columns, [W1a; W1b] for the Ya | Yb
            // table, table weights without column scales
            b.Wz = L.dup(p + "v2s.linear.weight", 3 * bcv);
            if (l < 4) {
                const size_t wb = svnet_edge_fp_tc_weight_bytes(b.Cs, b.Cv, b.Cout, b.Cvo, k);
                if (wb == 0) { L.fail(p + ": shape not covered by the full-precision tensor-core edge kernel"); break; }
                b.W1tc = static_cast<unsigned char*>(L.alloc(wb));
                if (b.W1tc && svnet_edge_fp_tc_pack_w(b.W1, K1, b.Cs, b.Cv, b.Cout, b.W1tc, stream) != SVNET_OK) L.fail("svnet_edge_fp_tc_pack_w failed");
                const int cs = b.Cs, cv = b.Cv;
                b.Wab = static_cast<float*>(L.alloc(sizeof(float) * (size_t)2 * b.Cout * cs));
                b.NC = 2 * b.Cvo + 6 + cv;
                b.Wt = static_cast<float*>(L.alloc(sizeof(float) * (size_t)b.NC * cv));
                float* scratch_ones = static_cast<float*>(L.alloc(sizeof(float) * cv));
                if (b.Wab && b.Wt && scratch_ones && L.ok) {
                    cudaMemcpy2DAsync(b.Wab, sizeof(float) * cs, b.W1, sizeof(float) * K1, sizeof(float) * cs, b.Cout, cudaMemcpyDeviceToDevice, L.st);
                    cudaMemcpy2DAsync(b.Wab + (size_t)b.Cout * cs, sizeof(float) * cs, b.W1 + cs, sizeof(float) * K1, sizeof(float) * cs, b.Cout,
                                      cudaMemcpyDeviceToDevice, L.st);
                    const size_t w = sizeof(float) * cv;
                    cudaMemcpy2DAsync(b.Wt, w, b.W2, sizeof(float) * bcv, w, b.Cvo, cudaMemcpyDeviceToDevice, L.st);
                    cudaMemcpy2DAsync(b.Wt + (size_t)b.Cvo * cv, w, b.W2 + cv, sizeof(float) * bcv, w, b.Cvo, cudaMemcpyDeviceToDevice, L.st);
                    cudaMemcpy2DAsync(b.Wt + (size_t)2 * b.Cvo * cv, w, b.Wz, sizeof(float) * bcv, w, 3, cudaMemcpyDeviceToDevice, L.st);
                    cudaMemcpy2DAsync(b.Wt + (size_t)(2 * b.Cvo + 3) * cv, w, b.Wz + cv, sizeof(float) * bcv, w, 3, cudaMemcpyDeviceToDevice, L.st);
                    eye_ones_kernel<<<sv_cdiv(cv * cv, 256), 256, 0, L.st>>>(b.Wt + (size_t)(2 * b.Cvo + 6) * cv, cv, scratch_ones);
                }
            }
            continue;
        }
        b.Wz = L.signed_copy(p + "v2s.linear.weight", 3 * bcv);
        b.zscale = L.dup(p + "v2s.linear.scale", 3);
        b.beta = L.dup(p + "linear1.beta", K1);
        b.scale1 = L.dup(p + "linear1.scale", b.Cout);
        b.scale2 = L.dup(p + "linear2.scale", b.Cvo);
        b.W1b = L.bits(b.W1, b.Cout, K1, zc);
        if (l < 4) {
            const size_t wb = svnet_edge_tc_weight_bytes(b.Cs, b.Cv, b.Cout, b.Cvo, k);
            if (wb == 0) { L.fail(p + ": shape not covered by the tensor-core edge kernel"); break; }
            b.W1tc = static_cast<unsigned char*>(L.alloc(wb));
            if (b.W1tc && svnet_edge_tc_pack_w(b.W1, K1, b.Cs, b.Cv, b.Cout, b.W1tc, stream) != SVNET_OK) L.fail("svnet_edge_tc_pack_w failed");
            // table weights [W2a | W2b | Wz_a | Wz_b | I] (rows) over the Cv input channels, and their column scales
            const int cv = b.Cv;
            b.NC = 2 * b.Cvo + 6 + cv;
            b.Wt = static_cast<float*>(L.alloc(sizeof(float) * (size_t)b.NC * cv));
            b.cst = static_cast<float*>(L.alloc(sizeof(float) * b.NC));
            const svnet_tensor* wz = L.find(p + "v2s.linear.weight", 3 * bcv);
            if (b.Wt && b.cst && wz && L.ok) {
                const size_t w = sizeof(float) * cv;
                cudaMemcpy2DAsync(b.Wt, w, b.W2, sizeof(float) * bcv, w, b.Cvo, cudaMemcpyDeviceToDevice, L.st);
                cudaMemcpy2DAsync(b.Wt + (size_t)b.Cvo * cv, w, b.W2 + cv, sizeof(float) * bcv, w, b.Cvo, cudaMemcpyDeviceToDevice, L.st);
                cudaMemcpy2DAsync(b.Wt + (size_t)2 * b.Cvo * cv, w, wz->data, sizeof(float) * bcv, w, 3, cudaMemcpyDeviceToDevice, L.st);
                cudaMemcpy2DAsync(b.Wt + (size_t)(2 * b.Cvo + 3) * cv, w, wz->data + cv, sizeof(float) * bcv, w, 3, cudaMemcpyDeviceToDevice, L.st);
                eye_ones_kernel<<<sv_cdiv(cv * cv, 256), 256, 0, L.st>>>(b.Wt + (size_t)(2 * b.Cvo + 6) * cv, cv, b.cst + 2 * b.Cvo + 6);
                cudaMemcpyAsync(b.cst, b.scale2, sizeof(float) * b.Cvo, cudaMemcpyDeviceToDevice, L.st);
                cudaMemcpyAsync(b.cst + b.Cvo, b.scale2, sizeof(float) * b.Cvo, cudaMemcpyDeviceToDevice, L.st);
                cudaMemcpyAsync(b.cst + 2 * b.Cvo, b.zscale, sizeof(float) * 3, cudaMemcpyDeviceToDevice, L.st);
                cudaMemcpyAsync(b.cst + 2 * b.Cvo + 3, b.zscale, sizeof(float) * 3, cudaMemcpyDeviceToDevice, L.st);
            }
        }
    }
    m->C5s = cs_out[4]; m->C5v = cv_out[4]; m->Cf = m->C5s + 3 * m->C5v;
    m->h1 = 512; m->h2 = 256;
    if (L.ok && pseg) {
        m->C6s = cs_out[5]; m->C6v = cv_out[5];
        const int cs_cat = 256, cv_cat = 96;
        if (binary) {
            m->f1_Wz = L.signed_copy("svfuse1.v2s.linear.weight", 3 * cv_cat);
            m->f1_zs = L.dup("svfuse1.v2s.linear.scale", 3);
            m->f2_Wz = L.signed_copy("svfuse2.v2s.linear.weight", 3 * m->C6v);
            m->f2_zs = L.dup("svfuse2.v2s.linear.scale", 3);
            m->f3_Wz = L.signed_copy("svfuse3.v2s.linear.weight", 3 * m->C5v);
            m->f3_zs = L.dup("svfuse3.v2s.linear.scale", 3);
        } else {      // full precision: plain v2s weights, no scales (zscale = NULL below)
            m->f1_Wz = L.dup("svfuse1.v2s.linear.weight", 3 * cv_cat);
            m->f2_Wz = L.dup("svfuse2.v2s.linear.weight", 3 * m->C6v);
            m->f3_Wz = L.dup("svfuse3.v2s.linear.weight", 3 * m->C5v);
        }
        m->c7_W = L.dup("conv7.0.weight", 64 * 16);
        L.fold("conv7.1", 64, &m->c7_a, &m->c7_c);
        // conv8 input = [glob (per cloud): s5 max | v2s(v5) max | svfuse2(conv6) | conv7(label)] ++ [svfuse1(s_cat, v_cat) per point]
        m->Kc = m->C5s + 3 * m->C5v + (m->C6s + 3 * m->C6v) + 64;
        const int Kp = cs_cat + 3 * cv_cat;
        auto seg_conv = [&](const char* name, int Cin, int Cout, svnet_model::SegConv* c, int split) {
            const std::string p = std::string(name) + ".";
            c->Cin = Cin; c->Cout = Cout;
            c->beta = c->scale = c->W = nullptr;
            c->bits = c->bits_c = nullptr;
            if (!binary) {     // full precision: the weight [Cout][Cin] as it is and the folded BN
                c->W = L.dup(p + "0.weight", (long)Cout * Cin);
                L.fold(p + "1", Cout, &c->bn_a, &c->bn_c);
                return;
            }
            const svnet_tensor* w = L.find(p + "0.weight", (long)Cout * Cin);
            c->beta = L.dup(p + "0.beta", Cin);
            c->scale = L.dup(p + "0.scale", Cout);
            L.fold(p + "1", Cout, &c->bn_a, &c->bn_c);
            if (!w) return;
            if (split > 0) {
                // sign planes of the per-cloud columns [:, :split] and of the per-point columns [:, split:]
                c->bits_c = static_cast<uint32_t*>(L.alloc(sizeof(uint32_t) * (size_t)((split + 31) / 32) * Cout));
                c->bits = static_cast<uint32_t*>(L.alloc(sizeof(uint32_t) * (size_t)((Cin - split + 31) / 32) * Cout));
                if (c->bits_c && c->bits && L.nz + 2 <= 16) {
                    if (svnet_pack_sign(w->data, Cout, split, Cin, c->bits_c, zc + L.nz, L.st) != SVNET_OK) L.fail("svnet_pack_sign failed");
                    if (svnet_pack_sign(w->data + split, Cout, Cin - split, Cin, c->bits, zc + L.nz + 1, L.st) != SVNET_OK) L.fail("svnet_pack_sign failed");
                }
                L.nz += 2;
            } else {
                c->bits = L.bits(w->data, Cout, Cin, zc);
            }
        };
        seg_conv("conv8", m->Kc + Kp, 256, &m->c8, m->Kc);
        seg_conv("conv9", 256, 256, &m->c9, 0);
        seg_conv("conv10", 256, 128, &m->c10, 0);
        m->c11_W = L.dup("conv11.weight", (long)num_class * 128);
    }
    if (L.ok && !pseg && !binary) {
        m->fuse_Wz = L.dup("svfuse.v2s.linear.weight", 3 * m->C5v);
        m->h1_W = L.dup("linear1.weight", (long)m->h1 * 2 * m->Cf);
        m->h2_W = L.dup("linear2.weight", (long)m->h2 * m->h1);
        L.fold("bn1", m->h1, &m->h1_a, &m->h1_c);
        L.fold("bn2", m->h2, &m->h2_a, &m->h2_c);
        m->h3_W = L.dup("linear3.weight", (long)num_class * m->h2);
        m->h3_b = L.dup("linear3.bias", num_class);
    }
    if (L.ok && !pseg && binary) {
        m->fuse_Wz = L.signed_copy("svfuse.v2s.linear.weight", 3 * m->C5v);
        m->fuse_zs = L.dup("svfuse.v2s.linear.scale", 3);
        const svnet_tensor* w1 = L.find("linear1.weight", (long)m->h1 * 2 * m->Cf);
        const svnet_tensor* w2 = L.find("linear2.weight", (long)m->h2 * m->h1);
        m->h1_bits = L.bits(w1 ? w1->data : nullptr, m->h1, 2 * m->Cf, zc);
        m->h2_bits = L.bits(w2 ? w2->data : nullptr, m->h2, m->h1, zc);
        m->h1_beta = L.dup("linear1.beta", 2 * m->Cf);
        m->h1_scale = L.dup("linear1.scale", m->h1);
        m->h2_beta = L.dup("linear2.beta", m->h1);
        m->h2_scale = L.dup("linear2.scale", m->h2);
        L.fold("bn1", m->h1, &m->h1_a, &m->h1_c);
        L.fold("bn2", m->h2, &m->h2_a, &m->h2_c);
        m->h3_W = L.dup("linear3.weight", (long)num_class * m->h2);
        m->h3_b = L.dup("linear3.bias", num_class);
    }
    if (L.ok) {
        int zh[16] = {0};
        int zeros = 0;
        if (cudaMemcpyAsync(zh, zc, sizeof(zh), cudaMemcpyDeviceToHost, L.st) != cudaSuccess || cudaStreamSynchronize(L.st) != cudaSuccess)
            L.fail("CUDA error while packing");
        for (int i = 0; i < 16; ++i) zeros += zh[i];
        if (L.ok && zeros != 0)
            L.fail("a binarised weight contains exact zeros (sign(0) = 0 plane not supported by the popcount kernels)");
    }
    if (!L.ok) {
        svnet_set_error("svnet_model_create: %s", L.err.c_str());
        svnet_model_destroy(m);
        return SVNET_ERR_ARG;
    }
    m->streams_ok = true;
    for (int i = 0; i < 4; ++i) {
        if (cudaStreamCreateWithFlags(&m->sub[i], cudaStreamNonBlocking) != cudaSuccess) m->streams_ok = false;
        if (cudaStreamCreateWithFlags(&m->aux[i], cudaStreamNonBlocking) != cudaSuccess) m->streams_ok = false;
    }
    for (int i = 0; i < 13; ++i)
        if (cudaEventCreateWithFlags(&m->ev[i], cudaEventDisableTiming) != cudaSuccess) m->streams_ok = false;
    *out = m;
    return SVNET_OK;
}

namespace {
// a large enough batch runs as up to four sub-batches of >= 16 384 points on the handle's streams (clouds are independent in
// eval mode, so the bits do not depend on the split); SVNET_MODEL_ONE_STREAM=1 keeps everything on the caller's stream
int split_count(const svnet_model* m, int B, int N)
{
    static const bool off = [] { const char* e = getenv("SVNET_MODEL_ONE_STREAM"); return e && e[0] == '1'; }();
    if (off || !m->streams_ok) return 1;
    static const int forced = [] { const char* e = getenv("SVNET_MODEL_SPLIT"); return e ? atoi(e) : 0; }();   // tuning aid
    if (forced >= 1 && forced <= 4) return forced > B ? B : forced;
    long n = ((long)B * N) / 16384;
    n = n < 1 ? 1 : (n > 4 ? 4 : n);
    return (int)(n > B ? B : n);
}
inline int sub_lo(int B, int n, int i) { return (int)((long)B * i / n); }

}  // namespace

extern "C" size_t svnet_model_workspace_bytes(const svnet_model* m, int B, int N)
{
    if (!m || m->pseg || B < 1 || N < 64 || N > 4096) return 0;
    const int ns = split_count(m, B, N);
    if (ns > 1) {
        size_t tot = 0;
        for (int i = 0; i < ns; ++i) {
            fwd_plan pi;
            if (!make_fwd_plan(m, sub_lo(B, ns, i + 1) - sub_lo(B, ns, i), N, &pi)) return 0;
            tot += pi.total;
        }
        return tot;
    }
    fwd_plan pl;
    if (!make_fwd_plan(m, B, N, &pl)) return 0;
    return pl.total;
}

namespace {

// the four edge layers (sv_dgcnn_cls.py:47-65, sv_dgcnn_partseg.py:81-103): fills the svcat table (s_cat, v_cat) in `ws`
int run_trunk(const svnet_model* m, const float* x, int B, int N, unsigned char* ws, const fwd_plan& pl, void* stream,
              cudaStream_t aux = nullptr, cudaEvent_t eF = nullptr, cudaEvent_t eJ = nullptr)
{
    cudaStream_t st = sv_stream(stream);
    const long R = (long)B * N;
    const int k = m->k;
    float* xyz = reinterpret_cast<float*>(ws + pl.xyz);
    int32_t* idx = reinterpret_cast<int32_t*>(ws + pl.idx);
    float* s_cat = reinterpret_cast<float*>(ws + pl.s_cat);
    float* v_cat = reinterpret_cast<float*>(ws + pl.v_cat);
    float* gate = reinterpret_cast<float*>(ws + pl.gate);
    float* table = reinterpret_cast<float*>(ws + pl.table);
    void* knn_ws = ws + pl.knn;
    const int lds = pl.Cs_cat, xs = pl.Cv_cat, ldv = 3 * pl.Cv_cat;
    int rc;
    xyz_rows_kernel<<<sv_cdiv(R, 256), 256, 0, st>>>(x, B, N, xyz);
    SV_CHECK_LAUNCH("svnet_model_forward(xyz)");
    int so = 0, vo = 0;
    svnet_view prev = {};
    for (int l = 0; l < 4; ++l) {
        const svnet_model::Block& b = m->conv[l];
        svnet_mview out = {};
        out.s = s_cat + so; out.lds = lds; out.Cs = b.Cout;
        out.v = v_cat + vo; out.ldv = ldv; out.xs = xs; out.Cv = b.Cvo;
        if (l == 0) {
            svnet_view xv = {};
            xv.s = xyz; xv.lds = 3; xv.Cs = 3;
            rc = svnet_knn_ws(&xv, B, N, k, idx, nullptr, knn_ws, pl.knn_bytes, stream);
            if (rc != SVNET_OK) return rc;
            rc = svnet_gate_xyz(xyz, idx, B, N, k, 2, m->Winit, b.G1, b.G2, b.H, b.Cvo, gate, stream);
            if (rc != SVNET_OK) return rc;
            svnet_edge_xyz_params p = {};
            p.xyz = xyz; p.idx = idx; p.B = B; p.N = N; p.k = k; p.nv = 2;
            p.Winit = m->Winit; p.Wz = b.Wz; p.W1 = b.W1; p.bn1_a = b.bn1_a; p.bn1_c = b.bn1_c;
            p.W2 = b.W2; p.bn2_a = b.bn2_a; p.bn2_c = b.bn2_c; p.gate = gate; p.Cout = b.Cout; p.Cvo = b.Cvo; p.out = out;
            rc = svnet_edge_xyz_fwd(&p, stream);
            if (rc != SVNET_OK) return rc;
        } else {
            // per-point float4 table [P | Q | T | U | v] of the tensor-core edge kernel
            svnet_gemm_params g = {};
            g.A = prev.v; g.lda_g = prev.ldv; g.lda_x = prev.xs; g.G = 3;
            g.W = b.Wt; g.ldw = b.Cv; g.M = 3 * R; g.N = b.NC; g.K = b.Cv;
            g.sign_w = m->binary; g.colscale = m->binary ? b.cst : nullptr; g.C = table; g.ldc_g = 4 * b.NC; g.ldc_x = 0; g.c4 = 1;
            g.groups_per_cloud = 1;
            // the tables do not depend on the graph: with an auxiliary stream they run next to the kNN kernels
            void* tst = stream;
            if (aux) {
                SV_CUDA(cudaEventRecord(eF, st));
                SV_CUDA(cudaStreamWaitEvent(aux, eF, 0));
                tst = aux;
            }
            rc = svnet_linear_rows_ws(&g, nullptr, 0, tst);
            if (rc != SVNET_OK) return rc;
            float* yab = nullptr;
            if (!m->binary) {
                // Ya | Yb = s [W1a; W1b]^T per point (the s part of linear1)
                yab = reinterpret_cast<float*>(ws + pl.yab);
                svnet_gemm_params y = {};
                y.A = prev.s; y.lda_g = prev.lds; y.lda_x = 0; y.G = 1;
                y.W = b.Wab; y.ldw = b.Cs; y.M = R; y.N = 2 * b.Cout; y.K = b.Cs;
                y.C = yab; y.ldc_g = 2 * b.Cout; y.ldc_x = 0; y.groups_per_cloud = 1;
                const size_t yb = svnet_linear_workspace_bytes(&y);
                rc = svnet_linear_rows_ws(&y, yb ? ws + pl.lin : nullptr, yb, tst);
                if (rc != SVNET_OK) return rc;
            }
            if (aux) SV_CUDA(cudaEventRecord(eJ, aux));
            rc = svnet_knn_ws(&prev, B, N, k, idx, nullptr, knn_ws, pl.knn_bytes, stream);
            if (rc != SVNET_OK) return rc;
            rc = svnet_gate_edge(&prev, idx, B, N, k, b.G1, b.G2, b.H, b.Cvo, gate, stream);
            if (rc != SVNET_OK) return rc;
            svnet_edge_params p = {};
            p.in = prev; p.idx = idx; p.B = B; p.N = N; p.k = k; p.binary = m->binary;
            p.Yab = yab;
            if (aux) SV_CUDA(cudaStreamWaitEvent(st, eJ, 0));
            p.Wz = b.Wz; p.zscale = b.zscale; p.beta = b.beta; p.W1b = b.W1b; p.scale1 = b.scale1;
            p.bn1_a = b.bn1_a; p.bn1_c = b.bn1_c; p.Cout = b.Cout;
            p.bn2_a = b.bn2_a; p.bn2_c = b.bn2_c; p.gate = gate; p.Cvo = b.Cvo; p.out = out;
            p.W1tc = b.W1tc; p.tab4 = table;
            rc = svnet_svblock_edge_fwd(&p, stream);
            if (rc != SVNET_OK) return rc;
        }
        prev.s = out.s; prev.lds = out.lds; prev.Cs = out.Cs;
        prev.v = out.v; prev.ldv = out.ldv; prev.xs = out.xs; prev.Cv = out.Cv;
        so += b.Cout; vo += b.Cvo;
    }
    return SVNET_OK;
}

}  // namespace

namespace {

// one (sub-)batch on stream `stream`; `aux` (optional) takes the chains that do not depend on the kNN graphs / the gate
int forward_cls_one(const svnet_model* m, const float* x, int B, int N, float* logits, unsigned char* ws, const fwd_plan& pl,
                    void* stream, cudaStream_t aux, cudaEvent_t eF, cudaEvent_t eJ)
{
    cudaStream_t st = sv_stream(stream);
    const long R = (long)B * N;
    float* s_cat = reinterpret_cast<float*>(ws + pl.s_cat);
    float* v_cat = reinterpret_cast<float*>(ws + pl.v_cat);
    float* gate = reinterpret_cast<float*>(ws + pl.gate);
    const int lds = pl.Cs_cat, xs = pl.Cv_cat, ldv = 3 * pl.Cv_cat;
    int rc = run_trunk(m, x, B, N, ws, pl, stream, aux, eF, eJ);
    if (rc != SVNET_OK) return rc;
    // ---- conv5 (per point) -> svfuse -> max | mean over the points ----
    // scalar branch (v2s + linear1 + pooling) on `sst` next to gate -> vector linear on the main stream
    void* sst = stream;
    if (aux) {
        SV_CUDA(cudaEventRecord(eF, st));
        SV_CUDA(cudaStreamWaitEvent(aux, eF, 0));
        sst = aux;
    }
    const svnet_model::Block& c5 = m->conv[4];
    float* v5 = reinterpret_cast<float*>(ws + pl.v5);
    float* g = reinterpret_cast<float*>(ws + pl.g);
    uint32_t* bits = reinterpret_cast<uint32_t*>(ws + pl.bits);
    uint32_t* mask = reinterpret_cast<uint32_t*>(ws + pl.mask);
    int32_t* nvalid = reinterpret_cast<int32_t*>(ws + pl.nvalid);
    const int Cf = m->Cf, K5 = pl.Cs_cat + 3 * pl.Cv_cat;
    svnet_view cat = {};
    cat.s = s_cat; cat.lds = lds; cat.Cs = pl.Cs_cat; cat.v = v_cat; cat.ldv = ldv; cat.xs = xs; cat.Cv = pl.Cv_cat;
    if (!m->binary) {
        // u = [s | v2s(v)] rows -> dense linear1 + BN + LeakyReLU -> max | mean over the points
        float* u5 = reinterpret_cast<float*>(ws + pl.u5);
        float* s5 = reinterpret_cast<float*>(ws + pl.s5);
        rc = svnet_rows_prep(&cat, R, c5.Wz, nullptr, nullptr, nullptr, u5, K5, nullptr, nullptr, nullptr, nullptr, sst);
        if (rc != SVNET_OK) return rc;
        svnet_gemm_params q = {};
        q.A = u5; q.lda_g = K5; q.lda_x = 0; q.G = 1; q.W = c5.W1; q.ldw = K5; q.M = R; q.N = c5.Cout; q.K = K5;
        q.bn_a = c5.bn1_a; q.bn_c = c5.bn1_c; q.act = SVNET_ACT_LEAKY; q.C = s5; q.ldc_g = c5.Cout; q.ldc_x = 0; q.groups_per_cloud = 1;
        const size_t qb = svnet_linear_workspace_bytes(&q);
        rc = svnet_linear_rows_ws(&q, qb ? ws + pl.lin : nullptr, qb, sst);
        if (rc != SVNET_OK) return rc;
    } else {
    rc = svnet_rows_prep(&cat, R, c5.Wz, c5.zscale, nullptr, c5.beta, nullptr, 0, nullptr, bits, mask, nvalid, sst);
    if (rc != SVNET_OK) return rc;
    }
    if (!m->binary) {
    } else if (pl.blp_bytes) {
        rc = svnet_binlinear_pool_ws(bits, mask, R, K5, c5.W1b, c5.Cout, c5.scale1, c5.bn1_a, c5.bn1_c, N, g, g + Cf, 2 * Cf,
                                     ws + pl.blp, pl.blp_bytes, sst);
        if (rc != SVNET_OK) return rc;
    } else {
        float* s5 = reinterpret_cast<float*>(ws + pl.s5);
        rc = svnet_binlinear_rows_ws(bits, mask, nvalid, R, K5, c5.W1b, c5.Cout, c5.scale1, nullptr, c5.bn1_a, c5.bn1_c, SVNET_ACT_LEAKY,
                                     nullptr, 1, s5, c5.Cout, nullptr, pl.bl_bytes ? ws + pl.blp : nullptr, pl.bl_bytes, sst);
        if (rc != SVNET_OK) return rc;
        rc = svnet_pool_rows(s5, c5.Cout, c5.Cout, B, N, g, g + Cf, 2 * Cf, sst);
        if (rc != SVNET_OK) return rc;
    }
    if (aux) SV_CUDA(cudaEventRecord(eJ, aux));
    rc = svnet_gate_rows(s_cat, lds, pl.Cs_cat, B, N, c5.G1, c5.G2, c5.H, c5.Cvo, gate, stream);
    if (rc != SVNET_OK) return rc;
    {
        svnet_gemm_params q = {};
        q.A = v_cat; q.lda_g = ldv; q.lda_x = xs; q.G = 3;
        q.W = c5.W2; q.ldw = c5.Cv; q.M = 3 * R; q.N = c5.Cvo; q.K = c5.Cv;
        q.sign_w = m->binary; q.colscale = m->binary ? c5.scale2 : nullptr; q.bn_a = c5.bn2_a; q.bn_c = c5.bn2_c; q.vbn = 1; q.gate = gate;
        q.groups_per_cloud = N;
        q.C = v5; q.ldc_g = 3 * c5.Cvo; q.ldc_x = c5.Cvo;
        rc = svnet_linear_rows_ws(&q, nullptr, 0, stream);
        if (rc != SVNET_OK) return rc;
    }
    if (aux) SV_CUDA(cudaStreamWaitEvent(st, eJ, 0));
    if (!m->binary) {
        rc = svnet_pool_rows(reinterpret_cast<float*>(ws + pl.s5), c5.Cout, c5.Cout, B, N, g, g + Cf, 2 * Cf, stream);
        if (rc != SVNET_OK) return rc;
    }
    svnet_view v5v = {};
    v5v.v = v5; v5v.ldv = 3 * c5.Cvo; v5v.xs = c5.Cvo; v5v.Cv = c5.Cvo;
    rc = svnet_svfuse_pool(&v5v, B, N, m->fuse_Wz, m->binary ? m->fuse_zs : nullptr, g + m->C5s, g + Cf + m->C5s, 2 * Cf, ws + pl.fuse, pl.fuse_bytes, stream);
    if (rc != SVNET_OK) return rc;
    // ---- head ----
    if (!m->binary) {
        // the full-precision first layer (2044 x 512 weights) as one GEMM over the batch, then the fused two-layer head
        float* h1 = reinterpret_cast<float*>(ws + pl.h1);
        svnet_gemm_params q = {};
        q.A = g; q.lda_g = 2 * Cf; q.lda_x = 0; q.G = 1; q.W = m->h1_W; q.ldw = 2 * Cf; q.M = B; q.N = m->h1; q.K = 2 * Cf;
        q.bn_a = m->h1_a; q.bn_c = m->h1_c; q.act = SVNET_ACT_LEAKY; q.C = h1; q.ldc_g = m->h1; q.ldc_x = 0; q.groups_per_cloud = 1;
        const size_t qb = svnet_linear_workspace_bytes(&q);
        rc = svnet_linear_rows_ws(&q, qb ? ws + pl.lin : nullptr, qb, stream);
        if (rc != SVNET_OK) return rc;
        svnet_head_params hf = {};
        hf.x = h1; hf.ldx = m->h1; hf.K0 = m->h1; hf.B = B; hf.nlayers = 2;
        hf.layer[0].Cout = m->h2; hf.layer[0].W = m->h2_W; hf.layer[0].bn_a = m->h2_a; hf.layer[0].bn_c = m->h2_c; hf.layer[0].act = SVNET_ACT_LEAKY;
        hf.layer[1].Cout = m->ncls; hf.layer[1].W = m->h3_W; hf.layer[1].bias = m->h3_b; hf.layer[1].act = SVNET_ACT_NONE;
        hf.out = logits; hf.ldo = m->ncls;
        return svnet_head_fwd(&hf, stream);
    }
    svnet_head_params h = {};
    h.x = g; h.ldx = 2 * Cf; h.K0 = 2 * Cf; h.B = B; h.nlayers = 3;
    h.layer[0].Cout = m->h1; h.layer[0].W1b = m->h1_bits; h.layer[0].beta = m->h1_beta; h.layer[0].scale = m->h1_scale;
    h.layer[0].bn_a = m->h1_a; h.layer[0].bn_c = m->h1_c; h.layer[0].act = SVNET_ACT_LEAKY;
    h.layer[1].Cout = m->h2; h.layer[1].W1b = m->h2_bits; h.layer[1].beta = m->h2_beta; h.layer[1].scale = m->h2_scale;
    h.layer[1].bn_a = m->h2_a; h.layer[1].bn_c = m->h2_c; h.layer[1].act = SVNET_ACT_LEAKY;
    h.layer[2].Cout = m->ncls; h.layer[2].W = m->h3_W; h.layer[2].bias = m->h3_b; h.layer[2].act = SVNET_ACT_NONE;
    h.out = logits; h.ldo = m->ncls;
    return svnet_head_fwd(&h, stream);
}

}  // namespace

extern "C" int svnet_model_forward(const svnet_model* m, const float* x, int B, int N, float* logits, void* workspace,
                                   size_t workspace_bytes, void* stream)
{
    SV_REQUIRE(m && x && logits, "svnet_model_forward: null pointer");
    SV_REQUIRE(!m->pseg, "svnet_model_forward: the handle is a part-segmentation model (svnet_model_forward_seg)");
    SV_REQUIRE(B >= 0 && N >= 64 && N <= 4096, "svnet_model_forward: N = %d not covered (64..4096)", N);
    if (B == 0) return SVNET_OK;
    SV_REQUIRE(workspace && !(reinterpret_cast<uintptr_t>(workspace) & 255), "svnet_model_forward: workspace null or not 256-byte aligned");
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    cudaStream_t st = sv_stream(stream);
    const int ns = split_count(m, B, N);
    if (ns == 1) {
        fwd_plan pl;
        SV_REQUIRE(make_fwd_plan(m, B, N, &pl), "svnet_model_forward: shape not covered by the tensor-core paths");
        SV_REQUIRE(workspace_bytes >= pl.total, "svnet_model_forward: workspace too small (svnet_model_workspace_bytes)");
        const bool ax = m->streams_ok;
        return forward_cls_one(m, x, B, N, logits, ws, pl, stream, ax ? m->aux[0] : nullptr, ax ? m->ev[0] : nullptr, ax ? m->ev[1] : nullptr);
    }
    SV_REQUIRE(workspace_bytes >= svnet_model_workspace_bytes(m, B, N), "svnet_model_forward: workspace too small (svnet_model_workspace_bytes)");
    SV_CUDA(cudaEventRecord(m->ev[8], st));
    size_t off = 0;
    for (int i = 0; i < ns; ++i) {
        const int lo = sub_lo(B, ns, i), Bi = sub_lo(B, ns, i + 1) - lo;
        fwd_plan pi;
        SV_REQUIRE(make_fwd_plan(m, Bi, N, &pi), "svnet_model_forward: shape not covered by the tensor-core paths");
        SV_CUDA(cudaStreamWaitEvent(m->sub[i], m->ev[8], 0));
        const int rc = forward_cls_one(m, x + (size_t)lo * 3 * N, Bi, N, logits + (size_t)lo * m->ncls, ws + off, pi, m->sub[i], m->aux[i],
                                       m->ev[2 * i], m->ev[2 * i + 1]);
        if (rc != SVNET_OK) return rc;
        off += pi.total;
        SV_CUDA(cudaEventRecord(m->ev[9 + i], m->sub[i]));
        SV_CUDA(cudaStreamWaitEvent(st, m->ev[9 + i], 0));
    }
    return SVNET_OK;
}

// ---- part segmentation (sv_dgcnn_partseg.py:80-128) -------------------------------------------------------------------
namespace {

struct seg_plan2 {
    fwd_plan t;
    size_t bits8, mask8, nvalid8, bits5, mask5, nvalid5, blp, s5, v5, glob, vp, v6, bits6, mask6, nvalid6, fuse, head, total;
    size_t u6;            // full precision: conv6's rows u = [s | v2s(v)] (conv5's: t.u5)
    size_t blp_bytes, bl_bytes, fuse_bytes, head_bytes;
};

svnet_seg_head_params seg_head_params(const svnet_model* m, int B, int N)
{
    svnet_seg_head_params h = {};
    h.sv.Cs = 256; h.sv.Cv = 96; h.sv.lds = 256; h.sv.ldv = 3 * 96; h.sv.xs = 96;
    h.B = B; h.N = N; h.Wz1 = m->f1_Wz; h.zscale1 = m->f1_zs; h.ldg = m->Kc; h.Kc = m->Kc;
    h.beta8 = m->c8.beta; h.W8c = m->c8.bits_c; h.W8p = m->c8.bits; h.scale8 = m->c8.scale; h.bn8_a = m->c8.bn_a; h.bn8_c = m->c8.bn_c; h.C8 = m->c8.Cout;
    h.beta9 = m->c9.beta; h.W9 = m->c9.bits; h.scale9 = m->c9.scale; h.bn9_a = m->c9.bn_a; h.bn9_c = m->c9.bn_c; h.C9 = m->c9.Cout;
    h.beta10 = m->c10.beta; h.W10 = m->c10.bits; h.scale10 = m->c10.scale; h.bn10_a = m->c10.bn_a; h.bn10_c = m->c10.bn_c; h.C10 = m->c10.Cout;
    h.W11 = m->c11_W; h.parts = m->ncls;
    return h;
}

svnet_seg_head_fp_params seg_head_fp_params(const svnet_model* m, int B, int N)
{
    svnet_seg_head_fp_params h = {};
    h.sv.Cs = 256; h.sv.Cv = 96; h.sv.lds = 256; h.sv.ldv = 3 * 96; h.sv.xs = 96;
    h.B = B; h.N = N; h.Wz1 = m->f1_Wz; h.ldg = m->Kc; h.Kc = m->Kc;
    h.W8 = m->c8.W; h.bn8_a = m->c8.bn_a; h.bn8_c = m->c8.bn_c; h.C8 = m->c8.Cout;
    h.W9 = m->c9.W; h.bn9_a = m->c9.bn_a; h.bn9_c = m->c9.bn_c; h.C9 = m->c9.Cout;
    h.W10 = m->c10.W; h.bn10_a = m->c10.bn_a; h.bn10_c = m->c10.bn_c; h.C10 = m->c10.Cout;
    h.W11 = m->c11_W; h.parts = m->ncls;
    return h;
}

// full precision: trunk (+ Ya | Yb table), conv5's u rows and scalar output, the global branch, the fp head
bool make_seg_plan_fp(const svnet_model* m, int B, int N, seg_plan2* pl, size_t o)
{
    const long R = (long)B * N;
    const int Kp = pl->t.Cs_cat + 3 * pl->t.Cv_cat, K6 = m->C5s + 3 * m->C5v;
    pl->bits8 = pl->mask8 = pl->nvalid8 = pl->bits5 = pl->mask5 = pl->nvalid5 = pl->blp = pl->s5 = pl->bits6 = pl->mask6 = pl->nvalid6 = 0;
    pl->blp_bytes = pl->bl_bytes = 0;
    size_t lb;
    o = plan_fp_rows(m, R, Kp, &pl->t, o, &lb);
    pl->v5 = o; o += up256(sizeof(float) * R * 3 * m->C5v);
    pl->glob = o; o += up256(sizeof(float) * B * m->Kc);
    pl->vp = o; o += up256(sizeof(float) * B * 3 * m->C5v);
    pl->u6 = o; o += up256(sizeof(float) * B * K6);
    pl->v6 = o; o += up256(sizeof(float) * B * 3 * m->C6v);
    // scratch of the fp linears outside the head (one at a time): plan_fp_rows' and conv6's
    lb = max_lin(lb, B, K6, m->C6s);
    pl->t.lin_bytes = lb;
    pl->t.lin = o; o += up256(lb);
    pl->fuse_bytes = svnet_svfuse_pool_workspace(B, m->C5v, N);
    pl->fuse = o; o += up256(pl->fuse_bytes);
    const svnet_seg_head_fp_params h = seg_head_fp_params(m, B, N);
    pl->head_bytes = svnet_seg_head_fp_workspace_bytes(&h);
    pl->head = o; o += up256(pl->head_bytes);
    pl->total = o;
    return pl->t.knn_bytes > 0 && pl->head_bytes > 0;
}

bool make_seg_plan(const svnet_model* m, int B, int N, seg_plan2* pl)
{
    const long R = (long)B * N;
    size_t o = plan_trunk(m, B, N, &pl->t);
    if (!m->binary) return make_seg_plan_fp(m, B, N, pl, o);
    pl->u6 = 0;
    const int cs = pl->t.Cs_cat, cv = pl->t.Cv_cat;
    const int Kp = cs + 3 * cv, Kpw = (Kp + 31) / 32;
    const int K6 = m->C5s + 3 * m->C5v, K6w = (K6 + 31) / 32;
    pl->bits8 = o; o += up256(sizeof(uint32_t) * R * Kpw);
    pl->mask8 = o; o += up256(sizeof(uint32_t) * R * Kpw);
    pl->nvalid8 = o; o += up256(sizeof(int32_t) * R);
    pl->bits5 = o; o += up256(sizeof(uint32_t) * R * Kpw);
    pl->mask5 = o; o += up256(sizeof(uint32_t) * R * Kpw);
    pl->nvalid5 = o; o += up256(sizeof(int32_t) * R);
    pl->blp_bytes = svnet_binlinear_pool_workspace_bytes(R, Kp, m->C5s, N);
    pl->bl_bytes = pl->blp_bytes ? 0 : svnet_binlinear_workspace_bytes(R, Kp, m->C5s);
    pl->blp = o; o += up256(pl->blp_bytes + pl->bl_bytes);
    pl->s5 = o; o += pl->blp_bytes ? 0 : up256(sizeof(float) * R * m->C5s);
    pl->v5 = o; o += up256(sizeof(float) * R * 3 * m->C5v);
    pl->glob = o; o += up256(sizeof(float) * B * m->Kc);
    pl->vp = o; o += up256(sizeof(float) * B * 3 * m->C5v);
    pl->v6 = o; o += up256(sizeof(float) * B * 3 * m->C6v);
    pl->bits6 = o; o += up256(sizeof(uint32_t) * B * K6w);
    pl->mask6 = o; o += up256(sizeof(uint32_t) * B * K6w);
    pl->nvalid6 = o; o += up256(sizeof(int32_t) * B);
    pl->fuse_bytes = svnet_svfuse_pool_workspace(B, m->C5v, N);
    pl->fuse = o; o += up256(pl->fuse_bytes);
    const svnet_seg_head_params h = seg_head_params(m, B, N);
    pl->head_bytes = svnet_seg_head_workspace_bytes(&h);
    pl->head = o; o += up256(pl->head_bytes);
    pl->total = o;
    return pl->t.knn_bytes > 0 && pl->head_bytes > 0;
}

}  // namespace

extern "C" size_t svnet_model_seg_workspace_bytes(const svnet_model* m, int B, int N)
{
    if (!m || !m->pseg || B < 1 || N < 64 || N > 4096) return 0;
    const int ns = split_count(m, B, N);
    if (ns > 1) {
        size_t tot = 0;
        for (int i = 0; i < ns; ++i) {
            seg_plan2 pi;
            if (!make_seg_plan(m, sub_lo(B, ns, i + 1) - sub_lo(B, ns, i), N, &pi)) return 0;
            tot += pi.total;
        }
        return tot;
    }
    seg_plan2 pl;
    if (!make_seg_plan(m, B, N, &pl)) return 0;
    return pl.total;
}

namespace {

// one (sub-)batch of the part-segmentation model on `stream`; `aux` (optional) takes the chains that do not depend on the
// gate / the per-cloud branch: conv8's per-point sign words and conv5's scalar branch, then svfuse3's pooling and the label branch
int forward_seg_one(const svnet_model* m, const float* x, const float* label_onehot, int B, int N, float* logits, unsigned char* ws,
                    const seg_plan2& pl, void* stream, cudaStream_t aux, cudaEvent_t eF, cudaEvent_t eJ)
{
    cudaStream_t st = sv_stream(stream);
    const long R = (long)B * N;
    int rc = run_trunk(m, x, B, N, ws, pl.t, stream, aux, eF, eJ);
    void* sst = stream;
    if (aux) {
        SV_CUDA(cudaEventRecord(eF, st));
        SV_CUDA(cudaStreamWaitEvent(aux, eF, 0));
        sst = aux;
    }
    if (rc != SVNET_OK) return rc;
    float* s_cat = reinterpret_cast<float*>(ws + pl.t.s_cat);
    float* v_cat = reinterpret_cast<float*>(ws + pl.t.v_cat);
    float* gate = reinterpret_cast<float*>(ws + pl.t.gate);
    const int lds = pl.t.Cs_cat, xs = pl.t.Cv_cat, ldv = 3 * pl.t.Cv_cat, Kp = lds + 3 * xs, Kc = m->Kc;
    const int C5s = m->C5s, C5v = m->C5v, C6s = m->C6s, C6v = m->C6v, C3 = C5s + 3 * C5v;
    svnet_view cat = {};
    cat.s = s_cat; cat.lds = lds; cat.Cs = lds; cat.v = v_cat; cat.ldv = ldv; cat.xs = xs; cat.Cv = xs;
    // conv8's per-point sign words: svfuse1(s_cat, v_cat) against beta8[Kc:] (the float table is never written)
    uint32_t* bits8 = reinterpret_cast<uint32_t*>(ws + pl.bits8);
    uint32_t* mask8 = reinterpret_cast<uint32_t*>(ws + pl.mask8);
    int32_t* nvalid8 = reinterpret_cast<int32_t*>(ws + pl.nvalid8);
    if (m->binary) {
        rc = svnet_rows_prep(&cat, R, m->f1_Wz, m->f1_zs, nullptr, m->c8.beta + Kc, nullptr, 0, nullptr, bits8, mask8, nvalid8, sst);
        if (rc != SVNET_OK) return rc;
    }
    // conv5 per point: scalar output only pooled (max) -> glob[:, :C5s]; vector output v5
    const svnet_model::Block& c5 = m->conv[4];
    float* glob = reinterpret_cast<float*>(ws + pl.glob);
    float* v5 = reinterpret_cast<float*>(ws + pl.v5);
    uint32_t* bits5 = reinterpret_cast<uint32_t*>(ws + pl.bits5);
    uint32_t* mask5 = reinterpret_cast<uint32_t*>(ws + pl.mask5);
    int32_t* nvalid5 = reinterpret_cast<int32_t*>(ws + pl.nvalid5);
    if (!m->binary) {
        // full precision: u = [s | v2s(v)] rows -> dense linear1 + BN + LeakyReLU -> max over the points (as the fp classifier)
        float* u5 = reinterpret_cast<float*>(ws + pl.t.u5);
        float* s5 = reinterpret_cast<float*>(ws + pl.t.s5);
        rc = svnet_rows_prep(&cat, R, c5.Wz, nullptr, nullptr, nullptr, u5, Kp, nullptr, nullptr, nullptr, nullptr, sst);
        if (rc != SVNET_OK) return rc;
        svnet_gemm_params q = {};
        q.A = u5; q.lda_g = Kp; q.lda_x = 0; q.G = 1; q.W = c5.W1; q.ldw = Kp; q.M = R; q.N = C5s; q.K = Kp;
        q.bn_a = c5.bn1_a; q.bn_c = c5.bn1_c; q.act = SVNET_ACT_LEAKY; q.C = s5; q.ldc_g = C5s; q.ldc_x = 0; q.groups_per_cloud = 1;
        rc = svnet_linear_rows_ws(&q, ws + pl.t.lin, pl.t.lin_bytes, sst);
        if (rc != SVNET_OK) return rc;
        rc = svnet_pool_rows(s5, C5s, C5s, B, N, glob, nullptr, Kc, sst);
        if (rc != SVNET_OK) return rc;
    } else {
        rc = svnet_rows_prep(&cat, R, c5.Wz, c5.zscale, nullptr, c5.beta, nullptr, 0, nullptr, bits5, mask5, nvalid5, sst);
        if (rc != SVNET_OK) return rc;
        if (pl.blp_bytes) {
            rc = svnet_binlinear_pool_ws(bits5, mask5, R, Kp, c5.W1b, C5s, c5.scale1, c5.bn1_a, c5.bn1_c, N, glob, nullptr, Kc, ws + pl.blp,
                                         pl.blp_bytes, sst);
            if (rc != SVNET_OK) return rc;
        } else {
            float* s5 = reinterpret_cast<float*>(ws + pl.s5);
            rc = svnet_binlinear_rows_ws(bits5, mask5, nvalid5, R, Kp, c5.W1b, C5s, c5.scale1, nullptr, c5.bn1_a, c5.bn1_c, SVNET_ACT_LEAKY,
                                         nullptr, 1, s5, C5s, nullptr, pl.bl_bytes ? ws + pl.blp : nullptr, pl.bl_bytes, sst);
            if (rc != SVNET_OK) return rc;
            rc = svnet_pool_rows(s5, C5s, C5s, B, N, glob, nullptr, Kc, sst);
            if (rc != SVNET_OK) return rc;
        }
    }
    if (aux) SV_CUDA(cudaEventRecord(eJ, aux));
    rc = svnet_gate_rows(s_cat, lds, lds, B, N, c5.G1, c5.G2, c5.H, c5.Cvo, gate, stream);
    if (rc != SVNET_OK) return rc;
    {
        svnet_gemm_params q = {};
        q.A = v_cat; q.lda_g = ldv; q.lda_x = xs; q.G = 3; q.W = c5.W2; q.ldw = c5.Cv; q.M = 3 * R; q.N = C5v; q.K = c5.Cv;
        q.sign_w = m->binary; q.colscale = m->binary ? c5.scale2 : nullptr; q.bn_a = c5.bn2_a; q.bn_c = c5.bn2_c; q.vbn = 1; q.gate = gate;
        q.groups_per_cloud = N;
        q.C = v5; q.ldc_g = 3 * C5v; q.ldc_x = C5v;
        rc = svnet_linear_rows_ws(&q, nullptr, 0, stream);
        if (rc != SVNET_OK) return rc;
    }
    if (aux) {
        // join (conv5's pooled scalars are conv6's input), then fork again: svfuse3's pooling of v5 and the label branch next
        // to pool -> conv6 -> svfuse2, whose one-row-per-cloud kernels leave the GPU almost idle
        SV_CUDA(cudaStreamWaitEvent(st, eJ, 0));
        SV_CUDA(cudaEventRecord(eF, st));
        SV_CUDA(cudaStreamWaitEvent(aux, eF, 0));
    }
    // global branch: svpool over the points -> conv6 (one row per cloud) -> svfuse2
    float* vp = reinterpret_cast<float*>(ws + pl.vp);
    float* v6 = reinterpret_cast<float*>(ws + pl.v6);
    rc = svnet_pool_rows(v5, 3 * C5v, 3 * C5v, B, N, nullptr, vp, 3 * C5v, stream);
    if (rc != SVNET_OK) return rc;
    const svnet_model::Block& c6 = m->conv[5];
    svnet_view pv = {};
    pv.s = glob; pv.lds = Kc; pv.Cs = C5s; pv.v = vp; pv.ldv = 3 * C5v; pv.xs = C5v; pv.Cv = C5v;
    uint32_t* bits6 = reinterpret_cast<uint32_t*>(ws + pl.bits6);
    uint32_t* mask6 = reinterpret_cast<uint32_t*>(ws + pl.mask6);
    int32_t* nvalid6 = reinterpret_cast<int32_t*>(ws + pl.nvalid6);
    if (m->binary) {
        rc = svnet_rows_prep(&pv, B, c6.Wz, c6.zscale, nullptr, c6.beta, nullptr, 0, nullptr, bits6, mask6, nvalid6, stream);
        if (rc != SVNET_OK) return rc;
        rc = svnet_binlinear_rows_ws(bits6, mask6, nvalid6, B, C3, c6.W1b, C6s, c6.scale1, nullptr, c6.bn1_a, c6.bn1_c, SVNET_ACT_LEAKY,
                                     nullptr, 1, glob + C3, Kc, nullptr, nullptr, 0, stream);
        if (rc != SVNET_OK) return rc;
    } else {
        float* u6 = reinterpret_cast<float*>(ws + pl.u6);
        rc = svnet_rows_prep(&pv, B, c6.Wz, nullptr, nullptr, nullptr, u6, C3, nullptr, nullptr, nullptr, nullptr, stream);
        if (rc != SVNET_OK) return rc;
        svnet_gemm_params q = {};
        q.A = u6; q.lda_g = C3; q.lda_x = 0; q.G = 1; q.W = c6.W1; q.ldw = C3; q.M = B; q.N = C6s; q.K = C3;
        q.bn_a = c6.bn1_a; q.bn_c = c6.bn1_c; q.act = SVNET_ACT_LEAKY; q.C = glob + C3; q.ldc_g = Kc; q.ldc_x = 0; q.groups_per_cloud = 1;
        rc = svnet_linear_rows_ws(&q, ws + pl.t.lin, pl.t.lin_bytes, stream);
        if (rc != SVNET_OK) return rc;
    }
    rc = svnet_gate_rows(glob, Kc, C5s, B, 1, c6.G1, c6.G2, c6.H, c6.Cvo, gate, stream);
    if (rc != SVNET_OK) return rc;
    {
        svnet_gemm_params q = {};
        q.A = vp; q.lda_g = 3 * C5v; q.lda_x = C5v; q.G = 3; q.W = c6.W2; q.ldw = C5v; q.M = 3L * B; q.N = C6v; q.K = C5v;
        q.sign_w = m->binary; q.colscale = m->binary ? c6.scale2 : nullptr; q.bn_a = c6.bn2_a; q.bn_c = c6.bn2_c; q.vbn = 1; q.gate = gate;
        q.groups_per_cloud = 1;
        q.C = v6; q.ldc_g = 3 * C6v; q.ldc_x = C6v;
        rc = svnet_linear_rows_ws(&q, nullptr, 0, stream);
        if (rc != SVNET_OK) return rc;
    }
    svnet_view v6v = {};
    v6v.v = v6; v6v.ldv = 3 * C6v; v6v.xs = C6v; v6v.Cv = C6v;
    rc = svnet_rows_prep(&v6v, B, m->f2_Wz, m->f2_zs, nullptr, nullptr, glob + C3 + C6s, Kc, nullptr, nullptr, nullptr, nullptr, stream);
    if (rc != SVNET_OK) return rc;
    // svfuse3 + max over the points: v2s(v5) reduced on the fly -> glob[:, C5s:C3]
    svnet_view v5v = {};
    v5v.v = v5; v5v.ldv = 3 * C5v; v5v.xs = C5v; v5v.Cv = C5v;
    rc = svnet_svfuse_pool(&v5v, B, N, m->f3_Wz, m->f3_zs, glob + C5s, nullptr, Kc, ws + pl.fuse, pl.fuse_bytes, sst);
    if (rc != SVNET_OK) return rc;
    // conv7: the one-hot object label -> 64 channels (fp Conv1d + BN + LeakyReLU)
    {
        svnet_gemm_params q = {};
        q.A = label_onehot; q.lda_g = 16; q.lda_x = 0; q.G = 1; q.W = m->c7_W; q.ldw = 16; q.M = B; q.N = 64; q.K = 16;
        q.bn_a = m->c7_a; q.bn_c = m->c7_c; q.act = SVNET_ACT_LEAKY; q.C = glob + C3 + C6s + 3 * C6v; q.ldc_g = Kc; q.ldc_x = 0; q.groups_per_cloud = 1;
        rc = svnet_linear_rows_ws(&q, nullptr, 0, sst);
        if (rc != SVNET_OK) return rc;
    }
    if (aux) {
        SV_CUDA(cudaEventRecord(eJ, aux));
        SV_CUDA(cudaStreamWaitEvent(st, eJ, 0));
    }
    // segmentation head
    if (!m->binary) {
        svnet_seg_head_fp_params h = seg_head_fp_params(m, B, N);
        h.sv = cat; h.glob = glob; h.logits = logits;
        return svnet_seg_head_fp_fwd(&h, ws + pl.head, pl.head_bytes, stream);
    }
    svnet_seg_head_params h = seg_head_params(m, B, N);
    h.glob = glob; h.bits8 = bits8; h.mask8 = mask8; h.nvalid8 = nvalid8; h.logits = logits;
    return svnet_seg_head_fwd(&h, ws + pl.head, pl.head_bytes, stream);
}

}  // namespace

extern "C" int svnet_model_forward_seg(const svnet_model* m, const float* x, const float* label_onehot, int B, int N, float* logits,
                                       void* workspace, size_t workspace_bytes, void* stream)
{
    SV_REQUIRE(m && x && label_onehot && logits, "svnet_model_forward_seg: null pointer");
    SV_REQUIRE(m->pseg, "svnet_model_forward_seg: the handle is not a part-segmentation model (svnet_model_forward)");
    SV_REQUIRE(B >= 0 && N >= 64 && N <= 4096, "svnet_model_forward_seg: N = %d not covered (64..4096)", N);
    if (B == 0) return SVNET_OK;
    SV_REQUIRE(workspace && !(reinterpret_cast<uintptr_t>(workspace) & 255), "svnet_model_forward_seg: workspace null or not 256-byte aligned");
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    cudaStream_t st = sv_stream(stream);
    const bool ax = m->streams_ok;
    const int ns = split_count(m, B, N);
    if (ns == 1) {
        seg_plan2 pl;
        SV_REQUIRE(make_seg_plan(m, B, N, &pl), "svnet_model_forward_seg: shape not covered by the tensor-core paths");
        SV_REQUIRE(workspace_bytes >= pl.total, "svnet_model_forward_seg: workspace too small (svnet_model_seg_workspace_bytes)");
        return forward_seg_one(m, x, label_onehot, B, N, logits, ws, pl, stream, ax ? m->aux[0] : nullptr, ax ? m->ev[0] : nullptr,
                               ax ? m->ev[1] : nullptr);
    }
    SV_REQUIRE(workspace_bytes >= svnet_model_seg_workspace_bytes(m, B, N), "svnet_model_forward_seg: workspace too small (svnet_model_seg_workspace_bytes)");
    SV_CUDA(cudaEventRecord(m->ev[8], st));
    size_t off = 0;
    for (int i = 0; i < ns; ++i) {
        const int lo = sub_lo(B, ns, i), Bi = sub_lo(B, ns, i + 1) - lo;
        seg_plan2 pi;
        SV_REQUIRE(make_seg_plan(m, Bi, N, &pi), "svnet_model_forward_seg: shape not covered by the tensor-core paths");
        SV_CUDA(cudaStreamWaitEvent(m->sub[i], m->ev[8], 0));
        const int rc = forward_seg_one(m, x + (size_t)lo * 3 * N, label_onehot + (size_t)lo * 16, Bi, N, logits + (size_t)lo * m->ncls * N, ws + off, pi,
                                       m->sub[i], m->aux[i], m->ev[2 * i], m->ev[2 * i + 1]);
        if (rc != SVNET_OK) return rc;
        off += pi.total;
        SV_CUDA(cudaEventRecord(m->ev[9 + i], m->sub[i]));
        SV_CUDA(cudaStreamWaitEvent(st, m->ev[9 + i], 0));
    }
    return SVNET_OK;
}
