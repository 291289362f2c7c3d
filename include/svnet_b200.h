/*
 * svnet_b200.h -- C ABI of libsvnet_b200.so (sm_100a CUDA kernels for the SVNet inference hot path).
 *
 * The reference (hellozhuo/svnet) has no FFI layer: its only stable boundary is the Python
 * nn.Module API (SURVEY.md 8(b)).  This ABI sits directly underneath that API; every entry point
 * cites the reference function whose arithmetic it replaces (paths relative to /root/reference).
 * svnet_b200/*.py (the host-side mirror of models/sv_layers.py, models/utils/sv_util.py and the
 * four SV model files) is the only caller; INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch types.  All pointers are DEVICE pointers on
 *     the current CUDA device unless stated otherwise; buffers are caller-owned (the library is
 *     stateless: no handles, no global mutable state, re-entrant across devices/threads).
 *   - every launch goes to `stream` (a cudaStream_t passed as void*); nothing synchronises.
 *   - return 0 on success; on failure a negative code, message via svnet_last_error()
 *     (thread-local).  Shapes are validated before any launch.
 *   - all floating point is fp32; indices are int32 inside the fused path, int64 at the
 *     reference-facing boundary (torch.topk returns int64, sv_util.py:24).
 *
 * Point-feature views.  A point carries scalars s (Cs floats) and vectors v (3 x Cv floats, xyz
 * outer / channel inner, sv_layers.py:88,113).  Kernels address them through strided views so that
 * layer outputs can be written straight into the concatenated (svcat, sv_util.py:134-144) table:
 *     s[r][c]    = s[r*lds + c]
 *     v[r][x][c] = v[r*ldv + x*xs + c]
 */
#ifndef SVNET_B200_H
#define SVNET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVNET_ABI_VERSION 3

/* error codes */
#define SVNET_OK 0
#define SVNET_ERR_ARG (-1)   /* bad shape / null pointer / unsupported size */
#define SVNET_ERR_CUDA (-2)  /* CUDA runtime error on launch */

/* activation codes */
#define SVNET_ACT_NONE 0
#define SVNET_ACT_LEAKY 1 /* LeakyReLU(0.2), sv_layers.py:167 */
#define SVNET_ACT_RELU 2  /* sv_pointnet_cls.py:78-79 */

typedef struct {
    const float* s; /* may be NULL when Cs == 0 */
    int lds;
    int Cs;
    const float* v; /* may be NULL when Cv == 0 */
    int ldv;        /* row stride (floats) */
    int xs;         /* xyz stride (floats) */
    int Cv;
} svnet_view;

typedef struct {
    float* s;
    int lds;
    int Cs;
    float* v;
    int ldv;
    int xs;
    int Cv;
} svnet_mview;

int svnet_version(void);
const char* svnet_last_error(void);

/* ---- one-time weight preparation ------------------------------------------------------------ */

/* sign(W) bit-planes for a binarised Linear/Conv1d weight (sv_layers.py:43-45,70).
 * W [rows][ldw] (first K columns used) -> bits_t [ceil(K/32)][rows] (word-major, bit b of word w
 * = (W[row][32w+b] > 0)).  *zero_count (device int) receives the number of exactly-zero weights
 * (sign(0)=0 is not representable in one plane: with a count > 0 the consumers need the non-zero
 * plane of svnet_pack_sign_nz as well). */
int svnet_pack_sign(const float* W, int rows, int K, int ldw, uint32_t* bits_t, int* zero_count, void* stream);

/* The same sign plane plus the non-zero plane of a ternary weight (torch.sign(W) in {-1, 0, +1}):
 * nz_t [ceil(K/32)][rows], bit b of word w = (W[row][32w+b] != 0), K tail 0.  -0.0 counts as zero
 * (as torch.sign(-0.0) == 0), subnormal weights as +-1.  bits_t and *zero_count as svnet_pack_sign.
 * The consumers below take nz_t as `W1nz` through their *_nz entry points; NULL there means every
 * weight is +-1 (the plain entry points are those calls with NULL), so a caller keeps a plane only
 * where the zero count of its slice is > 0. */
int svnet_pack_sign_nz(const float* W, int rows, int K, int ldw, uint32_t* bits_t, uint32_t* nz_t, int* zero_count,
                       void* stream);

/* eval-mode BatchNorm1d as y = x*a + c (torch.nn.BatchNorm1d with running stats; sv_layers.py:84,166):
 * a = w/sqrt(var+eps), c = b - mean*a. */
int svnet_fold_bn(const float* w, const float* b, const float* mean, const float* var, float eps, int C,
                  float* a, float* c, void* stream);

/* ---- graph construction --------------------------------------------------------------------- */

/* knn(x,k), sv_util.py:19-25 -- feature of point r is [s | v(x=0) | v(x=1) | v(x=2)]
 * (sv_util.py:100-101; layer 1: s = xyz, Cs = 3, Cv = 0).  score p_ij = ((-xx_j) - (-2 f_i.f_j)) - xx_i
 * in fp32 with sequential fmaf chains over channels; k largest per row, nearest first, ties ->
 * lowest index.  No BxNxN matrix is written.  idx32 and/or idx64 [B][N][k] (either may be NULL).
 * 1 <= k <= min(N,128). */
int svnet_knn(const svnet_view* in, int B, int N, int k, int32_t* idx32, int64_t* idx64, void* stream);

/* Same result, bit for bit, with caller-owned scratch: when `workspace` holds at least
 * svnet_knn_workspace_bytes() bytes (16-byte aligned) the pairwise scores run on the tcgen05 tensor
 * cores as a FILTER (bf16 hi/mid/lo planes, fp32 accumulators in tensor memory) and every decision the
 * filter cannot certify is re-taken with the exact fp32 chain above (csrc/knn_tc.cu).
 * svnet_knn_workspace_bytes() returns 0 for shapes the tensor-core path does not cover (k > 48,
 * N > 4096, N < 64, more than 160 channels); svnet_knn_ws then runs the CUDA-core kernel. */
size_t svnet_knn_workspace_bytes(const svnet_view* in, int B, int N, int k);
int svnet_knn_ws(const svnet_view* in, int B, int N, int k, int32_t* idx32, int64_t* idx64, void* workspace,
                 size_t workspace_bytes, void* stream);
/* Cumulative counters of the tensor-core path (profiling aid): rows, rows that needed exact
 * re-scoring, rows that took the brute-force path, queued survivors, then CTAs and summed SM cycles of
 * {pass A, threshold, pass B}, [9] = float bits of the largest observed |tensor-core score - exact score| /
 * (xx_i + xx_j), [10] = rows with more than 32 survivors (all re-scored exactly).  Counters are only
 * accumulated when the environment variable SVNET_KNN_TC_STATS=1 (same-address atomics).
 * Host pointer to 12 values; reset != 0 clears. */
int svnet_knn_tc_stats(unsigned long long* out12, int reset);

/* get_graph_feature (nv=2, sv_util.py:28-62) / get_graph_feature_cross (nv=3, sv_util.py:64-88):
 * xyz [B][N][3], idx int64 [B][N][k] -> out [B][N][k][3][nv].  Materialising parity path. */
int svnet_graph_feature_xyz(const float* xyz, const int64_t* idx, int B, int N, int k, int nv, float* out,
                            void* stream);

/* get_graph_feature_sv, sv_util.py:106-114: s [B][N][Cs], v [B][N][3][Cv] ->
 * sf [B][N][k][2Cs], vf [B][N][k][3][2Cv].  Materialising parity path. */
int svnet_graph_feature_sv(const float* s, const float* v, const int64_t* idx, int B, int N, int k, int Cs,
                           int Cv, float* sf, float* vf, void* stream);

/* ---- SVBlock gate (sv_layers.py:156-161,179-183): g = sigmoid(G2 relu(G1 mean_rows(s))) -------- */

/* rows variant: s [B][rows][lds] (Cs used); G1 [H][Cs], G2 [Co][H]; gate [B][Co] */
int svnet_gate_rows(const float* s, int lds, int Cs, int B, int rows, const float* G1, const float* G2, int H,
                    int Co, float* gate, void* stream);

/* edge variant for get_graph_feature_sv edges: the block input is s_e = [s_j - s_i | s_i]
 * (sv_util.py:114), whose mean over the N*k edges of a cloud is computed from the kNN in-degrees
 * without touching an edge tensor.  G1 [H][2*Cs]. */
int svnet_gate_edge(const svnet_view* in, const int32_t* idx, int B, int N, int k, const float* G1,
                    const float* G2, int H, int Co, float* gate, void* stream);

/* first-layer variant: s_e = init_scalar([x_j-x_i | x_i (| x_j x x_i)]) (sv_dgcnn_cls.py:49-50,
 * sv_pointnet_cls.py:35-36).  Winit [3][nv]; G1 [H][3*nv]. */
int svnet_gate_xyz(const float* xyz, const int32_t* idx, int B, int N, int k, int nv, const float* Winit,
                   const float* G1, const float* G2, int H, int Co, float* gate, void* stream);

/* ---- fused edge convolutions ---------------------------------------------------------------- */

/* First edge layer: get_graph_feature[_cross] + init_scalar + SVBlock(FP) + svpool, fused
 * (sv_dgcnn_cls.py:49-53, sv_pointnet_cls.py:35-39).  Everything is full precision in every model
 * (sv_dgcnn_cls.py:29-30). */
typedef struct {
    const float* xyz;   /* [B][N][3] */
    const int32_t* idx; /* [B][N][k] */
    int B, N, k, nv;    /* nv = 2 (DGCNN) or 3 (PointNet, cross product channel) */
    const float* Winit; /* init_scalar.linear.weight [3][nv] */
    const float* Wz;    /* conv.v2s.linear.weight    [3][nv] */
    const float* W1;    /* conv.linear1.weight       [Cout][6*nv] */
    const float* bn1_a; /* folded bn1 [Cout] */
    const float* bn1_c;
    const float* W2;    /* conv.linear2.weight       [Cvo][nv] */
    const float* bn2_a; /* folded bn2.bn [Cvo] */
    const float* bn2_c;
    const float* gate;  /* [B][Cvo] */
    int Cout, Cvo;      /* Cout <= 64, Cvo <= 32 */
    svnet_mview out;    /* pooled s (max over k) and v (mean over k) */
} svnet_edge_xyz_params;
int svnet_edge_xyz_fwd(const svnet_edge_xyz_params* p, void* stream);

/* Edge layers 2..4: get_graph_feature_sv + SVBlock + svpool fused (sv_dgcnn_cls.py:55-65,
 * sv_layers.py:172-196, sv_util.py:90-132).  Per edge (i, j = idx[i][e]):
 *   s_e = [s_j - s_i | s_i], v_e = [v_j - v_i | v_i]                      (sv_util.py:109,114)
 *   z = v_e Wz^T (* zscale), q[d][m] = sum_x v_e[x][d] z[x][m]             (sv_layers.py:116-125)
 *   u = [s_e | q]   (K = 2Cs + 6Cv)
 *   binary: t = sign(u + beta); y_o = scale1_o * sum_k t_k sign(W1)_ok     (sv_layers.py:36-49)
 *           computed as XNOR/popcount on packed words with a zero-mask plane (sign(0) = 0)
 *   fp:     y = W1 u, with the first 2Cs columns pre-reduced per point: y = (Ya_j - Ya_i) + Yb_i + W1q q
 *   s' = act(y*bn1_a + bn1_c); pooled s = max_e s'                         (sv_layers.py:188-190)
 *   w = v_e W2^T = (P_j - P_i) + Q_i  with per-point tables P = v W2a^T, Q = v W2b^T (scale2 folded in)
 *   v' = w/n * (n*bn2_a + bn2_c) * gate, n = |w|_2 + 1e-6; pooled v = mean_e v'   (sv_layers.py:94-100,194)
 */
typedef struct {
    svnet_view in;       /* per-point s (Cs) and v (3 x Cv) of the previous layer */
    const int32_t* idx;  /* [B][N][k] */
    int B, N, k;
    int binary;
    const float* Wz;     /* [3][2Cv]; already sign()ed when binary */
    const float* zscale; /* [3] or NULL (fp) */
    /* scalar branch, binary */
    const float* beta;    /* [K] */
    const uint32_t* W1b;  /* [Kw][Cout] sign bits, word-major (svnet_pack_sign) */
    const float* scale1;  /* [Cout] */
    /* scalar branch, fp */
    const float* Yab;     /* [B*N][2*Cout]: Ya = s W1[:, :Cs]^T | Yb = s W1[:, Cs:2Cs]^T */
    const float* W1q_t;   /* [6Cv][Cout] = W1[:, 2Cs:]^T (k-major) */
    const float* bn1_a;   /* [Cout] */
    const float* bn1_c;
    int Cout;
    /* vector branch */
    const float* PQ;      /* [B*N][3][2*Cvo]: P | Q */
    const float* bn2_a;   /* [Cvo] */
    const float* bn2_c;
    const float* gate;    /* [B][Cvo] */
    int Cvo;
    svnet_mview out;
    /* optional parity taps (may be NULL): per edge sign words / nonzero-mask words [B*N*k][Kw] */
    uint32_t* dbg_bits;
    uint32_t* dbg_mask;
    /* optional, binary layers: with both set (and a covered shape, svnet_edge_tc_weight_bytes() > 0) linear1 runs on the
     * tcgen05 tensor cores (csrc/edge_tc.cu): ternary activations are written as fp8 e4m3 bytes straight into the UMMA
     * operand, +-1 weights likewise, fp32 accumulators in tensor memory hold the exact integer dot products. */
    const unsigned char* W1tc; /* svnet_edge_tc_pack_w() of conv.linear1.weight, svnet_edge_tc_weight_bytes() bytes, 16-byte aligned */
    const float* tab4;         /* [B*N][svnet_edge_tc_table_cols(Cv, Cvo)][4], 16-byte aligned: per-point table of (x, y, z, 0)
                                * columns [P (Cvo) | Q (Cvo) | T (3) | U (3) | v (Cv)] -- P | Q as in `PQ` (which may then be NULL),
                                * T = v Wz[:, :Cv]^T zscale, U = v Wz[:, Cv:]^T zscale (frames z_e = T_j + U_i - T_i), v = the layer
                                * input vectors; one svnet_linear_rows call with `c4` set produces it */
} svnet_edge_params;
int svnet_svblock_edge_fwd(const svnet_edge_params* p, void* stream);
/* Binary layers with ternary weights: W1nz [Kw][Cout] is the non-zero plane of conv.linear1.weight (svnet_pack_sign_nz)
 * or NULL (every weight +-1: svnet_svblock_edge_fwd).  y_o = scale1_o * sum over words of
 * (popc(m & z_o) - 2 popc((a ^ w_o) & m & z_o)).  The tensor-core kernel takes its zeros from W1tc; otherwise a call with a
 * plane runs the generic kernel (the shape-specialised CUDA-core kernels are +-1 only). */
int svnet_svblock_edge_fwd_nz(const svnet_edge_params* p, const uint32_t* W1nz, void* stream);

/* Tensor-core variant of the binary edge layers (sv_layers.py:36-49 on sv_util.py:90-116's edge features).
 * svnet_edge_tc_weight_bytes() is 0 for shapes / k the kernel does not cover (covered: the six edge-layer shapes of
 * SV_DGCNN_CLS / SV_DGCNN_PSEG at k = 20 or 40; SVNET_EDGE_TC=0 disables the path).  svnet_edge_tc_pack_w() turns
 * conv.linear1.weight [Cout][2Cs + 6Cv] (row stride ldw) into sign bytes in the kernel's operand layout; exact zeros
 * follow sign(0) = 0 (sv_layers.py:45). */
size_t svnet_edge_tc_weight_bytes(int Cs, int Cv, int Cout, int Cvo, int k);
int svnet_edge_tc_table_cols(int Cv, int Cvo);
int svnet_edge_tc_pack_w(const float* W1, int ldw, int Cs, int Cv, int Cout, unsigned char* out, void* stream);

/* The same for the full-precision edge layers (sv_layers.py:29-31,186-190; csrc/edge_fp_tc.cu): the q part of linear1
 * (K = 6 Cv) runs on tcgen05 as six products of exact three-way bf16 splits (fp32-grade), the s part comes from the
 * per-point table `Yab` in the epilogue.  svnet_edge_fp_tc_weight_bytes() is 0 for shapes / k the kernel does not cover
 * (covered: the three fp edge-layer shapes of SV_DGCNN_CLS at k = 20 and those of SV_DGCNN_PSEG at k = 20 and 40 -- a set of
 * (shape, k) pairs: the classifier's shapes at k = 40 are not covered; SVNET_EDGE_FP_TC=0 disables the path);
 * svnet_edge_fp_tc_pack_w() turns conv.linear1.weight [Cout][2Cs + 6Cv] into the three weight planes.  A full-precision
 * svnet_svblock_edge_fwd call takes this kernel when `W1tc` (those planes), `tab4` (float4 table, full-precision weights)
 * and `Yab` are set; `W1q_t` and `PQ` may then be NULL. */
size_t svnet_edge_fp_tc_weight_bytes(int Cs, int Cv, int Cout, int Cvo, int k);
int svnet_edge_fp_tc_pack_w(const float* W1, int ldw, int Cs, int Cv, int Cout, unsigned char* out, void* stream);

/* Multi-GPU (SURVEY.md 8(e)): all-gather of the per-rank outputs -- `count_per_rank` floats from `local` of every rank into
 * `all` (rank-major) -- on the caller's ncclComm_t and stream; replaces nn.DataParallel's gather
 * (main_cls_dgcnn.py:125, main_partseg_dgcnn.py:116).  The library resolves ncclAllGather at the first call from the NCCL
 * already loaded in the process (PyTorch's) or from libnccl.so.2; it does not link against NCCL.  Inside an
 * ncclGroupStart/End pair when one thread drives several devices. */
int svnet_allgather_logits(void* nccl_comm, const float* local, float* all, size_t count_per_rank, void* stream);

/* ---- per-row building blocks (conv5, PointNet per-point blocks, heads, module-level API) ---- */

/* u = [s | v2s(v)] for every row (sv_layers.py:185-186 / SVFuse :218-219), rows handled three at a
 * time per warp.  Outputs (each optional):
 *   u_out  [rows][ldu]      float u                       (fp linear1 input, SVFuse output)
 *   z_out  [rows][9]        the 3x3 frames z              (trans_back, sv_layers.py:126-127)
 *   bits/mask [rows][Kw]    sign(u + beta) > 0 / != 0     (binary linear1 input)
 *   nvalid [rows]           number of non-zero signs per row (= popcount of the mask row)
 * z_in [rows][9] (optional) supplies the frames instead of computing them from Wz: this is the
 * einsum('bimj,bijk->bimk') projection of sv_pointnet_partseg.py:93.
 * K = Cs + 3Cv.  With Cv == 0 this is a plain sign-pack of a float matrix (Linear ba, Conv1d). */
int svnet_rows_prep(const svnet_view* in, long rows, const float* Wz, const float* zscale, const float* z_in,
                    const float* beta, float* u_out, int ldu, float* z_out, uint32_t* bits, uint32_t* mask, int32_t* nvalid,
                    void* stream);

/* y[r][o] = act(((nvalid_r - 2*popc((a_r ^ w_o) & m_r)) [+ cloud_dot[r / rows_per_cloud][o]]) * scale[o] * bn_a[o] + bn_c[o])
 * (sv_layers.py:49 on packed words; bn/act optional).  bits/mask [rows][Kw]; W1b [Kw][Cout].
 * If out_i32 != NULL the raw integer dot products are written instead (used to pre-reduce
 * per-cloud-constant channels of the seg head, sv_dgcnn_partseg.py:117-121). */
int svnet_binlinear_rows(const uint32_t* bits, const uint32_t* mask, const int32_t* nvalid, long rows, int K,
                         const uint32_t* W1b, int Cout, const float* scale, const float* bias, const float* bn_a, const float* bn_c,
                         int act, const int32_t* cloud_dot, long rows_per_cloud, float* out, int ldo,
                         int32_t* out_i32, void* stream);

/* Same result, bit for bit, with caller-owned scratch: with svnet_binlinear_workspace_bytes() bytes of
 * workspace (16-byte aligned) the products run on the tcgen05 tensor cores -- ternary activations and
 * +-1 weights are exact in bf16, the fp32 accumulators hold exact integers (csrc/binlinear_tc.cu).
 * svnet_binlinear_workspace_bytes() returns 0 for shapes that stay on the popcount kernel
 * (rows < 2048, K < 64, K > 640).  By default only calls of the form scale -> BN -> LeakyReLU on
 * rows % 128 == 0 take the tensor-core path (lean epilogue, 2x the popcount kernel at conv5's shape);
 * SVNET_BINLINEAR_TC=2 forces it for every covered call, =0 disables it. */
size_t svnet_binlinear_workspace_bytes(long rows, int K, int Cout);
int svnet_binlinear_rows_ws(const uint32_t* bits, const uint32_t* mask, const int32_t* nvalid, long rows, int K,
                            const uint32_t* W1b, int Cout, const float* scale, const float* bias, const float* bn_a,
                            const float* bn_c, int act, const int32_t* cloud_dot, long rows_per_cloud, float* out,
                            int ldo, int32_t* out_i32, void* workspace, size_t workspace_bytes, void* stream);
/* svnet_binlinear_rows_ws with ternary weights: W1nz [Kw][Cout] non-zero plane of the weight (svnet_pack_sign_nz) or NULL
 * (every weight +-1, the calls above).  dot = sum over words of popc(m & z_o) - 2 popc((a ^ w_o) & m & z_o): the count of
 * non-zero products depends on (row, channel) and replaces nvalid_r.  Same kernels, same tensor-core coverage. */
int svnet_binlinear_rows_nz(const uint32_t* bits, const uint32_t* mask, const int32_t* nvalid, long rows, int K,
                            const uint32_t* W1b, const uint32_t* W1nz, int Cout, const float* scale, const float* bias,
                            const float* bn_a, const float* bn_c, int act, const int32_t* cloud_dot, long rows_per_cloud,
                            float* out, int ldo, int32_t* out_i32, void* workspace, size_t workspace_bytes, void* stream);

/* Binarised Linear -> BN -> LeakyReLU fused with the per-cloud max / mean over the rows (tensor-core path
 * only): the (rows, Cout) activation is never written.  SV_DGCNN_CLS pools conv5's scalar output right away
 * (sv_dgcnn_cls.py:68-74).  rows_per_cloud % 128 == 0; svnet_binlinear_pool_workspace_bytes() returns 0 for
 * shapes that are not covered (use svnet_binlinear_rows + svnet_pool_rows then). */
size_t svnet_binlinear_pool_workspace_bytes(long rows, int K, int Cout, long rows_per_cloud);
int svnet_binlinear_pool_ws(const uint32_t* bits, const uint32_t* mask, long rows, int K, const uint32_t* W1b, int Cout,
                            const float* scale, const float* bn_a, const float* bn_c, long rows_per_cloud,
                            float* max_out, float* mean_out, int ldo, void* workspace, size_t workspace_bytes,
                            void* stream);
/* The same with ternary weights: W1nz as in svnet_binlinear_rows_nz (NULL: svnet_binlinear_pool_ws). */
int svnet_binlinear_pool_nz(const uint32_t* bits, const uint32_t* mask, long rows, int K, const uint32_t* W1b,
                            const uint32_t* W1nz, int Cout, const float* scale, const float* bn_a, const float* bn_c,
                            long rows_per_cloud, float* max_out, float* mean_out, int ldo, void* workspace,
                            size_t workspace_bytes, void* stream);

/* Generic fp32 linear over (grouped) rows: C[m][n] = epi(sum_k A[m][k] * W[n][k]), sequential fmaf
 * chain over k (== oracle order).  Row m lives at A + (m / G)*lda_g + (m % G)*lda_x; same for C.
 *   sign_w: use sign(W) (binary weights, fp activations: sv_layers.py:43-49 with ba unset)
 *   epilogue: *colscale[n], +bias[n], *bn_a[n]+bn_c[n], act -- each optional (NULL / 0)
 *   vbn != 0 (requires G == 3): VectorBN + gate epilogue over the 3 rows of a group
 *           (sv_layers.py:94-100,194): out = w/n*(n*bn_a+bn_c)*gate[group / groups_per_cloud][n] */
typedef struct {
    const float* A; long lda_g; int lda_x; int G;
    const float* W; int ldw;
    long M; int N, K;
    int sign_w;
    const float* colscale; const float* bias; const float* bn_a; const float* bn_c; int act;
    int vbn; const float* gate; long groups_per_cloud;
    float* C; long ldc_g; int ldc_x;
    int c4;  /* != 0 (needs G == 3, no vbn; tcgen05 path only): the three rows of group g are stored as one float4
              * (x, y, z, 0) per column at C + g*ldc_g + 4*n (ldc_x unused) -- the table layout of the tensor-core edge kernel */
} svnet_gemm_params;
int svnet_linear_rows(const svnet_gemm_params* p, void* stream);
/* With svnet_linear_workspace_bytes(p) bytes of caller-owned scratch (16-byte aligned) a plain fp32 linear
 * (G == 1, no sign_w / vbn / gate / c4, 32 <= N <= 512, 32 <= K <= 4096; chosen by (K, N) only, never by the row count) runs on the tcgen05 tensor cores with
 * both operands split exactly into three bf16 planes (six plane products, fp32 accumulation in tensor memory:
 * fp32-level accuracy, different summation order -> tolerance-level, csrc/gemm_tc3.cu).  0 bytes: not covered,
 * svnet_linear_rows_ws then behaves as svnet_linear_rows. */
size_t svnet_linear_workspace_bytes(const svnet_gemm_params* p);
int svnet_linear_rows_ws(const svnet_gemm_params* p, void* workspace, size_t workspace_bytes, void* stream);

/* Classification head, one CTA per cloud: up to three chained layers, each a binarised Linear
 * (W1b + beta [+ scale]) or an fp Linear (W [Cout][K], sign_w for binary weights / fp activations),
 * then optional bias, BatchNorm affine and activation (sv_dgcnn_cls.py:76-80, sv_pointnet_cls.py:76-81).
 * x [B][ldx] (K0 used) -> out [B][ldo]. */
typedef struct {
    int Cout;
    const uint32_t* W1b;  /* [Kw][Cout] sign bits or NULL */
    const float* beta;    /* [K] (binary) */
    const float* W;       /* [Cout][K] (fp) */
    int sign_w;
    const float* scale;   /* [Cout] or NULL */
    const float* bias;    /* [Cout] or NULL */
    const float* bn_a;    /* [Cout] or NULL */
    const float* bn_c;
    int act;
} svnet_head_layer;
typedef struct {
    const float* x; int ldx; int K0; int B;
    int nlayers;
    svnet_head_layer layer[3];
    float* out; int ldo;
} svnet_head_params;
int svnet_head_fwd(const svnet_head_params* p, void* stream);
/* Binary layers with ternary weights: W1nz[l] is the non-zero plane [Kw][Cout] of layer l's weight (svnet_pack_sign_nz) or
 * NULL (+-1 weights); W1nz itself may be NULL (svnet_head_fwd).  A call with any plane reads the sign planes from global
 * memory instead of prefetching them into shared memory. */
int svnet_head_fwd_nz(const svnet_head_params* p, const uint32_t* const W1nz[3], void* stream);

/* Part-segmentation head as one call (sv_dgcnn_partseg.py:112-126): conv8 over [per-cloud channels | svfuse1(s_cat, v_cat)]
 * -> conv9 -> conv10 (binarised Conv1d + BN + LeakyReLU, sv_layers.py:64-78) -> conv11 (fp Conv1d) -> logits in the
 * reference's (B, parts, N) order.  It sequences this library's kernels on `stream` with svnet_seg_head_workspace_bytes()
 * bytes of caller-owned scratch (16-byte aligned) and is bit-identical to the layer-by-layer calls.
 *   sv           per-point inputs (s_cat [R][lds] (Cs used), v_cat [R][3][Cv]), R = B*N rows
 *   Wz1/zscale1  svfuse1.v2s (sv_layers.py:206-220)
 *   glob [B][ldg]  the Kc per-cloud-constant leading input channels of conv8 (the `repeat(1, 1, num_points)` block)
 *   beta8 [Kc + Cs + 3Cv], W8c / W8p  sign bit-planes (svnet_pack_sign) of conv8.weight[:, :Kc] / [:, Kc:], scale8, bn8_a/_c
 *   bits8/mask8/nvalid8  optional: conv8's per-point sign words computed by the caller ahead of time (svnet_rows_prep on
 *                `sv` with beta8 + Kc, e.g. on another stream next to the global branch); sv/Wz1 may then be NULL
 *   beta9 [C8], W9, ...; beta10 [C9], W10, ...; W11 [parts][C10] fp32 */
typedef struct {
    svnet_view sv;
    int B; long N;
    const float* Wz1; const float* zscale1;
    const float* glob; int ldg; int Kc;
    const float* beta8; const uint32_t* W8c; const uint32_t* W8p; const float* scale8; const float* bn8_a; const float* bn8_c; int C8;
    const uint32_t* bits8; const uint32_t* mask8; const int32_t* nvalid8;
    const float* beta9; const uint32_t* W9; const float* scale9; const float* bn9_a; const float* bn9_c; int C9;
    const float* beta10; const uint32_t* W10; const float* scale10; const float* bn10_a; const float* bn10_c; int C10;
    const float* W11; int parts;
    float* logits;        /* [B][parts][N] */
} svnet_seg_head_params;
size_t svnet_seg_head_workspace_bytes(const svnet_seg_head_params* p);
int svnet_seg_head_fwd(const svnet_seg_head_params* p, void* workspace, size_t workspace_bytes, void* stream);
/* The same with ternary weights: non-zero planes (svnet_pack_sign_nz) of W8c, W8p, W9 and W10, each NULL when that plane's
 * weights are all +-1 (all NULL: svnet_seg_head_fwd).  Same workspace. */
int svnet_seg_head_fwd_nz(const svnet_seg_head_params* p, const uint32_t* W8c_nz, const uint32_t* W8p_nz, const uint32_t* W9_nz,
                          const uint32_t* W10_nz, void* workspace, size_t workspace_bytes, void* stream);

/* The same head of the full-precision model (binary = False: plain Conv1d weights, no beta / scale) as one call.  conv8's
 * input is [glob[b] repeated over the points | svfuse1(s_cat, v_cat)]; its per-cloud part W8[:, :Kc] glob[b] is computed
 * once per cloud and added to every point's W8[:, Kc:] u before BN + LeakyReLU, so the (B*N, Kc + Cs + 3Cv) table is never
 * written.  Every linear (per-cloud term, conv8 .. conv11) goes through svnet_linear_rows_ws as the layer-by-layer calls do:
 * the three-plane tcgen05 fp linear where it covers (K, N), e.g. not conv11 with fewer than 32 parts (chosen by (K, N) only:
 * a cloud's logits do not depend on its batch); tolerance-level against the layer-by-layer calls (conv8's K is split).
 * svnet_seg_head_fp_workspace_bytes() is 0 when the per-point conv8 (K = Cs + 3Cv, C8), which carries the per-cloud term,
 * is not covered by the tcgen05 linear (SVNET_LINEAR_TC=0).
 *   sv / Wz1      svfuse1's input and its v2s weight [3][Cv] (full precision: no scale); its (B*N, Cs + 3Cv) rows go to
 *                 the workspace
 *   glob [B][ldg] the Kc per-cloud-constant leading input channels of conv8
 *   W8 [C8][Kc + Cs + 3Cv], W9 [C9][C8], W10 [C10][C9] with folded BatchNorm affines; W11 [parts][C10] */
typedef struct {
    svnet_view sv;
    int B; long N;
    const float* Wz1;
    const float* glob; int ldg; int Kc;
    const float* W8; const float* bn8_a; const float* bn8_c; int C8;
    const float* W9; const float* bn9_a; const float* bn9_c; int C9;
    const float* W10; const float* bn10_a; const float* bn10_c; int C10;
    const float* W11; int parts;
    float* logits;        /* [B][parts][N] */
} svnet_seg_head_fp_params;
size_t svnet_seg_head_fp_workspace_bytes(const svnet_seg_head_fp_params* p);
int svnet_seg_head_fp_fwd(const svnet_seg_head_fp_params* p, void* workspace, size_t workspace_bytes, void* stream);

/* VectorBN on materialised rows (module-level parity for sv_layers.VectorBN, :86-102):
 * v [rows][3][C] contiguous -> out. */
int svnet_vector_bn_rows(const float* v, long rows, int C, const float* bn_a, const float* bn_c, float* out,
                         void* stream);

/* Pool over the rows of each cloud: x [B][rows][ld] (C used).  max_out / mean_out [B][ldo] (C
 * written), each optional (svpool dim=1, sv_util.py:125-131; adaptive_{max,avg}_pool1d,
 * sv_dgcnn_cls.py:72-73).  v-shaped inputs are pooled as 3*Cv scalar columns. */
int svnet_pool_rows(const float* x, int ld, int C, int B, long rows, float* max_out, float* mean_out, int ldo,
                    void* stream);

/* SVFuse + global pooling of SV_DGCNN_CLS (sv_layers.py:206-220 with sv_dgcnn_cls.py:70-74), fused:
 * q = v2s(v) [rows][3*Cv] is reduced on the fly to the per-cloud column max and mean; the fused table
 * never reaches HBM.  in->v [B*rows_per_cloud][3][Cv] (in->Cs must be 0 / s ignored); Wz [3][Cv],
 * zscale [3] or NULL; max_out / mean_out [B][ldo] (either may be NULL); 3*Cv <= 512.
 * workspace: svnet_svfuse_pool_workspace() bytes (partials, combined in a fixed order). */
size_t svnet_svfuse_pool_workspace(int B, int Cv, long rows_per_cloud);
int svnet_svfuse_pool(const svnet_view* in, int B, long rows_per_cloud, const float* Wz, const float* zscale,
                      float* max_out, float* mean_out, int ldo, void* workspace, size_t workspace_bytes, void* stream);

/* ---- whole-model entry (SURVEY.md 8(b)) ------------------------------------------------------------------------
 * The SV-DGCNN classifier, binary or full precision (models/sv_dgcnn_cls.py:22-82), from a checkpoint's tensors to logits.
 * svnet_model_create() takes the state_dict as (name, device pointer, element count) triples -- the reference's key names
 * without the 'module.' prefix (SURVEY 8(a) a-keys), fp32, contiguous -- copies what it needs and packs it once (sign
 * bit-planes, folded BatchNorm affines, tensor-core operand bytes, per-point table weights); it synchronises `stream` before
 * it returns, the caller's tensors may then be freed.  Covered: kind "SV_DGCNN_CLS", k = 20 (binary = 1 also k = 40); kind
 * "SV_DGCNN_PSEG" below.  A state_dict that lacks a tensor of the kind / precision asked for fails with its name.
 * svnet_model_forward(): x [B][3][N] -> logits [B][num_class] on `stream`, with svnet_model_workspace_bytes(m, B, N) bytes of
 * caller-owned scratch (256-byte aligned; 0: shape not covered -- 64 <= N <= 4096).  It allocates
 * nothing and never synchronises the host, so it can be captured into a CUDA graph; inside, the work forks from `stream` onto
 * streams owned by the handle (up to four sub-batches, auxiliary chains) and joins it again -- one handle must not run two forwards
 * concurrently.  The logits are bit-identical to the nn.Module path (svnet_b200.SV_DGCNN_CLS), which makes the same calls
 * through this header. */
typedef struct { const char* name; const float* data; long numel; } svnet_tensor;
typedef struct svnet_model svnet_model;
int svnet_model_create(const char* kind, int k, int binary, int num_class, const svnet_tensor* tensors, int n_tensors,
                       void* stream, svnet_model** out);
size_t svnet_model_workspace_bytes(const svnet_model* m, int B, int N);
int svnet_model_forward(const svnet_model* m, const float* x, int B, int N, float* logits, void* workspace,
                        size_t workspace_bytes, void* stream);
void svnet_model_destroy(svnet_model* m);
/* kind "SV_DGCNN_PSEG" (models/sv_dgcnn_partseg.py:40-128; binary = 1 or 0, k = 20 or 40, num_class = number of parts):
 * x [B][3][N], label_onehot [B][16] -> logits [B][parts][N], with svnet_model_seg_workspace_bytes() bytes of scratch.
 * Full precision (binary = 0): the state_dict has no beta / scale tensors; conv5 / conv6 are dense linears over
 * u = [s | v2s(v)], svfuse1..3 plain v2s, and the head is svnet_seg_head_fp_fwd -- the same calls as the nn.Module path. */
size_t svnet_model_seg_workspace_bytes(const svnet_model* m, int B, int N);
int svnet_model_forward_seg(const svnet_model* m, const float* x, const float* label_onehot, int B, int N, float* logits,
                            void* workspace, size_t workspace_bytes, void* stream);

/* Input side of the eval loop (SURVEY.md 8(f) f3): out[b][c][n] = sum_d pts[b][n][d] * R[b][d][c]
 * (pytorch3d Rotate.transform_points, then permute(0,2,1): main_cls_dgcnn.py:229-235).
 * pts [B][N][3], R [B][3][3] or NULL (permute only) -> out [B][3][N]. */
int svnet_rotate_permute(const float* pts, const float* R, int B, int N, float* out, void* stream);

/* svpool over k on materialised edge tensors (module-level parity, sv_util.py:118-132) is
 * svnet_pool_rows with B := B*N and rows := k. */

#ifdef __cplusplus
}
#endif
#endif /* SVNET_B200_H */
