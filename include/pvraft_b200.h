/*
 * pvraft_b200 -- C ABI of the B200-native (sm_100a) PV-RAFT hot path.
 *
 * The reference (weiyithu/PV-RAFT) has no FFI layer: its boundary is the Python nn.Module API
 * (SURVEY.md section 8b).  This header is the drop-in boundary underneath that API: every entry
 * point below replaces the ATen / torch-scatter op sequence of one reference function, cited as
 * `file:line` relative to the reference tree.  The Python mirror of the reference modules
 * (pvraft_b200/*.py, model/*.py) binds these symbols with ctypes -- see INTEGRATION.md.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.  `stream` is a cudaStream_t
 *     passed as void*.  All pointers are DEVICE pointers on the current device.
 *   - Every call is asynchronous on `stream`, allocates nothing, never synchronises, keeps no
 *     state between calls (re-entrant); the caller owns every buffer.
 *   - Return value: 0 = ok; < 0 = pvraft_status (argument / capability error, nothing launched);
 *     > 0 = cudaError_t of the failed launch.  pvraft_last_error_string() describes the last
 *     non-zero return on the calling thread.
 *   - Tensors are contiguous fp32 unless stated.  Point-major layout [B,N,C] is used for every
 *     per-point feature array (one point's channels are contiguous), coordinates are [B,N,3].
 *   - GroupNorm statistics travel as raw double-precision sums ("stats": [B,8,2] = per sample,
 *     per group (sum, sum of squares)); producers ACCUMULATE with atomics, so the caller zeroes
 *     them (cudaMemsetAsync) before the producing call.
 *   - Weights are passed in the reference's own state_dict layouts ([Cout,Cin(,1(,1))] row-major).
 */
#ifndef PVRAFT_B200_H
#define PVRAFT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PVRAFT_VERSION 100 /* 0.1.0 */

#if defined(__GNUC__)
#define PVRAFT_API __attribute__((visibility("default")))
#else
#define PVRAFT_API
#endif

typedef enum pvraft_status {
    PVRAFT_OK = 0,
    PVRAFT_ERR_BAD_ARG = -1,     /* null pointer, non-positive size ... */
    PVRAFT_ERR_UNSUPPORTED = -2, /* shape outside what the kernels are built for */
    PVRAFT_ERR_SMEM = -3         /* working set does not fit the 227 KB shared memory of an SM */
} pvraft_status;

#define PVRAFT_KNN 32        /* model/corr.py:9, model/extractor.py:9 -- hard-coded in the reference */
#define PVRAFT_GN_GROUPS 8   /* model/corr.py:17,25 ; model/flot/gconv.py:27,30,33 */
#define PVRAFT_MOMENTS 16    /* doubles per sample for the kNN-branch moment accumulator */

PVRAFT_API int pvraft_version(void);
PVRAFT_API const char* pvraft_last_error_string(void);
/* number of SMs / max opt-in dynamic shared memory of the current device (plumbing for the host) */
PVRAFT_API int pvraft_device_info(int* sm_count, int* smem_optin_bytes);

/* ------------------------------------------------------------------------------------------------
 * All-pairs feature correlation on the tcgen05 tensor cores with an fp32-accurate 3xTF32 split.
 * Replaces CorrBlock.calculate_corr, model/corr.py:95-100: corr[b,i,j] = <fmap1[b,i,:], fmap2[b,j,:]> / sqrt(C).
 *   fmap1, fmap2 [B,N,C] POINT-major f32 -> corr [B,N,N] f32.   N % 128 == 0, C % 32 == 0.
 *   workspace: pvraft_corr_matmul_workspace_bytes(B,N,C) bytes (16-byte aligned) for the hi/lo operand splits.
 * --------------------------------------------------------------------------------------------- */
PVRAFT_API int64_t pvraft_corr_matmul_workspace_bytes(int B, int N, int C);
PVRAFT_API int pvraft_corr_matmul_fwd(const float* fmap1, const float* fmap2, int B, int N, int C, float* corr, void* workspace,
                           void* stream);

/* ------------------------------------------------------------------------------------------------
 * Correlation truncation: the K largest entries of every row of a dense correlation matrix.
 * Replaces torch.topk(corr, k, dim=2, sorted=True) in CorrBlock.init_module, model/corr.py:37-40.
 *   corr [B,N,M] -> val [B,N,K] f32, idx [B,N,K] int32 column ids, written in ASCENDING COLUMN order
 *   (value ties at the K-th place: lowest columns win).  The reference's descending-value order carries
 *   no meaning downstream; pvraft_corr_reorder rearranges every row for the lookup kernel anyway.
 * Requires 1 <= K <= min(M, 1024) and M <= 49152 (the row is staged in shared memory).
 * --------------------------------------------------------------------------------------------- */
PVRAFT_API int pvraft_corr_topk_fwd(const float* corr, int B, int N, int M, int K, float* val, int32_t* idx, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Bank-aware arrangement of the truncated state, once per forward (no reference counterpart: the order of
 * the K candidates inside a row carries no meaning in model/corr.py beyond fp summation order).
 * Every row of (val, idx) [rows, K] is permuted so that the 32 candidates the lookup kernel gathers with
 * one instruction fall into (nearly) distinct shared-memory banks.  Out of place; deterministic.
 * --------------------------------------------------------------------------------------------- */
PVRAFT_API int pvraft_corr_reorder(const float* val_in, const int32_t* idx_in, int64_t rows, int K, float* val_out,
                                   int32_t* idx_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Point-voxel correlation lookup (index + reduce part), one fused pass over the K candidates of
 * every point.  Replaces CorrBlock.get_voxel_feature up to (not incl.) out_conv, model/corr.py:47-71,
 * and CorrBlock.get_knn_feature up to (not incl.) knn_conv, model/corr.py:75-91.
 *   corr_val [B,N,K] f32, corr_idx [B,N,K] int32 (rows of xyz2), xyz2_pad [B,N,4] = (x,y,z,0) rows of the second cloud
 *   (pvraft_xyz_pad_fwd, once per forward; 16-byte aligned, as corr_idx), coords [B,N,3]
 *   -> vox      [B,N,vox_ld]     (vox_ld >= levels*27, 0 = dense; pad columns are written as zeros so that the
 *                                consumer can read rows with 128-bit loads)  channel = level*27 + cell; mean corr of the candidates whose
 *                                round((xyz-coords)/r_level) lies in {-1,0,1}^3  (round-half-even,
 *                                true fp32 division; r_level = base_scale * 2^level)
 *   -> knn_sel  [B,N,32,4]       (corr, dx, dy, dz) of the 32 candidates nearest to coords
 *                                (distance = (dx*dx+dy*dy)+dz*dz, no FMA); order within a point is
 *                                unspecified; exact-distance ties at the 32nd place are broken deterministically
 *   -> knn_slot [B,N,32] int32   candidate slot (0..K-1) of each selected neighbour; may be NULL
 *   -> moments  [B,16] double    first/second moments of the 4-vector over the sample's N*32 edges, accumulated with
 *                                atomics into a buffer the caller has ZEROED: [0..3]=sum f_i, [4..13]=sum f_i f_j (i<=j,
 *                                row-major upper triangle), [14]=edge count, [15]=scratch (the kernel's work counter);
 *                                may be NULL (then the points are split statically)
 *   -> dbg_cube [B,N,K,levels] int8  cell id or -1 of every candidate AS DERIVED BY THE FUSED KERNEL ITSELF (the coarsest-cube
 *                                pre-test, the compaction and the per-level cell codes); test hook, NULL in production
 * K in {32,64,128,256,512,1024}; 1 <= levels <= 4; knn fixed at 32.
 * --------------------------------------------------------------------------------------------- */
/* The same lookup on the reduced-precision state of BASELINE.json configs[2] ("bf16 mode", SURVEY.md H7): correlation values as
 * bf16 bit patterns and candidate ids as uint16 (N <= 65536) -- 4 B instead of 8 B per candidate and iteration.  Index math
 * (coordinates, cells, kNN distances) stays fp32 and bit-exact; values are widened to fp32 exactly and accumulated in fp32, so
 * the outputs equal pvraft_corr_lookup_fwd on the bf16-rounded correlations.  K in {128,256,512,1024}.
 * pvraft_corr_state_pack_bf16 converts a reordered fp32/int32 state (round to nearest even; inf stays inf, a NaN becomes a quiet
 * NaN of the same sign). */
PVRAFT_API int pvraft_corr_lookup_bf16_fwd(const uint16_t* corr_val_bf16, const uint16_t* corr_idx_u16, const float* xyz2_pad,
                                const float* coords, int B, int N, int K, int levels, float base_scale, float* vox, int vox_ld,
                                float* knn_sel, int32_t* knn_slot, double* moments, int8_t* dbg_cube, void* stream);
PVRAFT_API int pvraft_corr_state_pack_bf16(const float* val, const int32_t* idx, int64_t n, uint16_t* val_out, uint16_t* idx_out, void* stream);

/* xyz [rows,3] -> out [rows,4] = (x,y,z,0): the gather table of the lookup kernel (one 128-bit load per candidate). */
PVRAFT_API int pvraft_xyz_pad_fwd(const float* xyz, int64_t rows, float* out, void* stream);
PVRAFT_API int pvraft_corr_lookup_fwd(const float* corr_val, const int32_t* corr_idx, const float* xyz2_pad, const float* coords,
                           int B, int N, int K, int levels, float base_scale, float* vox, int vox_ld, float* knn_sel,
                           int32_t* knn_slot, double* moments, int8_t* dbg_cube, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Generic fused (GroupNorm -> activation -> 1x1 conv [-> bias] [-> ReLU]) layer over points with
 * GroupNorm statistics of the OUTPUT accumulated on the fly.  It is the dense building block of
 * CorrBlock.out_conv[0] (model/corr.py:16), SetConv.fc2/fc3 and the fc1 pre-transform
 * (model/flot/gconv.py:26-33,58-85), FlotRefine.fc (model/refine.py:14,21).
 * --------------------------------------------------------------------------------------------- */
typedef enum pvraft_in_mode {
    PVRAFT_IN_PLAIN = 0,  /* x = in                                                     */
    PVRAFT_IN_GN = 1,     /* x = act(GN(in))            using in_stats/in_gamma/in_beta  */
    PVRAFT_IN_GN_MINMAX = 2 /* x = act(GN(in_max or in_min)): per channel picks max when the GN scale is >= 0,
                               min otherwise (max-pool over neighbours commuted with the monotone GN+LeakyReLU) */
} pvraft_in_mode;

typedef enum pvraft_act {
    PVRAFT_ACT_NONE = 0,
    PVRAFT_ACT_RELU = 1,
    PVRAFT_ACT_LRELU = 2 /* slope in act_slope (LeakyReLU 0.1, or PReLU with its learned slope) */
} pvraft_act;

typedef struct pvraft_linear_args {
    const float* in;        /* [B,N,cin] (PLAIN/GN) or the per-channel max array (GN_MINMAX) */
    const float* in_min;    /* [B,N,cin] per-channel min (GN_MINMAX only) */
    const double* in_stats; /* [B,8,2] sums of the un-normalised input (GN modes) */
    const float* in_gamma;  /* [cin] */
    const float* in_beta;   /* [cin] */
    double in_count;        /* number of elements per (sample, group) behind in_stats */
    int in_mode;            /* pvraft_in_mode */
    int in_act;             /* pvraft_act applied after the input GroupNorm */
    float in_slope;
    const float* weight;    /* [cout,w_cin] row-major; row stride w_ld floats (0 = w_cin): lets fc1.weight[:, :cin] be used in place */
    int w_ld;
    int w_cin;              /* weight columns used (0 = cin); input columns w_cin..cin-1 are padding and are ignored */
    const float* bias;      /* [cout] or NULL */
    const float* residual;  /* [B,N,cout] added to the output after bias/activation, or NULL (model/refine.py:22) */
    int out_act;            /* pvraft_act applied to the output (NONE or RELU) */
    float* out;             /* [B,N,cout] */
    double* out_stats;      /* [B,8,2] ACCUMULATED sums of `out`, or NULL (cout % 8 == 0 required) */
    int B, N, cin, cout;
} pvraft_linear_args;

PVRAFT_API int pvraft_linear_fwd(const pvraft_linear_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * The same fused layer on the tcgen05 tensor cores (TMA + TMEM), fp32-accurate through a 3xTF32 operand split.
 * Up to three activation sources are concatenated along K (e.g. [h | inp | motion] of the ConvGRU,
 * model/update.py:32,36); the GroupNorm(+max/min selection)+activation prologue and the bias / ReLU / residual /
 * GroupNorm-statistics epilogue match pvraft_linear_fwd; two extra epilogues implement the ConvGRU gates
 * (model/update.py:34-39).  Requirements: points per sample N % 128 == 0; every source has a multiple of 32
 * channels; weights pre-split with pvraft_tc_weight_split into hi/lo [n_pad, K] (n_pad = cout rounded up to 16, <= 128).
 * --------------------------------------------------------------------------------------------- */
typedef enum pvraft_tc_epilogue {
    PVRAFT_TC_PLAIN = 0,   /* out = act(acc + bias) (+ residual), optional output statistics                  */
    PVRAFT_TC_GRU_ZR = 1,  /* acc = [z|r] pre-activations (n_pad = 128): out = sigmoid(z), out2 = sigmoid(r) * h */
    PVRAFT_TC_GRU_Q = 2,   /* acc = q pre-activation: out = (1 - z) * h + z * tanh(acc + bias)                  */
    PVRAFT_TC_FLOW = 3     /* FlowHead tail (model/update.py:72) + RAFT update (model/RAFTSceneFlow.py:45-46), cout = 64:
                              out[B,N,3] = delta = w3 . relu(acc + bias) + b3; coords2_out = coords2 + delta;
                              flow_out = coords2_out - coords1 (the last two optional)                         */
} pvraft_tc_epilogue;

typedef struct pvraft_tc_linear_args {
    const float* in[3];     /* activation sources [B,N,in_channels[i]]; unused entries NULL */
    int in_channels[3];
    const float* in_min;    /* per-channel minima paired with in[0] (GroupNorm prologue with max/min selection) or NULL */
    const double* in_stats; /* [B,8,2] -> GroupNorm prologue on source 0 (further sources are taken as they are), or NULL */
    const float* in_gamma;
    const float* in_beta;
    double in_count;
    int in_act;             /* pvraft_act */
    float in_slope;
    const float* w_hi;      /* [n_pad, K] tf32 high parts, K = sum of in_channels */
    const float* w_lo;      /* [n_pad, K] tf32 low parts */
    int n_pad, cout;
    const float* bias;      /* [cout] or NULL (GRU_ZR: bias of z; GRU_Q: bias of q) */
    const float* bias2;     /* GRU_ZR: bias of r */
    int out_act;
    const float* residual;  /* PLAIN: [B,N,cout] added to the output, or NULL.  GRU epilogues: per-point term added to the
                               pre-activations ([B,N,128] = [z|r] for GRU_ZR, [B,N,64] for GRU_Q) -- the contribution of the
                               context features, constant over the RAFT iterations -- or NULL */
    float* out;             /* [B,N,cout] */
    float* out2;            /* GRU_ZR: r*h [B,N,64] */
    const float* h;         /* GRU epilogues: previous hidden state [B,N,64] */
    const float* z;         /* GRU_Q: update gate [B,N,64] */
    double* out_stats;      /* [B,8,2] accumulated, or NULL */
    int epilogue;           /* pvraft_tc_epilogue */
    int B, N;
    const float* tail;      /* PLAIN, or NULL: [B,N,3] copied into output columns cout..cout+2 (out row stride cout+3 = n_pad):
                               the MotionEncoder's `cat([out, flow])`, model/update.py:20 */
    const float* w3;        /* FLOW: flow_head.out_conv.2.weight [3,64] */
    const float* b3;        /* FLOW: flow_head.out_conv.2.bias [3] */
    const float* coords1;   /* FLOW: [B,N,3] or NULL */
    const float* coords2;   /* FLOW: [B,N,3] or NULL */
    float* coords2_out;     /* FLOW: [B,N,3] or NULL (may alias coords2) */
    float* flow_out;        /* FLOW: [B,N,3] or NULL */
    float* flow_user;       /* FLOW: second copy of the flow, row r written at row row_map[r] ([B*N,3]) -- the caller's
                               point order when the cloud was spatially reordered for locality -- or NULL */
    const int32_t* row_map; /* FLOW: [B*N] destination rows of flow_user */
    int params_settled;     /* nonzero: w_hi, w_lo, bias, bias2, w3, b3 were last written at least three launches ago on this
                               stream (or before a synchronisation).  The kernel is launched with programmatic stream
                               serialization and then fetches them while the previous kernel drains.  0 is always safe. */
    int32_t* done;          /* [B] zero-initialised counters or NULL: every finished 128-point tile adds 8 to its sample's entry
                               (release), after its rows and GroupNorm sums are written */
    const int32_t* wait_on; /* NULL, or the `done` array of the launch IMMEDIATELY BEFORE this one on the stream, which produced
                               this layer's inputs: the kernel then starts on a sample as soon as that launch has finished it
                               (acquire on its counter) instead of waiting for the whole grid.  Needs params_settled; outputs must
                               not alias anything the previous launch reads.  Ignored (full wait) otherwise. */
} pvraft_tc_linear_args;

PVRAFT_API int pvraft_tc_linear_fwd(const pvraft_tc_linear_args* a, void* stream);
/* hi = tf32(w), lo = tf32(w - hi) of the window w[0:rows, col0:col0+cols] of a row-major matrix with row stride ld,
 * written zero-padded as [rows_pad, cols_pad]. */
PVRAFT_API int pvraft_tc_weight_split(const float* w, int rows, int cols, int ld, int col0, int rows_pad, int cols_pad,
                           float* hi, float* lo, void* stream);

/* out[B,N,C] (or channel-major [B,C,N] when transpose_out != 0) = act(GN(in)) -- the trailing
 * GroupNorm+LeakyReLU of SetConv (model/flot/gconv.py:33,82-83) when nothing follows it. */
PVRAFT_API int pvraft_gn_act_fwd(const float* in, const double* stats, const float* gamma, const float* beta, double count,
                      int act, float slope, int B, int N, int C, int transpose_out, float* out, const float* slope_dev, void* stream);
/* slope_dev (here and in pvraft_gn_act_bwd): optional DEVICE pointer to the slope -- the one-element nn.PReLU weight -- read by the
 * kernel instead of `slope`; the training path uses it so that a parameter the optimizer changes every step needs no host read-back. */

/* ------------------------------------------------------------------------------------------------
 * Correlation feature head (+ optional MotionEncoder), one persistent kernel.
 *  feature stage (when y1 != NULL): out_conv[1:] on the voxel branch + knn_conv/max/knn_out on the
 *    kNN branch, summed.  Replaces model/corr.py:17-19 (GN, PReLU, Conv1d 128->64), :24-29,:91-93, :45.
 *      y1 [B,N,128] = out_conv[0] output (pvraft_linear_fwd) with y1_stats [B,8,2];
 *      knn_sel [B,N,32,4], moments [B,16] from pvraft_corr_lookup_fwd  -> corr_feat [B,N,64] (may be NULL)
 *  motion stage (when motion != NULL): MotionEncoder.forward, model/update.py:15-21, on the feature
 *    just computed (or on corr_in [B,N,64] when y1 == NULL) and flow [B,N,3] -> motion [B,N,64]
 *    (channels 0..60 learned, 61..63 = flow).
 * --------------------------------------------------------------------------------------------- */
typedef struct pvraft_corrfeat_args {
    const float* y1;
    const double* y1_stats;
    const float* gn1_gamma; /* corr_block.out_conv.1.weight [128] */
    const float* gn1_beta;  /* corr_block.out_conv.1.bias   [128] */
    const float* prelu1;    /* corr_block.out_conv.2.weight [1]   */
    const float* w_out;     /* corr_block.out_conv.3.weight [64,128] */
    const float* b_out;     /* corr_block.out_conv.3.bias   [64]  */
    const float* knn_sel;
    const double* moments;
    const float* w_knn;     /* corr_block.knn_conv.0.weight [64,4] */
    const float* b_knn;     /* corr_block.knn_conv.0.bias   [64]   */
    const float* gnk_gamma; /* corr_block.knn_conv.1.weight [64]   */
    const float* gnk_beta;  /* corr_block.knn_conv.1.bias   [64]   */
    const float* preluk;    /* corr_block.knn_conv.2.weight [1]    */
    const float* w_kout;    /* corr_block.knn_out.weight [64,64]   */
    const float* b_kout;    /* corr_block.knn_out.bias   [64]      */
    float* corr_feat;       /* [B,N,64] or NULL */
    const float* corr_in;   /* [B,N,64], used only when y1 == NULL */
    const float* flow;      /* [B,N,3] */
    const float* w_cc; const float* b_cc;   /* update_block.motion_encoder.conv_corr [64,64],[64] */
    const float* w_cf; const float* b_cf;   /* update_block.motion_encoder.conv_flow [64,3],[64]  */
    const float* w_cm; const float* b_cm;   /* update_block.motion_encoder.conv      [61,128],[61] */
    float* motion;          /* [B,N,64] or NULL */
    int B, N;
} pvraft_corrfeat_args;

PVRAFT_API int pvraft_corr_feature_fwd(const pvraft_corrfeat_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * The ALU part of the feature head, for the tcgen05 path (the 1x1 convolutions around it run as pvraft_tc_linear_fwd):
 *   kfeat[b,n,c] = max over the 32 selected candidates of PReLU(GroupNorm(knn_conv.0(f)))      (model/corr.py:86-92)
 *   cflow[b,n,c] = relu(conv_flow(flow))                                                        (model/update.py:17)
 * knn_sel [B,N,32,4] and moments [B,PVRAFT_MOMENTS] come from pvraft_corr_lookup_fwd; the GroupNorm statistics follow
 * from the moments, so no pass over the [B,64,N,32] tensor of the reference is needed.  flow/cflow may be NULL.
 * --------------------------------------------------------------------------------------------- */
typedef struct pvraft_knn_branch_args {
    const float* knn_sel;
    const double* moments;
    const float* w_knn;     /* corr_block.knn_conv.0.weight [64,4] */
    const float* b_knn;     /* corr_block.knn_conv.0.bias   [64]   */
    const float* gnk_gamma; /* corr_block.knn_conv.1.weight [64]   */
    const float* gnk_beta;  /* corr_block.knn_conv.1.bias   [64]   */
    const float* preluk;    /* corr_block.knn_conv.2.weight [1]    */
    float preluk_host;      /* the same slope as known to the host (selects the convex fast path without a device read);
                               NaN = read it from `preluk` (costs one stream synchronisation) */
    float* kfeat;           /* [B,N,64] */
    const float* flow;      /* [B,N,3] or NULL */
    const float* w_cf; const float* b_cf;   /* update_block.motion_encoder.conv_flow [64,3],[64] */
    float* cflow;           /* [B,N,64] or NULL */
    int B, N;
} pvraft_knn_branch_args;

PVRAFT_API int pvraft_knn_branch_fwd(const pvraft_knn_branch_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * ConvGRU.  Replaces model/update.py:31-40 with x = [inp, motion] (update.py:84).
 *   net, inp, motion [B,N,64] -> net_out [B,N,64]   (net_out may alias net)
 * --------------------------------------------------------------------------------------------- */
typedef struct pvraft_gru_args {
    const float* net;
    const float* inp;
    const float* motion;
    const float* w_z; const float* b_z;     /* update_block.gru.convz [64,192],[64] */
    const float* w_r; const float* b_r;     /* update_block.gru.convr */
    const float* w_q; const float* b_q;     /* update_block.gru.convq */
    float* net_out;
    int B, N;
} pvraft_gru_args;

PVRAFT_API int pvraft_gru_fwd(const pvraft_gru_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * SetConv edge stage: per point, over its 32 graph neighbours j:  y_e = P_j - P_i + W_e . (x_j - x_i)
 * (x = point coordinates; x_j - x_i is the graph's edge feature), reduced to per-channel max and min over the neighbours, with the
 * GroupNorm statistics of all N*32*C pre-activation values accumulated.  Replaces the gather +
 * fc1 + (statistics of) gn1 + max-pool of SetConv.forward, model/flot/gconv.py:65-80.
 *   fc1p [B,N,C], nbr [B,N,32] int32 (LOCAL neighbour ids), edge_feats [B,N,32,3] (= graph.edge_feats),
 *   w_fc1 [C,cin+3] (columns cin..cin+2 are read)
 *   -> ymax, ymin [B,N,C]; stats [B,8,2] accumulated.   C % 8 == 0, C <= 128.
 *   order [B,N] int32 or NULL: the LOCAL point processed r-th in every sample (pvraft_point_order_fwd: a Morton rank table).
 *   It changes no result, only which points a CTA works on at the same time, so that their overlapping neighbourhoods are
 *   gathered from L1 instead of L2.
 * --------------------------------------------------------------------------------------------- */
PVRAFT_API int pvraft_setconv_edge_fwd(const float* fc1p, const int32_t* nbr, const float* edge_feats, const float* w_fc1, int cin,
                            int B, int N, int C, float* ymax, float* ymin, double* stats, const int32_t* order, void* stream);

/* ------------------------------------------------------------------------------------------------
 * FlowHead output stage + RAFT coordinate update.  Replaces model/update.py:69,71-72 (conv1, cat,
 * out_conv) after the SetConv's last GroupNorm+LeakyReLU (gconv.py:82-83), and
 * model/RAFTSceneFlow.py:45-46 (coords2 += delta; flow = coords2 - coords1).
 *   z3 [B,N,64] (setconv.fc3 output) + z3_stats, net [B,N,64], coords1/coords2 [B,N,3]
 *   -> delta [B,N,3], coords2_out [B,N,3] (may alias coords2), flow_out [B,N,3] (may be NULL)
 * --------------------------------------------------------------------------------------------- */
typedef struct pvraft_flowout_args {
    const float* z3;
    const double* z3_stats;
    const float* gn3_gamma; const float* gn3_beta; /* setconv.gn3 [64] */
    const float* net;
    const float* w_c1; const float* b_c1;          /* flow_head.conv1 [64,64],[64] */
    const float* w_o0; const float* b_o0;          /* flow_head.out_conv.0 [64,128],[64] */
    const float* w_o2; const float* b_o2;          /* flow_head.out_conv.2 [3,64],[3] */
    const float* coords1;
    const float* coords2;
    float* delta;
    float* coords2_out;
    float* flow_out;
    int B, N;
} pvraft_flowout_args;

PVRAFT_API int pvraft_flow_out_fwd(const pvraft_flowout_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * k nearest neighbours.  Backs knn_point (model/pointconv.py:28-39) and the adjacency of
 * Graph.construct_graph (model/flot/graph.py:53-60, which argsorts a full N x N matrix).
 *   xyz [B,N,3] (candidates), query [B,S,3] -> idx [B,S,k] int32 LOCAL candidate ids, unordered;
 *   rel [B,S,k,3] = xyz[idx] - query (the graph's edge features, graph.py:69-74), or NULL.
 * mode 0: distance = (|q|^2 + |x|^2) - 2 q.x      (graph.py:53-57 op order)
 * mode 1: distance = (-2 q.x + |q|^2) + |x|^2     (pointconv.py:21-24 op order)
 * with q.x = fma(qz,xz, fma(qy,xy, qx*xx)) and |.|^2 = (x*x+y*y)+z*z.  1 <= k <= 32, N >= k.
 * Ties at the k-th place: lowest candidate id.
 * workspace: pvraft_knn_workspace_bytes(B, N) bytes of device scratch (16-byte aligned) enable the
 * uniform-grid search (N <= 16384); with workspace == NULL (or larger N) the brute-force kernel runs.  Both
 * return the same set.
 * --------------------------------------------------------------------------------------------- */
PVRAFT_API int64_t pvraft_knn_workspace_bytes(int B, int N);
PVRAFT_API int pvraft_knn_fwd(const float* xyz, const float* query, int B, int N, int S, int k, int mode, int32_t* idx,
                   float* rel, void* workspace, void* stream);

/* A spatially coherent order of every cloud: perm[b, r] = index of the point that comes r-th along a Morton (Z-order) curve
 * over the cells of the kNN grid.  No counterpart in the reference (point order carries no meaning in model/*.py); the
 * RAFT driver uses it to make the SetConv gathers of consecutive points overlap in L1/L2.  64 <= N <= 16384;
 * workspace: pvraft_knn_workspace_bytes(B, N) bytes. */
PVRAFT_API int pvraft_point_order_fwd(const float* xyz, int B, int N, int32_t* perm, void* workspace, void* stream);

/* ================================================================================================
 * Gradient contract (SURVEY.md section 8b): what tools/engine.py:131-147 differentiates through.
 * The training path runs layer by layer; each backward entry point below pairs with a forward one.
 * Parameter-gradient outputs are ACCUMULATED with atomics into buffers the caller has zeroed.
 * ============================================================================================= */

/* 1x1 convolution (pvraft_linear_fwd without prologue / activation), weight and bias gradient:
 *   x [rows,cin], dy [rows,cout]  ->  dW[o,i] += sum_r dy[r,o] x[r,i]  (row stride dw_ld floats, 0 = cin),  db[o] += sum_r dy[r,o] (or NULL).
 * The data gradient dx = dy . W is pvraft_linear_fwd with the transposed weight.  cin <= 256, cout <= 128. */
PVRAFT_API int pvraft_linear_wgrad(const float* x, const float* dy, int64_t rows, int cin, int cout, float* dW, int dw_ld, float* db,
                        void* stream);

/* GroupNorm(8) + activation backward (model/corr.py:17-18,25-26; model/flot/gconv.py:27-36 via autograd in the reference):
 *   x, dy [B,rows,C]; stats [B,8,2] raw sums of x (as produced in the forward); count = rows * C/8; act/slope as pvraft_gn_act_fwd
 *   -> dx [B,rows,C]; dgamma, dbeta [C] double (accumulated); dslope [1] double (PReLU slope gradient, or NULL);
 *      gsum [B,8,2] double scratch, ZEROED by the caller. */
PVRAFT_API int pvraft_gn_act_bwd(const float* x, const float* dy, const double* stats, const float* gamma, const float* beta, double count,
                      int act, float slope, int B, int64_t rows, int C, double* gsum, double* dgamma, double* dbeta, double* dslope,
                      float* dx, const float* slope_dev, const uint8_t* arg, void* stream);
/* Backward of a linear layer with cin <= 4 and cout in {16,32,48,64,96,128} (the SetConv edge term and the knn_conv: rows = B*N*32) in one
 * pass over dy: dW [cout,dw_ld] += dy^T x, db [cout] += column sums (or NULL), dx [rows,cin] = dy W (or NULL).  W is [cout,w_ld]. */
PVRAFT_API int pvraft_linear_bwd_small(const float* x, const float* dy, const float* W, int64_t rows, int cin, int cout, int w_ld, float* dW,
                            int dw_ld, float* db, float* dx, void* stream);
/* GroupNorm + activation + max over each point's 32 consecutive rows, fused (model/flot/gconv.py:76-80, model/corr.py:87-92):
 *   x [B, pts*32, C] -> y [B,pts,C], arg [B,pts,C] uint8 (first row attaining the maximum); count = pts*32 * C/8.
 * Its backward is pvraft_gn_act_bwd with `arg` set and dy = d y [B,pts,C]: the dense, 31/32-zero gradient of the max is never formed. */
PVRAFT_API int pvraft_gn_act_maxk_fwd(const float* x, const double* stats, const float* gamma, const float* beta, double count, int act,
                           float slope, int B, int64_t pts_per_sample, int C, float* y, uint8_t* arg, const float* slope_dev, void* stream);

/* SetConv edge stage, layer-wise (model/flot/gconv.py:65-73, fc1 factorised as in pvraft_setconv_edge_fwd):
 *   forward : E[b,n,j,:] <- P[b,nbr[b,n,j],:] - P[b,n,:] + E[b,n,j,:]  (in place; E = W_e . edge_feats from pvraft_linear_fwd),
 *             stats [B,8,2] accumulated sums of the result (or NULL)
 *   backward: dP[b,nbr,:] += dT[b,n,j,:]; dP[b,n,:] -= sum_j dT[b,n,j,:]   (dP zeroed by the caller; dE = dT)
 *   P [B,N,C], nbr [B,N,32] int32 local ids, E/dT [B,N,32,C]. */
PVRAFT_API int pvraft_edge_fwd(const float* P, const int32_t* nbr, float* E, int B, int N, int C, double* stats, void* stream);
PVRAFT_API int pvraft_edge_bwd(const float* dT, const int32_t* nbr, int B, int N, int C, float* dP, void* stream);

/* max over the 32 neighbours (model/flot/gconv.py:80, model/corr.py:92): x [pts,32,C] -> y [pts,C], arg [pts,C] uint8 (first
 * maximum); backward writes dx [pts,32,C] = dy at arg, 0 elsewhere. */
PVRAFT_API int pvraft_maxk_fwd(const float* x, int64_t pts, int C, float* y, uint8_t* arg, void* stream);
PVRAFT_API int pvraft_maxk_bwd(const float* dy, const uint8_t* arg, int64_t pts, int C, float* dx, void* stream);

/* Backward of pvraft_corr_lookup_fwd w.r.t. corr_val (model/corr.py:47-66,84; indices and coordinates carry no gradient:
 * corr.py:52-62 is under no_grad and RAFTSceneFlow.py:41 detaches the coordinates):
 *   g_vox [B,N,vox_ld], g_sel [B,N,32,4] (channel 0 used), knn_slot [B,N,32] from the forward -> d_corr [B,N,K] (overwritten). */
PVRAFT_API int pvraft_corr_lookup_bwd(const int32_t* corr_idx, const float* xyz2_pad, const float* coords, const int32_t* knn_slot,
                           const float* g_vox, int vox_ld, const float* g_sel, int B, int N, int K, int levels, float base_scale,
                           float* d_corr, void* stream);

/* Backward of the truncated correlation (model/corr.py:95-100 + the top-k gather of :37-38), sparse over the K kept entries:
 *   g [B,N,K], idx [B,N,K] (same stored order), fmap1/fmap2 [B,N,C] point-major
 *   -> d_fmap1 [B,N,C] (overwritten), d_fmap2 [B,N,C] (ACCUMULATED, zeroed by the caller).  C in {32,64,128,256}. */
PVRAFT_API int pvraft_corr_init_bwd(const float* g, const int32_t* idx, const float* fmap1, const float* fmap2, int B, int N, int C, int K,
                         float* d_fmap1, float* d_fmap2, void* stream);

/* Training extras on the device (SURVEY.md 8f row f3).  est, gt [points,3]; mask [points] (> 0 = valid) or NULL.
 *   pvraft_flow_metrics_fwd: acc[6] double, ZEROED by the caller, accumulates over the valid points
 *       [0] sum |ex|+|ey|+|ez|  (tools/loss.py:34-38: loss = acc[0] / (3 acc[1]))      [1] number of valid points
 *       [2] sum ||e||           (tools/metric.py:24-29: EPE = acc[2] / acc[1])
 *       [3],[4],[5] points with (epe<.05 or rel<.05), (epe<.1 or rel<.1), (epe>.3 or rel>.1), rel = epe/(||gt||+1e-4)  (metric.py:66-77)
 *   pvraft_flow_l1_bwd: d_est = g[0] * weight * sign(est - gt) / (3 acc[1]) on valid points, 0 elsewhere; g is a DEVICE scalar
 *       (the upstream gradient), acc the forward's accumulator: no host synchronisation between forward and backward. */
PVRAFT_API int pvraft_flow_metrics_fwd(const float* est, const float* gt, const float* mask, int64_t points, double* acc, void* stream);
PVRAFT_API int pvraft_flow_l1_bwd(const float* est, const float* gt, const float* mask, int64_t points, const double* acc, const float* g,
                       float weight, float* d_est, void* stream);

/* sizeof() of the argument structs as compiled into the library (0 = linear, 1 = corrfeat, 2 = gru,
 * 3 = flowout, 4 = tc_linear; -1 otherwise): lets a foreign-language binding verify its struct layout at load time. */
PVRAFT_API int pvraft_sizeof(int which);

/* [B,C,N] <-> [B,N,C] transposes used at the reference-layout seams of the Python modules. */
PVRAFT_API int pvraft_transpose_fwd(const float* in, int B, int R, int C, float* out, void* stream); /* [B,R,C] -> [B,C,R] */

#ifdef __cplusplus
}
#endif
#endif /* PVRAFT_B200_H */
