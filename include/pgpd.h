/* pgpd.h -- C ABI of libpgpd.so: the B200-native PointNet grasp-quality hot path.
 *
 * This is the drop-in boundary for ONE path of lianghongzhuo/PointNetGPD:
 *   STN3d.forward         PointNetGPD/model/pointnet.py:27-45
 *   PointNetfeat.forward  PointNetGPD/model/pointnet.py:137-151   (global_feat=True)
 *   PointNetCls.forward   PointNetGPD/model/pointnet.py:189-194
 * and the autograd backward of those three (driven by main_1v.py:72-75).
 * The reference has no FFI of its own (it is pure torch.nn); the entry points below are
 * what a ctypes binding inside model/pointnet.py binds instead of the torch.nn op chain
 * (see INTEGRATION.md for the stub).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to contiguous fp32 (int64 where stated);
 *     the caller owns all memory, the library never allocates, never synchronises,
 *     never changes the current device and keeps no global mutable state (re-entrant:
 *     nn.DataParallel calls it from one thread per device, main_1v.py:163-165);
 *   - `stream` is a cudaStream_t passed as void*;
 *   - functions return 0 on success or a negative PGPD_E_* code; the message of the last
 *     error on the calling thread is pgpd_last_error();
 *   - x is [B,3,N] channel-major exactly as the reference model receives it
 *     (main_1v.py:69-73: data.float() of shape [B,3,N]);
 *   - weights use the reference parameter layout: Conv1d(k=1) weight [out,in,1] and
 *     Linear weight [out,in], both row-major [out][in]; conv / fc weight pointers must be
 *     16-byte aligned (PGPD_E_ARG otherwise).
 */
#ifndef PGPD_H_
#define PGPD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGPD_VERSION 100          /* 0.1.0 */

/* ---- error codes ------------------------------------------------------------------ */
#define PGPD_OK            0
#define PGPD_E_ARG        -1      /* bad argument (null pointer, B<1, N<1, k<1, ...)          */
#define PGPD_E_WORKSPACE  -2      /* workspace too small / misaligned                          */
#define PGPD_E_BATCH1     -3      /* train mode with one value per channel: the reference's    *
                                   * BatchNorm raises ValueError there (torch _verify_batch_size) */
#define PGPD_E_CUDA       -4      /* a CUDA runtime call or kernel launch failed               */
#define PGPD_E_UNSUPPORTED -5

/* ---- which module is being evaluated (the three reference nn.Modules) -------------- */
#define PGPD_STN   1              /* STN3d:        x -> trans[B,3,3]                           */
#define PGPD_FEAT  2              /* PointNetfeat: x -> (G[B,1024], trans)                     */
#define PGPD_CLS   3              /* PointNetCls:  x -> (logp[B,k], trans)                     */

/* ---- flags -------------------------------------------------------------------------- */
#define PGPD_F_TRAIN   0x1        /* module.training: batch statistics + running-stat update   */
#define PGPD_F_SAVE    0x2        /* keep what pgpd_backward needs in the workspace            */
#define PGPD_F_SIMT    0x100      /* force the fp32 CUDA-core kernels (no tcgen05); debugging  */
/* pgpd_backward in two calls, so that a data-parallel caller can start the gradient exchange of the first half while the
 * second half is still being computed (main_1v.py:163-165 wraps the model in nn.DataParallel; DESIGN.md section 7):
 *   PGPD_F_BWD_HEAD : classifier head + trunk tower (+ the gradient reaching the T-Net output); needs dout
 *   PGPD_F_BWD_STN  : T-Net head + T-Net tower; must follow a PGPD_F_BWD_HEAD call on the same workspace
 * neither bit (or both): the whole backward in one call.  Only meaningful for PGPD_FEAT / PGPD_CLS. */
#define PGPD_F_BWD_HEAD 0x10
#define PGPD_F_BWD_STN  0x20

/* nn.Conv1d(k=1) / nn.Linear (pointnet.py:12-18,127-129,182-184) */
typedef struct pgpd_lin {
    const float* w;               /* [out][in] */
    const float* b;               /* [out]     */
} pgpd_lin;

/* nn.BatchNorm1d, eps=1e-5, momentum=0.1 (pointnet.py:21-25,130-132,185-186) */
typedef struct pgpd_bn {
    const float* gamma;           /* weight [C]                                                 */
    const float* beta;            /* bias   [C]                                                 */
    float* running_mean;          /* [C]  updated in place when PGPD_F_TRAIN                    */
    float* running_var;           /* [C]  updated in place when PGPD_F_TRAIN (unbiased)         */
    int64_t* num_batches_tracked; /* scalar, += 1 when PGPD_F_TRAIN; may be NULL                */
} pgpd_bn;

/* shared-MLP tower 3->64->128->1024 + global max-pool (pointnet.py:29-33 / :144-149) */
typedef struct pgpd_tower {
    pgpd_lin conv[3];
    pgpd_bn  bn[3];
} pgpd_tower;

/* FC head 1024->512->256->out (pointnet.py:35-37 / :191-193) */
typedef struct pgpd_head {
    pgpd_lin fc[3];
    pgpd_bn  bn[2];
} pgpd_head;

/* PointNetCls = feat.stn (tower+head) , feat (tower) , classifier head */
typedef struct pgpd_model {
    pgpd_tower stn_tower;         /* feat.stn.conv1-3 / bn1-3   */
    pgpd_head  stn_head;          /* feat.stn.fc1-3  / bn4-5    (out = 9)                        */
    pgpd_tower trunk;             /* feat.conv1-3 / feat.bn1-3                                  */
    pgpd_head  cls_head;          /* fc1-3 / bn1-2              (out = k)                        */
} pgpd_model;

/* gradient outputs, same shapes as the parameters; every pointer is written (not accumulated) */
typedef struct pgpd_lin_grad { float* dw; float* db; } pgpd_lin_grad;
typedef struct pgpd_bn_grad  { float* dgamma; float* dbeta; } pgpd_bn_grad;
typedef struct pgpd_tower_grad { pgpd_lin_grad conv[3]; pgpd_bn_grad bn[3]; } pgpd_tower_grad;
typedef struct pgpd_head_grad  { pgpd_lin_grad fc[3];   pgpd_bn_grad bn[2]; } pgpd_head_grad;
typedef struct pgpd_model_grad {
    pgpd_tower_grad stn_tower;
    pgpd_head_grad  stn_head;
    pgpd_tower_grad trunk;
    pgpd_head_grad  cls_head;
} pgpd_model_grad;

/* library version (PGPD_VERSION of the build) */
int pgpd_version(void);

/* message of the last failure on this thread ("" if none) */
const char* pgpd_last_error(void);

/* 1 if the library was built with the tcgen05 (sm_100a tensor-core) kernels */
int pgpd_has_tensor_core_path(void);

/* Kernels launched by this library from the calling thread since it was loaded. */
unsigned long long pgpd_launch_count(void);

/* Optional timing of the dominant kernel (the layer-3 GEMM + max-pool of a tower forward):
 * pgpd_profile_enable(1) makes every following launch of that kernel on the calling thread record
 * a CUDA-event pair on its stream; pgpd_profile_read synchronises those events, returns the number
 * of launches and their summed duration, and resets the accumulator.
 * pgpd_profile_enable(2): "sticky" mode for CUDA graphs -- launches made while the stream is being captured record
 * external event nodes into the graph, every replay re-records them, and pgpd_profile_read (which then does not
 * reset) returns the durations of the most recent replay. */
int pgpd_profile_enable(int on);
int pgpd_profile_read(int* launches, float* total_ms);

/* Bytes of workspace pgpd_forward/pgpd_backward need for (what,B,N,k,flags).  The same
 * buffer must be handed, untouched, from pgpd_forward(PGPD_F_SAVE) to pgpd_backward. */
size_t pgpd_workspace_bytes(int what, int B, int N, int k, int flags);

/* Forward of STN3d / PointNetfeat / PointNetCls.
 *   out   : PGPD_CLS  -> logp [B,k]   (log_softmax, pointnet.py:194)
 *           PGPD_FEAT -> G    [B,1024] (pointnet.py:148-151)
 *           PGPD_STN  -> ignored (may be NULL)
 *   trans : [B,3,3] (pointnet.py:37-44); always written
 * Only the sub-structs of `m` the module uses are read (PGPD_STN: stn_tower+stn_head;
 * PGPD_FEAT: + trunk; PGPD_CLS: all). */
int pgpd_forward(int what, const pgpd_model* m, const float* x, int B, int N, int k, int flags,
                 float* out, float* trans, void* workspace, size_t workspace_bytes, void* stream);

/* Backward of the same module, after pgpd_forward(..., PGPD_F_TRAIN|PGPD_F_SAVE, ...) with the
 * same (what,m,x,B,N,k) and workspace.
 *   dout   : gradient w.r.t. `out`  (PGPD_STN: NULL)
 *   dtrans : gradient w.r.t. `trans` [B,3,3], or NULL for zero
 * Writes every gradient of `g` the module owns.  The input x gets no gradient (no reference
 * script asks for one: main_1v.py:69-75). */
int pgpd_backward(int what, const pgpd_model* m, const pgpd_model_grad* g, const float* x,
                  int B, int N, int k, int flags, const float* dout, const float* dtrans,
                  void* workspace, size_t workspace_bytes, void* stream);

/* ---- tower-level entry points (same kernels; used by the parity tests and benchmarks) ---
 * pooled[B,1024] = maxpool_N( [relu]( bn3(conv3( relu(bn2(conv2( relu(bn1(conv1( T^T x ))))))))))
 *   trans      : [B,3,3] or NULL (identity)           (pointnet.py:140-143)
 *   relu_last  : 1 for STN3d (pointnet.py:31), 0 for PointNetfeat (pointnet.py:147)          */
size_t pgpd_tower_workspace_bytes(int B, int N, int flags);
int pgpd_tower_forward(const pgpd_tower* t, const float* x, const float* trans, int B, int N,
                       int relu_last, int flags, float* pooled,
                       void* workspace, size_t workspace_bytes, void* stream);
/* dtrans_out: [B,3,3] gradient w.r.t. trans (written only if trans != NULL), may be NULL */
int pgpd_tower_backward(const pgpd_tower* t, const pgpd_tower_grad* g, const float* x,
                        const float* trans, int B, int N, int relu_last, int flags,
                        const float* dpooled, float* dtrans_out,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- GPDClassifier, the paper's baseline CNN (PointNetGPD/model/gpd.py:5-31; SURVEY.md section 8f row 4) ---------------------
 *   x [B][C][60][60] -> conv1(C->20,5x5) -> maxpool2 -> conv2(20->50,5x5) -> maxpool2 -> fc1(7200->500)+ReLU -> fc2(500->2)
 *   -> log_softmax.  Weights in the reference layouts: Conv2d [out][in][5][5], Linear [out][in] (fc1.w 16-byte aligned).
 *   The optional Dropout2d of the reference (if_dropout=True, training) draws from torch's RNG stream and is not provided.
 *   pgpd_gpd_forward(..., PGPD_F_SAVE) keeps what pgpd_gpd_backward needs in the workspace. */
typedef struct pgpd_gpd { pgpd_lin conv1, conv2, fc1, fc2; } pgpd_gpd;
typedef struct pgpd_gpd_grad { pgpd_lin_grad conv1, conv2, fc1, fc2; } pgpd_gpd_grad;
size_t pgpd_gpd_workspace_bytes(int B, int C, int flags);
int pgpd_gpd_forward(const pgpd_gpd* m, const float* x, int B, int C, int flags, float* logp,
                     void* workspace, size_t workspace_bytes, void* stream);
int pgpd_gpd_backward(const pgpd_gpd* m, const pgpd_gpd_grad* g, const float* x, int B, int C, int flags,
                      const float* dlogp, void* workspace, size_t workspace_bytes, void* stream);

/* ---- the dual-cloud network (PointNetGPD/model/pointnet.py:48-120,157-174; SURVEY.md section 8f row 4) ---------------------------
 *   PGPD_DUAL_STN  : SimpleSTN3d        x [B,3,N] -> trans [B,3,3]          tower 3->64->128->256, head 256->128->64->9 (+ I)
 *   PGPD_DUAL_FEAT : DualPointNetfeat   x [B,6,N] -> (G [B,1024], trans1 + trans2): one SimpleSTN3d per 3-channel half, each half
 *                                       transformed by its own T-Net, trunk 6->64->128->1024 (no ReLU before the pool)
 *   PGPD_DUAL_CLS  : DualPointNetCls    x [B,6,N] -> (logp [B,k], trans1 + trans2)
 * The tower / head structs are the ones above with this network's widths (stn*_tower.conv[2].w is [256][128], stn*_head.fc[0].w
 * [128][256], trunk.conv[0].w [64][6], ...).  PGPD_DUAL_STN reads stn1_* only.  fp32 CUDA-core kernels (csrc/dual.cuh); flags as for
 * pgpd_forward (PGPD_F_TRAIN, PGPD_F_SAVE).  No reference script constructs these classes. */
#define PGPD_DUAL_STN  11
#define PGPD_DUAL_FEAT 12
#define PGPD_DUAL_CLS  13
typedef struct pgpd_dual {
    pgpd_tower stn1_tower; pgpd_head stn1_head;       /* feat.stn1.*                                   */
    pgpd_tower stn2_tower; pgpd_head stn2_head;       /* feat.stn2.*                                   */
    pgpd_tower trunk;                                 /* feat.conv1-3 / feat.bn1-3                     */
    pgpd_head  cls_head;                              /* fc1-3 / bn1-2                                 */
} pgpd_dual;
typedef struct pgpd_dual_grad {
    pgpd_tower_grad stn1_tower; pgpd_head_grad stn1_head;
    pgpd_tower_grad stn2_tower; pgpd_head_grad stn2_head;
    pgpd_tower_grad trunk;
    pgpd_head_grad  cls_head;
} pgpd_dual_grad;
size_t pgpd_dual_workspace_bytes(int what, int B, int N, int k, int flags);
/*   out : PGPD_DUAL_CLS -> logp [B,k]; PGPD_DUAL_FEAT -> G [B,1024]; PGPD_DUAL_STN -> ignored;   trans: [B,3,3], always written */
int pgpd_dual_forward(int what, const pgpd_dual* m, const float* x, int B, int N, int k, int flags,
                      float* out, float* trans, void* workspace, size_t workspace_bytes, void* stream);
/*   after pgpd_dual_forward(..., PGPD_F_TRAIN | PGPD_F_SAVE, ...) on the same workspace; dout: gradient w.r.t. out (PGPD_DUAL_STN:
 *   NULL), dtrans: gradient w.r.t. trans or NULL for zero (PGPD_DUAL_STN: required).  Writes every gradient the module owns. */
int pgpd_dual_backward(int what, const pgpd_dual* m, const pgpd_dual_grad* g, const float* x, int B, int N, int k, int flags,
                       const float* dout, const float* dtrans, void* workspace, size_t workspace_bytes, void* stream);

/* ---- data preparation in front of the model (SURVEY.md section 8f rows 1-2) ------------------------------------
 * Gripper-box crop of one cloud for G grasps (BaseGraspDataset.collect_pc, PointNetGPD/model/dataset.py:51-76;
 * kinect2grasp.py:178-235).
 *   pc      : [P][3] fp32 cloud points (row-major, as the reference's numpy arrays)
 *   frames  : [G][15] fp64 per grasp: center[3], rotation rows (approach, binormal, minor_normal)[9], half extents
 *             (x,y,z)[3] -- the quantities dataset.py:16-59 derives from the 12-float grasp row on the host
 *   counts  : [G] number of points inside each box, or NULL
 *   offsets : [G] start of each grasp's output segment (exclusive prefix sum of counts); needed with out_*
 *   out_pts : [sum][3] fp32 local coordinates of the inside points, ascending cloud index; out_idx: their indices
 * Call once with counts only, prefix-sum on the host, call again with offsets + outputs.  Arithmetic is fp64 like
 * numpy in the reference, so the selected index sets are identical. */
int pgpd_crop_box(const float* pc, int P, const double* frames, int G, const int* offsets, int* counts,
                  float* out_pts, int* out_idx, void* stream);

/* Resample C point sets (concatenated in pts [total][3], delimited by offsets [C+1]) to exactly N points each,
 * `repeat` independent draws (dataset.py:438-444; kinect2grasp.py:473-478): a uniformly random subset of N distinct
 * points when the set has >= N points, N uniform draws with replacement otherwise.  Deterministic in `seed`.
 *   out_x   : [C*repeat][3][N] fp32, channel-major = the model's input layout;  out_idx: [C*repeat][N] or NULL */
int pgpd_resample(const float* pts, const int* offsets, int C, int N, int repeat, unsigned long long seed,
                  float* out_x, int* out_idx, void* stream);

/* GPD image projection (BaseGraspDataset.project_pc / cal_projection, PointNetGPD/model/dataset.py:78-198) of one cloud
 * for G grasps, after pgpd_crop_box:
 *   pc, frames       : as for pgpd_crop_box
 *   offsets, idx     : [G+1] segment bounds and [offsets[G]] ascending cloud indices of the in-box points (pgpd_crop_box)
 *   chann            : 3 (normals of the [x,y,z] image) or 12 ([occupancy, normal] of the orders [0,1,2], [1,2,0], [0,2,1])
 *   out              : [G][chann][60][60] fp32, the layout pgpd_gpd_forward reads (out[c][y][x] = the reference's
 *                      image[x][y][c]); all zeros for a grasp with fewer than 50 in-box points
 *   valid            : [G] bytes, 1 where the box holds >= 50 points (the reference's item is None otherwise)
 * Normals: up to 30 nearest cloud points within distance 0.1 (itself included), covariance in the grasp frame (fp64),
 * eigenvector of the smallest eigenvalue from the closed-form symmetric 3x3 solver; fewer than 3 neighbours or a zero
 * covariance give (0,0,1).  Deterministic: the same inputs give bit-identical outputs.
 * The workspace (256-byte aligned) comes from pgpd_gpd_project_workspace_bytes(P, G, offsets[G], chann); a grasp whose
 * points lie beyond what the given workspace holds is written as NaN with valid = 0. */
size_t pgpd_gpd_project_workspace_bytes(int P, int G, int total_in_box, int chann);
int pgpd_gpd_project(const float* pc, int P, const double* frames, int G, const int* offsets, const int* idx, int chann,
                     float* out, unsigned char* valid, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PGPD_H_ */
