/*
 * casapose_b200 — C ABI of the B200-native (sm_100a) keypoint-voting hot path.
 *
 * The reference (fraunhoferhhi/casapose) has no FFI / plugin / custom-op interface: the
 * boundary of this path is plain Python taking tf.Tensors.  Every entry point below
 * therefore cites the reference PYTHON interface it stands behind; the Python package
 * casapose_b200.pose_estimation keeps those names and signatures and hands raw device
 * pointers (obtained through DLPack) to this library via ctypes.  INTEGRATION.md shows
 * the binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative casa_status; the message of the
 *     last failure on the calling thread is casa_last_error().  No exception crosses.
 *   - all tensors are dense, C-contiguous, float32 NHWC exactly like the reference's
 *     tensors; the caller owns inputs and outputs, the library never frees them.
 *     The *_typed entry points also read the network outputs (mask / seg, vertex, direct,
 *     conf) as float16 or bfloat16 (casa_dtype); outputs and gradients stay float32.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *   - a handle is bound to one device, owns the workspace, and is not thread-safe;
 *     use one handle per stream / thread.
 */
#ifndef CASAPOSE_B200_H_
#define CASAPOSE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CASA_VERSION 100

typedef enum casa_status {
  CASA_OK = 0,
  CASA_ERR_INVALID = -1,    /* bad shape / argument */
  CASA_ERR_CUDA = -2,       /* a CUDA runtime call failed */
  CASA_ERR_WORKSPACE = -3,  /* pixel lists do not fit pix_capacity (mask is not one-hot) */
  CASA_ERR_INPUT = -4,      /* device-side input check failed (idx out of range, ...) */
  CASA_ERR_NODEVICE = -5
} casa_status;

/* Bits of the device status word (debug.status / casa_last_status). */
#define CASA_STATUS_MASK_NOT_BINARY 1u  /* a mask value other than 0 or 1 was seen          */
#define CASA_STATUS_PIX_OVERFLOW 2u     /* sum_c tn0 > pix_capacity for some image            */
#define CASA_STATUS_IDX_RANGE 4u        /* a caller-supplied idx was outside [0, tn)          */
#define CASA_STATUS_EMPTY_AFTER_CAP 8u  /* the max_num down-sampling removed every pixel      */
#define CASA_STATUS_LS_NONFINITE 16u    /* CoordLSVotingWeighted produced a non-finite R/q/p  */

typedef struct casa_handle casa_handle;

/*
 * Element type of a network output read by the *_typed entry points.  Each 16-bit element is widened exactly to
 * float32 when it is loaded and everything after the load is the float32 path, so every output (keypoints, debug
 * intermediates, status bits, gradients) is bit-identical to the float32 call on the upcast tensor.
 */
typedef enum casa_dtype { CASA_FLOAT32 = 0, CASA_FLOAT16 = 1, CASA_BFLOAT16 = 2 } casa_dtype;

int casa_version(void);
const char* casa_last_error(void);

/* One handle per device/stream user.  device < 0 selects the current device. */
int casa_create(int device, casa_handle** out);
int casa_destroy(casa_handle* h);

/*
 * Parameters of ransac_voting_layer_all_masks
 * (/root/reference/casapose/pose_estimation/ransac_voting.py:446-484; same names,
 * same defaults: inlier_thresh=0.99, confidence=0.99, max_iter=20, min_num=5,
 * max_num=30000; round_hyp_num is 512 at the reference's call sites,
 * pose_evaluation.py:50-58).
 */
typedef struct casa_ransac_params {
  int32_t b, h, w;        /* batch, image height, image width                               */
  int32_t oc;             /* object classes (mask channels), 1..32                          */
  int32_t vn;             /* keypoints per object (vertex is [b,h,w,vn,2]), 1..16            */
  int32_t round_hyp_num;  /* hypotheses per round (hn), 1..4096                             */
  int32_t max_iter;       /* 1..64                                                          */
  float inlier_thresh;
  float confidence;
  float min_num;
  float max_num;
  uint64_t seed;          /* Philox4x32-10 key (csrc/philox.cuh); stands in for tf.random   */
  int32_t image_offset;   /* global index of image 0 (so a sharded batch draws the same     */
                          /* random numbers as the unsharded one)                           */
  int32_t pix_capacity;   /* per-image pixel-list capacity; 0 = h*w (enough for one-hot)    */
  int32_t force_exact;    /* 1 = disable the filtered predicate (tests only)                */
  int32_t vertex_per_class; /* 0: vertex is [b,h,w,vn,2]; 1: [b,h,w,oc,vn,2] (PVNet-style, one field per class;  */
                            /* pose_evaluation.py:38-45 gathers the arg-max class's vectors)              */
} casa_ransac_params;

/*
 * Optional per-call debug outputs (device pointers, any may be NULL).  These are the
 * intermediates of ransac_voting_batch (ransac_voting.py:275-368) the parity tests compare.
 */
typedef struct casa_ransac_debug {
  int32_t* tn0;      /* [b,oc]                 foreground_num                       :287 */
  int32_t* tn;       /* [b,oc]                 pixels after the max_num cap         :310 */
  int32_t* rounds;   /* [b,oc]                 cur_iter at loop exit                :341 */
  int32_t* counts;   /* [b,oc,max_iter,hn,vn]  cur_inlier_counts per round          :327 */
  int32_t* win_idx;  /* [b,oc,max_iter,vn]     cur_win_idx per round                :328 */
  float* hyps;       /* [b,oc,max_iter,hn,vn,2] cur_hyp_pts per round               :322 */
  float* win_pts;    /* [b,oc,vn,2]            all_win_pts at loop exit             :337 */
  float* win_ratio;  /* [b,oc,vn]              all_win_ratio at loop exit           :338 */
  float* ata;        /* [b,oc,vn,3]            ATA (xx, xy, yy)                     :361 */
  float* atb;        /* [b,oc,vn,2]            ATb                                  :362 */
  int32_t* refined;  /* [b,oc]                 1 if every ATA was invertible        :364 */
  uint32_t* pix;     /* [b,pix_capacity]       compacted pixel lists (y<<16|x)      :303 */
  int32_t* pix_off;  /* [b,oc]                 start of each class list inside pix       */
  uint64_t* stats;   /* [4] filter statistics: units scored, units sent to the exact     */
                     /*     predicate, exact-list hypotheses, tiles scored exactly        */
} casa_ransac_debug;

/* Bytes of device workspace the handle will hold for these shapes (grown on demand). */
size_t casa_ransac_workspace_bytes(const casa_ransac_params* p);

/*
 * ransac_voting_layer_all_masks(mask, vertex, round_hyp_num, ...) -> [b,oc,vn,2] (x,y) px.
 *   mask      device float32 [b,h,w,oc]   values in {0,1}
 *   vertex    device float32 [b,h,w,vn,2] (dy,dx) per keypoint
 *   idxs      optional device int32 [b,oc,max_iter,hn,vn,2] pixel-pair indices in [0,tn)
 *             (NULL = draw them from the Philox stream)           ransac_voting.py:319
 *   selection optional device float32 [b,oc,h,w] in [0,1)          ransac_voting.py:296
 *   out_points device float32 [b,oc,vn,2]
 * Asynchronous on `stream` except for one 4-byte read-back per RANSAC round (the
 * reference's data-dependent `while`, ransac_voting.py:318-347).
 */
int casa_ransac_vote(casa_handle* h, const casa_ransac_params* p, const float* mask,
                     const float* vertex, const int32_t* idxs, const float* selection,
                     float* out_points, const casa_ransac_debug* debug, void* stream);

/*
 * Fused pre-step of estimate_and_evaluate_poses / pose_estimation
 * (/root/reference/casapose/pose_estimation/pose_evaluation.py:36-47, 241-252):
 *   mask = one_hot(argmax(output_seg, 3))[..., 1:]   without materialising the float one-hot.
 *   seg  device float32 [b,h,w,1+oc] segmentation scores (arg-max takes the first maximum)
 */
int casa_ransac_vote_seg(casa_handle* h, const casa_ransac_params* p, const float* seg,
                         const float* vertex, const int32_t* idxs, const float* selection,
                         float* out_points, const casa_ransac_debug* debug, void* stream);

/*
 * casa_ransac_vote (mask_is_seg == 0) or casa_ransac_vote_seg (mask_is_seg != 0) with the mask / seg scores and the
 * vector field in any casa_dtype, each with its own (a float32 one-hot mask with a bfloat16 field is fine).
 * casa_ransac_vote and casa_ransac_vote_seg are the CASA_FLOAT32 case of this call.  idxs, selection and out_points
 * keep their types.  Alignment only picks the load width: the mask's 128-bit loads need a 16-byte aligned base and
 * (h*w*oc) % (16 / element size) == 0, the fused direction gather a vertex aligned to one (dy, dx) pair.
 */
int casa_ransac_vote_typed(casa_handle* h, const casa_ransac_params* p, int mask_is_seg, casa_dtype mask_dtype,
                           const void* mask, casa_dtype vertex_dtype, const void* vertex, const int32_t* idxs,
                           const float* selection, float* out_points, const casa_ransac_debug* debug, void* stream);

/*
 * Same call with HOST buffers; returns after out_points is on the host.
 * Pinned (page-locked, device-mapped) buffers take the fast path: the mask is DMA-copied in up to 4 image
 * ranges on a copy stream while the previous range is voted on, and the vector field is NOT copied — the
 * gather kernel reads only the masked pixels' rows from the mapped host buffer (about 200 MB instead of
 * 511 MB over PCIe for sixteen 480x640 frames).  Pageable buffers are staged in one piece.
 */
int casa_ransac_vote_host(casa_handle* h, const casa_ransac_params* p, const float* mask_host,
                          const float* vertex_host, float* out_points_host);

/*
 * The host-buffer call with several calls in flight, for callers that stream batches — the evaluation loop of
 * /root/reference/test_casapose.py:439-443 calls ransac_voting_layer_all_masks (pose_evaluation.py:50-58) once
 * per batch and looks at the keypoints afterwards.  casa_ransac_vote_host_async hands the call to a driver
 * thread of the handle and returns a ticket at once; casa_host_wait(ticket) blocks until that call's keypoints
 * are in out_points_host and returns its error code (casa_last_error() holds its message).  Two calls run at a
 * time (CASA_HOST_DEPTH=1..4): the host threads pack the mask of call i+1 while the GPU votes on the last image
 * ranges of call i.  A third call waits inside casa_ransac_vote_host_async for the oldest one.  The buffers of
 * a call must stay valid and untouched until its ticket has been waited for; results are bit-identical to
 * casa_ransac_vote_host.  casa_sync() waits for every call in flight and reports the first error of a call
 * nobody waited for.
 */
int casa_ransac_vote_host_async(casa_handle* h, const casa_ransac_params* p, const float* mask_host,
                                const float* vertex_host, float* out_points_host, int64_t* ticket);
int casa_host_wait(casa_handle* h, int64_t ticket);

/*
 * CoordLSVotingWeighted(name, num_classes, num_points, sigmoid_weights, filter_estimates,
 * output_second_largest_component)([seg, direct, w])
 * (/root/reference/casapose/pose_estimation/voting_layers_2d.py:5-122).
 *   seg     device float32 [b,h,w,num_classes]   segmentation logits (class 0 = background)
 *   direct  device float32 [b,h,w,2*vn]          (dy,dx) per keypoint
 *   conf    device float32 [b,h,w,vn]            confidence logits
 *   out     device float32 [b,num_classes-1,vn,2]  (y,x) pixels            voting_layers_2d.py:122
 * Fully asynchronous on `stream` unless check_finite is set (one 32-byte read-back that stands in
 * for the reference's tf.Assert on non-finite R / q / p, :109-121 -> CASA_ERR_INPUT).
 * casa_ls_vote and casa_ls_vote_backward accept any 4-byte-aligned float buffer for seg, direct, conf, out,
 * grad_points, grad_direct and grad_conf (e.g. a contiguous view that starts one float into an allocation, or a
 * DLPack export with a byte offset); wider vector loads are used only where the pointer allows them.  The
 * debug buffers (casa_ls_debug) need their element type's natural alignment.  The *_typed variants take seg,
 * direct and conf in one casa_dtype (they are splits of one network output), each aligned to one element.
 */
typedef struct casa_ls_params {
  int32_t b, h, w;
  int32_t num_classes;       /* 1 + object classes, 2..33                                   */
  int32_t vn;                /* num_points, 1..16                                           */
  int32_t sigmoid_weights;   /* 0: softplus (:35), 1: sigmoid (:33)                         */
  int32_t filter_estimates;  /* keep only the selected connected component (:43-79)         */
  int32_t second_largest;    /* output_second_largest_component (:58-73)                    */
  int32_t min_component;     /* 0 = the reference's 50 (:66)                                */
  int32_t check_finite;      /* 1: synchronise, raise on non-finite results (the reference's tf.Assert :109-121) and retry   */
                             /*    a pixel-list overflow with the measured capacity; 0: fully asynchronous, both conditions */
                             /*    are reported by casa_sync                                                                */
  int32_t pix_capacity;      /* slots per image of the pixel lists; 0 = h*w.  A pixel is listed once per class whose        */
                             /* softmax(1e6 seg) is non-zero, so near-tied logits need more than h*w (up to oc*h*w)         */
} casa_ls_params;

typedef struct casa_ls_debug {
  double* sums;       /* [b,oc,vn,5]  float64 sums R00, R01, R11, q0, q1               :113-114 */
  uint8_t* labels;    /* [b,h,w]      class whose int(hot + 0.1) is 1, else 0          :44      */
  int32_t* selected;  /* [b,oc]       root pixel of the kept component, -1 none, -2 label 0 :72-76 */
  int32_t* parent;    /* [b,h,w]      component root of every labelled pixel            :53      */
  int32_t* tn;        /* [b,oc]       pixels with hot != 0                                       */
} casa_ls_debug;

int casa_ls_vote(casa_handle* h, const casa_ls_params* p, const float* seg, const float* direct,
                 const float* conf, float* out_points, const casa_ls_debug* debug, void* stream);
int casa_ls_vote_typed(casa_handle* h, const casa_ls_params* p, casa_dtype dtype, const void* seg, const void* direct,
                       const void* conf, float* out_points, const casa_ls_debug* debug, void* stream);
/*
 * casa_ls_vote_typed, and the object availability count of poses_pnp taken from the same softmax
 * (/root/reference/casapose/pose_estimation/pose_evaluation.py:183-190):
 *   hot_counts  device int32 [b,num_classes-1]  pixels with softmax(1e6 seg)[..., c] > 0.1 (float32), c >= 1
 * must not be NULL.  out_points and the debug outputs are those of casa_ls_vote_typed, bit for bit.
 * hot_counts is zeroed and written inside the call, ordered like out_points: on `stream`, or on the lanes of
 * casa_set_async(h, n), after casa_join / casa_sync.
 */
int casa_ls_vote_counts(casa_handle* h, const casa_ls_params* p, casa_dtype dtype, const void* seg, const void* direct,
                        const void* conf, float* out_points, int32_t* hot_counts, const casa_ls_debug* debug, void* stream);

/*
 * Backward of CoordLSVotingWeighted w.r.t. `direct` and the confidence logits (SURVEY.md 8f-4) — what TF's
 * autodiff produces for the layer inside the training step (/root/reference/train_casapose.py:536-595);
 * `seg` is behind tf.stop_gradient (voting_layers_2d.py:37) and receives no gradient.  Re-runs the forward
 * (stateless), then the closed-form adjoint of the 2x2 pseudo-inverse solve and one pass over the listed pixels.
 *   grad_points device float32 [b,oc,vn,2]   dL/d(output), (y,x) order like the output
 *   out_points  device float32 [b,oc,vn,2]   forward result, or NULL
 *   grad_direct device float32 [b,h,w,2*vn]  written (zero where no class is hot)
 *   grad_conf   device float32 [b,h,w,vn]    written
 * A zero direction vector gets a zero gradient (TensorFlow's sqrt gradient yields NaN there).
 */
int casa_ls_vote_backward(casa_handle* h, const casa_ls_params* p, const float* seg, const float* direct,
                          const float* conf, const float* grad_points, float* out_points, float* grad_direct,
                          float* grad_conf, void* stream);
/* The same with seg, direct and conf in `dtype`; grad_direct and grad_conf are written as float32 all the same. */
int casa_ls_vote_backward_typed(casa_handle* h, const casa_ls_params* p, casa_dtype dtype, const void* seg,
                                const void* direct, const void* conf, const float* grad_points, float* out_points,
                                float* grad_direct, float* grad_conf, void* stream);

/*
 * Batched PnP on the GPU — the step right after the voting path (SURVEY.md 8f-2).  Stands in for the
 * reference's host-side pnp / map_offsets / map_pnp
 * (/root/reference/casapose/pose_estimation/ransac_voting.py:13-57, 487-514): robust initial pose from point
 * subsets (OpenCV's randomised EPnP-RANSAC cannot be replayed bit for bit), then the Levenberg-Marquardt
 * minimum of the reprojection error over ALL points in float64, flip if t_z < 0, zeros if |sum(points)| < 0.01
 * or on failure.
 *   points2d device float32 [n,vn,2] (x,y) pixels     points3d device float32 [n,vn,3]
 *   camera   device float32 [n,3,3] (zero skew)        offsets  device float32 [n,10] or NULL (:494-504)
 *   poses    device float32 [n,3,4] = [R|t]
 * vn in 6..16.  Asynchronous on `stream`.
 */
int casa_pnp(casa_handle* h, int32_t n, int32_t vn, const float* points2d, const float* points3d,
             const float* camera, const float* offsets, float* poses, void* stream);

/*
 * Backward of PnP w.r.t. the 2-D points — the "fast" implicit-function gradient of the reference's BPnP layer
 * (/root/reference/casapose/pose_estimation/bpnp_layers.py:138-277, Chen et al., CVPR 2020):
 * grad_points2d = J (J^T J)^-1 grad_y, J = d projection / d pose at the given pose (Gauss-Newton Hessian, no
 * residual-curvature terms), so the gradient depends on the pose, the 3-D points and the camera only.
 *   points3d   device float32 [n,vn,3]           camera device float32 [n,3,3] (zero skew)
 *   poses      device float32 [n,3,4] [R|t] (pose_form 12: what casa_pnp / poses_pnp write; a t_z < 0 flip, -[R|t],
 *              is recognised by det(R) < 0) or [n,6] (rvec, tvec) (pose_form 6: what BPNP_fast returns)
 *   grad_poses device float32, same shape as poses: dL/d poses
 *   grad_points2d device float32 [n,vn,2] (x,y), written densely
 * An object gets an exact zero gradient if its pose is all zero, if a point lies at z <= 0 under the (un-flipped)
 * pose, or if J^T J is numerically singular (e.g. collinear points).  vn in 6..16; n == 0 is a no-op.  One kernel,
 * no workspace, no synchronisation: asynchronous on `stream` and usable inside a captured graph.
 */
int casa_pnp_backward(casa_handle* h, int32_t n, int32_t vn, const float* points3d, const float* camera,
                      const float* poses, int32_t pose_form, const float* grad_poses, float* grad_points2d, void* stream);

/*
 * ADD / ADD-S / 2-D reprojection errors of a batch of poses (SURVEY.md 8f-3).  Stands in for the reference's
 * map_estimates + evaluate_poses (/root/reference/casapose/pose_estimation/ransac_voting.py:561-625, 628-687):
 * per object one row [err_2d, err_3d, valid_3d, valid_2d, missing, false_positive]; the caller sums rows over
 * the batch like :668-675.  err_3d is the mean point distance (ADD) or, for models with 7862 / 3417 points
 * (:618), the mean closest-point distance (ADD-S).  The reference takes the closest point from the float64 expansion
 * |a|^2 - 2ab + |b|^2 (:596-610); the kernel takes it from the direct float32 difference (a-b).(a-b), which has no
 * cancellation (relative error 2e-7 of the squared distance): identical verdicts, errors within 1e-5 relative
 * (tests/test_gpu_pose_metric.py).
 *   poses, poses_gt device float32 [n,3,4]            camera       device float32 [n,3,3]
 *   model_points    device float32 [m,maxp,3]         model_counts device int32   [m]  points used per model
 *   obj_model       device int32   [n] model of each object, or NULL: object i uses model i % m
 *   diameters       device float32 [n]                valid        device int32   [n]  valid_points_filter
 *   out_rows        device float32 [n,6]
 * Asynchronous on `stream`; scratch is owned by the handle.
 */
int casa_pose_errors(casa_handle* h, int32_t n, int32_t m, int32_t maxp, const float* poses, const float* poses_gt,
                     const float* camera, const float* model_points, const int32_t* model_counts,
                     const int32_t* obj_model, const float* diameters, const int32_t* valid,
                     float allowed_error_2d, float* out_rows, void* stream);

/*
 * Synchronous and asynchronous calls.  casa_ransac_vote / casa_ransac_vote_seg enqueue ONE CUDA graph per call on
 * `stream`: compaction, the first RANSAC round, a device-driven WHILE over the remaining rounds (the reference's
 * data-dependent tf.while_loop, ransac_voting.py:318-347, never returns to the host), refinement and solve.
 *   synchronous (default): the call waits for the 32-byte loop state of its own graph — not for refinement and
 *     solve — and returns CASA_ERR_WORKSPACE / CASA_ERR_INPUT if the device raised a status bit; like the reference's
 *     eager call, the result tensor itself is complete only after the stream has been synchronised.
 *   asynchronous (casa_set_async(h, 1)): the call returns as soon as the graph is enqueued, so consecutive calls
 *     queue back to back on the GPU (the data-parallel serving loop).  casa_sync(h) waits for every call issued on
 *     the handle (including refinement / solve) and returns the first error any of them raised; at most 256 calls
 *     may be outstanding before the library collects the oldest ones itself.
 *   asynchronous on n lanes (casa_set_async(h, n), n = 2..4): as above, and consecutive votes rotate over n internal
 *     lanes (own workspace, own stream, forked from `stream` by an event at call time), so that the compaction and
 *     hypothesis kernels and the refinements of n votes overlap — they are latency-bound — while the scoring kernels run
 *     back to back, each filling the GPU alone.  The inputs of a vote must stay untouched and its output is NOT ordered
 *     on `stream` until casa_join(h, stream) (device-side: `stream` waits for the lanes) or casa_sync(h) (host-side).
 *     casa_allgather_points_overlapped follows the lane of the last vote by itself.  casa_get_timing's k_score event
 *     pairs include the time a launch waits behind the previous lane's k_score: time the kernel in mode 0 / 1.  Debug
 *     calls, the host-buffer entry point and the LS layer always run on the caller's stream.
 */
int casa_set_async(casa_handle* h, int mode);
int casa_sync(casa_handle* h);
int casa_join(casa_handle* h, void* stream);

/*
 * DLPack entry point: the same vote with the tensors handed over as DLManagedTensor* (the pointer inside a "dltensor"
 * PyCapsule produced by any framework's __dlpack__: TensorFlow's tf.experimental.dlpack.to_dlpack, CuPy, JAX, PyTorch).
 * This is the drop-in's counterpart of the reference's only foreign-code seam, tf.numpy_function
 * (ransac_voting.py:513, bpnp_layers.py:322).  Device type, device id, dtype, dimensions and C-contiguous
 * strides are validated here, in C; b, h, w, oc, vn and vertex_per_class are taken from the tensors (the other fields of
 * `p` are used as given); `out` is a caller-allocated [b,oc,vn,2] tensor of the same device.  The three capsules are
 * CONSUMED in every case: their deleters are called exactly once — at once if the call is rejected, otherwise when the
 * GPU work queued on `stream` by this call has finished (polled at later calls on the handle, casa_sync, casa_destroy).
 * mask_is_seg != 0: `mask` holds [b,h,w,1+oc] segmentation scores (casa_ransac_vote_seg).  `mask` and `vertex` may be
 * float32 (DLPack code 2, 32 bits), float16 (code 2, 16 bits) or bfloat16 (code 4, 16 bits), as in
 * casa_ransac_vote_typed; `out` is float32.
 */
int casa_ransac_vote_dlpack(casa_handle* h, const casa_ransac_params* p, void* mask_dlm, void* vertex_dlm, void* out_dlm,
                            int mask_is_seg, void* stream);

/*
 * Multi-GPU: the path shards by image with no data-path collective (the reference maps independently over images,
 * ransac_voting.py:483; its only multi-GPU mechanism, MirroredStrategy at train_casapose.py:195, shards the batch
 * the same way); only the [b, oc, vn, 2] keypoints of every rank are all-gathered (576 B per frame).  The gather is
 * part of the C ABI so that a caller without torch.distributed (a TensorFlow replica thread) can use it:
 *   casa_nccl_unique_id   rank 0 creates the 128-byte NCCL id and distributes it by any means it has
 *   casa_comm_init        every rank: ncclCommInitRank on the handle's device (owned by the handle)
 *   casa_comm_attach      or borrow the framework's own ncclComm_t (never destroyed by this library)
 *   casa_allgather_points ncclAllGather of `floats_per_rank` float32 per rank on `stream` (nccl_comm NULL: the handle's)
 *   casa_allgather_points_overlapped  the same on the handle's own gather stream, ordered only behind what is queued
 *                         on `after_stream` at the time of the call: the exchange of step i overlaps the voting of
 *                         step i+1 and no compute stream ever waits for a peer; `slot` (0..7) names the completion
 *                         event, casa_gather_wait(h, slot, stream) makes `stream` wait for it ((void*)-1: the host).
 * NCCL is resolved with dlopen("libnccl.so.2") at the first call (CASA_NCCL_LIB overrides), so the library loads without it.
 */
int casa_nccl_unique_id(void* id128);
int casa_comm_init(casa_handle* h, const void* id128, int rank, int world);
int casa_comm_attach(casa_handle* h, void* nccl_comm, int rank, int world);
int casa_comm_destroy(casa_handle* h);
int casa_allgather_points(casa_handle* h, void* nccl_comm, const float* local, float* gathered, int64_t floats_per_rank,
                          void* stream);
int casa_allgather_points_overlapped(casa_handle* h, const float* local, float* gathered, int64_t floats_per_rank,
                                     void* after_stream, int slot);
int casa_gather_wait(casa_handle* h, int slot, void* stream);

/* Device status word of the last casa_ransac_vote on this handle (CASA_STATUS_* bits); after casa_ransac_vote_host
 * (or casa_host_wait) the OR over the image ranges of that call. */
int casa_last_status(casa_handle* h, uint32_t* status);
/* Number of kernels the last call launched on this handle (casa_ransac_vote_host: all its image ranges). */
int casa_last_launches(casa_handle* h, int64_t* launches);

/*
 * Measurement hooks (bench.py).  With timing enabled the scoring-kernel launch of the first round of every call is
 * bracketed by CUDA events on the caller's stream (event-record nodes of the call's graph; later rounds run inside
 * the graph's WHILE body, which cannot hold event nodes).  casa_get_timing returns the summed duration of those
 * launches (ms), their number, and the filter statistics
 * stats[0] = units scored (hypothesis x pixel x keypoint tests, all rounds), stats[1] = units decided by the
 * exact predicate, stats[2] = exact-list hypotheses, stats[3] = stage-2 (hypothesis pair, chunk) events
 * — of the LAST call for a synchronous handle, accumulated over the calls since the previous query for an
 * asynchronous one (the query collects them, i.e. waits for their loop states).
 */
int casa_set_timing(casa_handle* h, int enable);
int casa_get_timing(casa_handle* h, double* score_ms, int64_t* score_launches, uint64_t* stats4);

/*
 * Test hook of the host mask packer casa_ransac_vote_host uses (no device involved): packs mask [npx][oc] float32
 * into one membership word per pixel, bit c = (mask[p][c] != 0) as tf.not_equal counts it (ransac_voting.py:304:
 * NaN is set, -0 is not), on `threads` host threads in `parts` consecutive ranges.  Returns 1 if a set element
 * differs from 1.0 (what the vote reports as CASA_STATUS_MASK_NOT_BINARY), 0 if not, a negative error code otherwise.
 */
int casa_selftest_pack(const float* mask, uint32_t* bits, int64_t npx, int oc, int threads, int parts);

/*
 * Self-test of the filtered inlier predicate: draws n adversarial (pixel, hypothesis)
 * pairs concentrated on the decision boundary and compares filter+fallback with the
 * reference-exact float32 sequence (ransac_voting.py:230-249).
 * spread = half-width (rad) of the sampled band around the boundary; a negative spread additionally draws extreme
 * magnitudes (coordinates to 65535, |d| in 2^[-19,29], pixel-hypothesis distances 2^[-17,59]).
 * out[0]=tested, out[1]=mismatches, out[2]=sent to exact fallback, out[3]=exact inliers.
 */
int casa_selftest_filter(casa_handle* h, uint64_t n, uint64_t seed, float inlier_thresh,
                         float spread, uint64_t* out4_host);

/* Measured FP32 FMA issue rate of this GPU (TFLOP/s), the denominator for "% of FP32 peak" (16 independent FFMA chains per
 * thread, best of 4 timed launches).  variant must be 0; the instruction-mix explorations of round 1 are not part of the
 * library any more (casapose_b200/csrc/experimental/). */
int casa_measure_fp32_peak(casa_handle* h, int variant, double* tflops, double* ms);

#ifdef __cplusplus
}
#endif
#endif /* CASAPOSE_B200_H_ */
