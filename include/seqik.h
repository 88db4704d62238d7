/* seqik.h -- C ABI of libseqik_sm100.so, the B200 (sm_100a) implementation of SeqIKPy's
 * leg inverse-kinematics hot path.
 *
 * The reference (NeLy-EPFL/sequential-inverse-kinematics, pure Python) has no FFI seam;
 * its seam is the Python class API.  Each entry point below states which reference
 * function(s) it replaces (paths relative to the reference repository root).  The
 * binding a maintainer of the reference would add is a ctypes stub: see INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch tensors:
 *     tensor.data_ptr()); the library allocates nothing that outlives a call;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = the
 *     legacy default stream) of the calling thread's current device;
 *   - return value: 0 ok, SEQIK_EINVAL bad argument, SEQIK_ECUDA CUDA error; the message
 *     is available (per host thread) from seqik_last_error();
 *   - strides are in ELEMENTS (floats), not bytes; the innermost key-point block
 *     ([5][3], [9][3], [7]) is always contiguous;
 *   - a "chain" is one leg of one trial; frames of a chain are solved serially (warm
 *     start), chains are independent.  DOF order everywhere: ThC_yaw, ThC_pitch, ThC_roll,
 *     CTr_pitch, CTr_roll, FTi_pitch, TiTa_pitch (the insertion order of the reference's
 *     joint_angles_dict, seqikpy/leg_inverse_kinematics.py:285-320).
 */
#ifndef SEQIK_H_
#define SEQIK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SEQIK_ABI_VERSION 13  /* 13: seqik_head_apply_backward_f32, seqik_head_affine_backward_f32/_f64; 12: seqik_align_apply_backward_f32, seqik_leg_affine_backward_f32; 11: seqik_pchip_resample_backward_f32/_f64; 10: seqik_head_angles_backward_f32; 9: seqik_fk_backward_f32; 8: seqik_origin_rows_f32; 7: seqik_leg_affine_from_pose_f32; 6: schedule 3 (frame-parallel blocks), seqik_fk_expand_host_f32; 5: solver flag bits 6-7, phase periods in bits 21-27 */
#define SEQIK_OK 0
#define SEQIK_EINVAL (-1)
#define SEQIK_ECUDA (-3)

/* flags of seqik_leg_solve_f32 */
#define SEQIK_FLAG_GN_STAGE(s) (1u << (s))   /* s = 0..3: stage s+1 takes the Gauss-Newton step when it fits the
                                                trust region (what scipy's TRF does on the longer chains, DESIGN.md) */
#define SEQIK_FLAG_ESCAPE (1u << 4)          /* singularity escape: a solve that ends on the sin(pitch) = 0 singularity of its
                                                roll/pitch pair may continue from the closed-form solution (DESIGN.md 2) */
#define SEQIK_FLAG_SKIP_CONFIRM (1u << 5)    /* stop a solve WITHOUT the evaluation that would only confirm convergence: when the
                                                model was accurate on the previous step (actual/predicted within 25 % of 1) and now
                                                predicts a reduction below ftol * cost for a plain Gauss-Newton step.  The skipped
                                                step is < ~3e-6 rad; saves one of the ~5 evaluations of a warm-started solve */
#define SEQIK_FLAG_NEWTON (1u << 6)          /* Newton steps: where the Gauss-Newton step is admissible (fits the trust region, stays in
                                                the box) and the full Hessian of the two-angle model -- J^T J plus the residual-curvature
                                                term, closed form -- is safely positive definite, take the Newton step instead.  Key
                                                points are noisy, so the residual does not vanish at the solution and Gauss-Newton
                                                converges linearly; Newton reaches the same minimiser in fewer evaluations (config 3:
                                                5.3 -> 4.1 per solve in stage 1) and ends closer to it than the reference's ftol stop */
#define SEQIK_FLAG_CLOSED_FORM (1u << 7)     /* closed-form warm step (stage pipeline schedule): before the next frame of a carried solve
                                                the iterate is moved to the point of the sphere |w| = L nearest to the new target, on
                                                the warm start's branch -- the minimiser the iteration would converge to -- when that
                                                is a short (< 0.5 rad), strictly interior, well-conditioned move; the solve then ends
                                                with its first evaluation or is polished by the iteration.  Every other case (first
                                                frame of a call, re-derivation frames, active bounds, near-singular or ill-conditioned
                                                targets, large moves) runs from the warm start as without the flag.  Config 3:
                                                4.1 -> 1.2 evaluations per solve */
#define SEQIK_FLAG_REFERENCE_ITERATES 0x3Fu  /* the reference's own iterates: Gauss-Newton mode in all four stages + escape +
                                                skip-confirm, evaluation counts and termination statuses as scipy's */
#define SEQIK_FLAG_DEFAULT 0xFFu             /* the above + Newton steps + closed-form warm step (each set validated against the
                                                reference's shipped angles and forward kinematics) */
#define SEQIK_FLAG_SCHED_SHIFT 8             /* bits 8..11: kernel schedule, 0 = automatic,
                                                1 = one lane per chain, 2 = stage pipeline (four lanes per chain),
                                                3 = frame-parallel blocks (a warp per chain, 32 frames per pass; needs all four
                                                stages and the closed-form warm step in every stage, i.e. the default flags;
                                                results are bit-identical to schedule 2) */
#define SEQIK_FLAG_SCHED_MASK (0xFu << SEQIK_FLAG_SCHED_SHIFT)
#define SEQIK_FLAG_GATE_SHIFT 21             /* bits 21..24: period (1..15 loop iterations) of the open/close phases of schedule 2, 0 = automatic.
                                                Scheduling only: results do not depend on it */
#define SEQIK_FLAG_TRIP_SHIFT 25             /* bits 25..27: period (1..7 loop iterations) of the evaluation block of schedule 2, 0 = automatic.
                                                Scheduling only */
#define SEQIK_FLAG_FK_JOINTS (1u << 20)      /* fk holds only the four joint rows that carry information: [n_chain][n_frame][4][3] =
                                                rows 5..8 of the full layout (Coxa-Femur, Femur-Tibia, Tibia-Tarsus, Claw).  Rows 0-3
                                                of the full layout repeat the input origin and row 4 repeats row 5; leaving them out
                                                cuts the result from 136 to 76 bytes per leg-frame, which is what an end-to-end
                                                call over PCIe is bound by (DESIGN.md 7) */
#define SEQIK_FLAG_BLOCK_VARIANT_SHIFT 28    /* bits 28..29: kernel variant of schedule 3, 0 = automatic (by batch size), 1 = lean (large batches),
                                                2 = robust (replay-heavy recordings: stage-granular replays).  Scheduling only */
#define SEQIK_FLAG_CPW_SHIFT 12              /* bits 12..17: chains per warp of schedule 2 (1..8) / resident warps per SM of schedule 3
                                                (1..32), 0 = automatic */

int seqik_abi_version(void);
const char* seqik_last_error(void);

/* Per-chain constants of seqik_leg_solve_f32 / seqik_fk_f32: one row of 32 floats per chain.
 *   [0..3]   segment lengths Coxa, Femur, Tibia, Tarsus (KinematicChainSeq.body_size,
 *            seqikpy/kinematic_chain.py:170-421; utils.calculate_body_size utils.py:89-123)
 *   [4..10]  lower bounds, [11..17] upper bounds of the 7 DOFs (bounds_dof)
 *   [18..24] seeds of the 7 DOFs = the ACTIVE slots of INITIAL_ANGLES[leg]["stage_k"]
 *            (seqikpy/data.py:4-22; leg_inverse_kinematics.py:272,376)
 *   [25..28] squared norm of the INERT slots (Base link, frozen links, last link) of the four
 *            stage seed vectors: they enter scipy's initial trust radius and xtol test
 *   [29..31] reserved (0)
 */
#define SEQIK_CHAIN_PARAM_FLOATS 32

/* 4-stage sequential leg IK + stage-4 forward kinematics.
 * Replaces LegInvKinSeq.run_ik_and_fk / calculate_ik_stage
 * (seqikpy/leg_inverse_kinematics.py:200-403) together with what they call:
 * KinematicChainSeq.create_leg_chain (seqikpy/kinematic_chain.py:99-421),
 * ikpy Chain.inverse_kinematics / forward_kinematics and scipy.optimize.least_squares.
 *
 *   pose    [n_chain][n_frame][5][3] key points (row 0 = Thorax-Coxa origin, row s = target of
 *           stage s), addressed as pose + c*pose_chain_stride + t*pose_frame_stride
 *   affine  NULL, or [n_chain][8] = (fixed_coxa xyz, scale, template_coxa xyz, 0): the
 *           AlignPose.align_leg map (seqikpy/alignment.py:471-485) applied on load
 *   params  [n_chain][32] (layout above)
 *   angles  [n_chain][n_frame][7] out.  When stage_mask does not start at stage 1 it is also an
 *           INPUT: the DOFs of the earlier stages are read from it per frame and frozen -- the
 *           `angles=self.joint_angles_dict, t=t` of kinematic_chain.py:99-150
 *   fk      NULL, or [n_chain][n_frame][9][3] out (rows 0-3 origin, 4-5 Coxa-Femur joint,
 *           6 Femur-Tibia, 7 Tibia-Tarsus, 8 Claw: leg_inverse_kinematics.py:71-77,279-282);
 *           rows of stages after the last solved one are left untouched.  With SEQIK_FLAG_FK_JOINTS:
 *           [n_chain][n_frame][4][3], the joint rows only
 *   warm    NULL, or 7 angles per chain (addressed warm + c*warm_chain_stride) that replace the seeds of `params`:
 *           pass the last solved frame of the same chains (angles + (t0-1)*ang_frame_stride) to continue a
 *           recording in frame chunks -- bit-identical to one call over all frames, which is what lets the host
 *           pipeline copy chunk k+1 in and chunk k-1 out while chunk k is solved
 *   status  NULL, or [n_chain] out: 1 normal; 0 if some solve stopped at max_nfev; -1 if some solve met a non-finite
 *           residual (NaN/inf key point; scipy raises "Residuals are not finite in the initial point" there): that
 *           solve is skipped, its DOFs keep the previous frame's values
 *   nfev    NULL, or [n_chain][4] out: function evaluations summed over frames, per stage
 *   stage_mask  bit s set = solve stage s+1; the set bits must be contiguous
 *           (stages=[a..b] of run_ik_and_fk, leg_inverse_kinematics.py:350-353)
 *   flags   SEQIK_FLAG_* above: SEQIK_FLAG_DEFAULT for production use; SEQIK_FLAG_REFERENCE_ITERATES to walk the
 *           reference's own iterates (evaluation counts and termination statuses as scipy's); scheduling fields
 *           (schedule, chains per warp, phase periods: tuning and tests) never change results; SEQIK_FLAG_FK_JOINTS
 *           selects the compact fk layout
 */
int seqik_leg_solve_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride,
                        const float* affine, const float* params,
                        float* angles, int64_t ang_chain_stride, int64_t ang_frame_stride,
                        float* fk, int64_t fk_chain_stride, int64_t fk_frame_stride,
                        const float* warm, int64_t warm_chain_stride,
                        int32_t* status, uint32_t* nfev,
                        int64_t n_chain, int64_t n_frame, uint32_t stage_mask, uint32_t flags, void* stream);

/* Generic (single-target) leg IK: all 7 joints solved at once against ONE target, the claw.
 * Replaces LegInvKinGeneric.run_ik_and_fk / calculate_ik_stage (seqikpy/leg_inverse_kinematics.py:473-613) together
 * with KinematicChainGeneric.create_leg_chain (seqikpy/kinematic_chain.py:444-532), ikpy Chain.inverse_kinematics /
 * forward_kinematics and scipy.optimize.least_squares on that chain.
 *
 * JOINT ORDER of this entry point = the link order of the generic chain: ThC_roll, ThC_yaw, ThC_pitch, CTr_pitch,
 * CTr_roll, FTi_pitch, TiTa_pitch (roll FIRST: kinematic_chain.py:464-488) -- for params, warm and angles alike.
 *
 *   pose    [n_chain][n_frame][k][3] key points, k > target_row; row 0 = Thorax-Coxa origin, row target_row = the end
 *           effector (the reference takes the LAST key point, leg_inverse_kinematics.py:582); other rows are not read
 *   params  [n_chain][32]: [0..3] segment lengths, [4..10] lower / [11..17] upper bounds, [18..24] seeds (slots 1..7 of
 *           INITIAL_ANGLES[leg]["stage_4"], applied positionally to the generic chain exactly as the reference does,
 *           leg_inverse_kinematics.py:583), [25] squared norm of the two inert seed slots (Base link, Claw)
 *   angles  [n_chain][n_frame][7] out;  fk NULL, or [n_chain][n_frame][9][3] out (rows 0-3 origin, 4-5 Coxa-Femur
 *           joint, 6 Femur-Tibia, 7 Tibia-Tarsus, 8 Claw);  warm / status / nfev ([n_chain], evaluations summed over
 *           frames) as in seqik_leg_solve_f32
 *   flags   bits SEQIK_FLAG_CPW_SHIFT..+5: chains per warp (1..32), 0 = automatic; bits SEQIK_FLAG_SCHED_SHIFT..+3: 0 automatic
 *           (2 while the batch is resident at once, else 1), 1 one lane per chain, 2 eight lanes per chain (a joint per lane,
 *           sums over the joints by butterfly shuffles; up to 4 chains per warp).  Same iteration, different summation
 *           order; other bits must be 0
 *
 *   status  per chain: -1 if some frame was skipped (a non-finite key point; it takes precedence over everything else),
 *           else 0 if some solve stopped at the evaluation limit (100 * 9), else 1.  A skipped frame counts one evaluation
 *           in nfev, its angles are the ones it was seeded with (the previous frame's, or the seed for frame 0), its fk
 *           rows are those angles placed at its own origin (so not finite when the origin is not), and the next frame
 *           starts from the same angles: the frames after it are bit-identical to a call without the skipped frame.
 *           Returned angles lie strictly inside the limits in the working precision.
 *
 * The reference's generic solve is under-determined (3 equations, 7 unknowns) and its answer depends on rounding noise
 * (DESIGN.md 5.4): this entry point restates the same iteration, reproduces the reference solve by solve from the same
 * seed (tests) and reaches the same claw residual, but a free-running recording follows its own path on the
 * self-motion manifold.  In FP64 both mappings take the same iterates as the host build of seqik_generic.cuh on every
 * solve that rounding-level perturbations do not change (tests/test_gpu_generic_cert.py). */
int seqik_leg_solve_generic_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride, int32_t target_row,
                                const float* params,
                                float* angles, int64_t ang_chain_stride, int64_t ang_frame_stride,
                                float* fk, int64_t fk_chain_stride, int64_t fk_frame_stride,
                                const float* warm, int64_t warm_chain_stride,
                                int32_t* status, uint32_t* nfev,
                                int64_t n_chain, int64_t n_frame, uint32_t flags, void* stream);
/* Same with FP64 data AND FP64 device arithmetic (B200's FP64 pipe runs at half the FP32 rate; a lane-per-chain solve is
 * latency-bound, so the cost is ~2x).  The reference's generic iteration amplifies rounding (its candidate-step choice
 * flips on near-ties): in FP64 the device agrees with scipy solve by solve as often as scipy agrees with itself under
 * a 1e-12 mm input perturbation (~98 % of solves within 1e-3 rad), in FP32 on ~90 %.  The dict API uses this one. */
int seqik_leg_solve_generic_f64(const double* pose, int64_t pose_chain_stride, int64_t pose_frame_stride, int32_t target_row,
                                const double* params,
                                double* angles, int64_t ang_chain_stride, int64_t ang_frame_stride,
                                double* fk, int64_t fk_chain_stride, int64_t fk_frame_stride,
                                const double* warm, int64_t warm_chain_stride,
                                int32_t* status, uint32_t* nfev,
                                int64_t n_chain, int64_t n_frame, uint32_t flags, void* stream);

/* Forward kinematics only: angles -> 9x3 joint positions.
 * Replaces LegInvKinBase.calculate_fk (seqikpy/leg_inverse_kinematics.py:71-77) on the stage-4 chain.
 *   angles [n_chain][n_frame][7], origin [n_chain][n_frame][3] (or [n_chain][3] with
 *   origin_frame_stride = 0), params as above, fk [n_chain][n_frame][9][3]; all dense. */
int seqik_fk_f32(const float* angles, const float* origin, int64_t origin_frame_stride, const float* params,
                 float* fk, int64_t n_chain, int64_t n_frame, void* stream);

/* Backward of seqik_fk_f32 (vector-Jacobian product): the gradient of a loss L with respect to the angles, the origin and
 * the segment lengths, given grad_fk = dL/dfk.  New in this library: the reference has no gradients, so this replaces
 * nothing in it.
 *   angles, origin, origin_frame_stride, params: as for seqik_fk_f32 (params[0..3] are the only entries FK reads).  The
 *   gradients do not depend on the origin (FK is a translation by it): it is checked for NULL but not read.
 *   grad_fk      [n_chain][n_frame][9][3] in
 *   grad_angles  [n_chain][n_frame][7] out (required)
 *   grad_origin  NULL (skip), or [n_chain][n_frame][3] out: dL/dorigin PER FRAME, also when origin_frame_stride = 0 (the
 *                caller sums over frames).  Per coordinate, in float32 and in this order (g_r = row r of grad_fk):
 *                  S4 = g8;  S3 = g7 + S4;  S2 = g6 + S3;  S1 = (g4 + g5) + S2;
 *                  grad_origin = (((g0 + g1) + g2) + g3) + S1
 *   grad_lengths NULL (skip), or [n_chain][n_frame][4] out: per-frame contributions to dL/dparams[0..3] (the caller sums
 *                over frames; no other params entry has a gradient)
 * All arrays dense.  The forward is recomputed with the arithmetic of seqik_fk_f32; results are deterministic (no
 * atomics) and do not depend on the launch path. */
int seqik_fk_backward_f32(const float* angles, const float* origin, int64_t origin_frame_stride, const float* params,
                          const float* grad_fk, float* grad_angles, float* grad_origin, float* grad_lengths,
                          int64_t n_chain, int64_t n_frame, void* stream);

/* Head roll/pitch/yaw and antenna yaw/pitch (L then R).
 * Replaces HeadInverseKinematics.compute_head_angles (seqikpy/head_inverse_kinematics.py:103-142, 163-307).
 *   r_head, l_head [n_trial][n_frame][2][3] (base, tip); neck [n_trial][n_frame][3] (neck_stride 3) or
 *   [n_trial][3] (neck_stride 0: one point per trial, the (1,1,3) template Neck of alignment.py:375-376)
 *   affine_r, affine_l: NULL, or [n_trial][8] head-alignment rows (see seqik_head_affine_f32) applied on load
 *   rest [n_trial][2] = (rest_head_pitch, rest_antenna_pitch) (head_inverse_kinematics.py:309-329)
 *   out [n_trial][7][n_frame]: head_roll, head_pitch, head_yaw, antenna_yaw_L, antenna_pitch_L,
 *   antenna_yaw_R, antenna_pitch_R
 * Any 4-byte aligned r_head / l_head works: 8-byte aligned inputs are read with 64-bit loads, others (e.g. a view at an odd
 * float offset) with 32-bit loads, with bit-identical results. */
int seqik_head_angles_f32(const float* r_head, const float* l_head, const float* neck, int64_t neck_stride,
                          const float* affine_r, const float* affine_l, const float* rest,
                          float* out, int64_t n_trial, int64_t n_frame, void* stream);

/* Backward of seqik_head_angles_f32 (vector-Jacobian product): the gradient of a loss L with respect to the antenna key
 * points and the neck, given grad_out = dL/dout.  New in this library: the reference has no gradients, so this replaces
 * nothing in it.
 *   r_head, l_head, neck, neck_stride, affine_r, affine_l: as for seqik_head_angles_f32.  The rest angles are additive
 *   constants of the angles and do not enter the gradient (dL/drest_head_pitch = sum of dL/dhead_pitch,
 *   dL/drest_antenna_pitch = -sum of dL/dantenna_pitch L and R).
 *   grad_out     [n_trial][7][n_frame] in, the layout of seqik_head_angles_f32's out
 *   grad_r_head, grad_l_head  [n_trial][n_frame][2][3] out (required): dL/d(base xyz, tip xyz)
 *   grad_neck    NULL (skip), or [n_trial][n_frame][3] out: dL/dneck PER FRAME, also when neck_stride = 0 (the caller
 *                sums over frames)
 * The gradients are taken with respect to the points AS PASSED.  With affine rows, the points are first mapped as
 * seqik_head_angles_f32 maps them (seqik_head_apply_f32's arithmetic), and the gradient of a raw point is the gradient of
 * the aligned point times the row's scale, aff[3] for a base and aff[7] for a tip: one float32 multiplication, the last
 * operation.  The affine rows themselves get no gradient.
 * Degenerate frames: every angle is the signed angle between two vectors projected onto a coordinate plane.  Where such a
 * projected vector has float32 squared length exactly 0, that vector's terms contribute 0 (torch.atan2's gradient at
 * (0, 0)); when it is the roll's hor|x=0, the roll's propagation into the antenna angles is 0 as well.  A vector with a
 * subnormal squared length (shorter than ~1e-19) is taken at squared length FLT_MIN.  For finite inputs no output is NaN
 * or inf unless the gradient itself overflows float32.
 * All arrays dense.  The forward's roll is recomputed with its arithmetic, so the de-rotated vectors are the forward's;
 * results are deterministic (no atomics) and do not depend on the pointer alignment (8-byte aligned r_head / l_head /
 * grad_r_head / grad_l_head move as 64-bit loads and stores, others as 32-bit ones, with bit-identical results). */
int seqik_head_angles_backward_f32(const float* r_head, const float* l_head, const float* neck, int64_t neck_stride,
                                   const float* affine_r, const float* affine_l, const float* grad_out,
                                   float* grad_r_head, float* grad_l_head, float* grad_neck,
                                   int64_t n_trial, int64_t n_frame, void* stream);

/* AlignPose statistics: mean of the 0.45 and 0.55 quantiles (numpy "linear" interpolation) of each series.
 * Replaces _get_mean_quantile over the series built by AlignPose.get_fixed_pos / get_mean_length
 * (seqikpy/alignment.py:83-87, 392-415).
 *   series [n_series][n] (dense rows); counts NULL, or [n_series] int32: only the counts[i] SMALLEST values of
 *   row i take part (rows padded with +inf, see seqik_head_series_f32); out [n_series];
 *   scratch: unused (may be NULL); kept so that the signature is stable
 * Values are ordered by their bits: -0 sorts below +0, a NaN with the sign bit clear above +inf and one with the sign
 * bit set below -inf; a NaN among the four order statistics makes the result NaN.  The four order statistics are
 * exact; each quantile is a + (b - a) f in float32 with f = float32(q (m - 1) - floor(q (m - 1))), m the values taking
 * part, and out = 0.5f (q45 + q55).  counts[i] <= 0 gives NaN; counts[i] > n is outside the contract. */
int seqik_mid_quantile_f32(const float* series, const int32_t* counts, float* scratch, float* out,
                           int64_t n_series, int64_t n, void* stream);

/* Leg-segment series for the statistics: for each chain the 3 coordinates of key point 0 and the 4
 * segment lengths |kp[s+1]-kp[s]| per frame -> series [n_chain][7][n_frame].
 * Replaces the array construction of AlignPose.get_fixed_pos / get_mean_length (alignment.py:392-415). */
int seqik_leg_series_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride,
                         float* series, int64_t n_chain, int64_t n_frame, void* stream);

/* Leg affine rows from the statistics (AlignPose.find_scale_leg + align_leg, alignment.py:417-423, 465-485).
 *   stats [n_chain][7] (seqik_mid_quantile_f32 of the leg series); consts [n_chain][4] = (template
 *   {leg}_Coxa xyz, model leg length already reduced by the tarsus unless include_claw);
 *   affine [n_chain][8] out = (fixed_coxa xyz, scale, template xyz, 0) */
int seqik_leg_affine_f32(const float* stats, const float* consts, int include_claw, float* affine,
                         int64_t n_chain, void* stream);

/* The three calls above in one (AlignPose.get_fixed_pos / get_mean_length / find_scale_leg, alignment.py:392-423, and the
 * affine row of align_leg, :465-485): key points [n_chain][n_frame][5][3] -> affine [n_chain][8].  Recordings of up to 1024
 * frames run ONE fused kernel -- a CTA per chain streams the key points through shared memory once (60 B per leg-frame, the
 * only DRAM traffic), seven warps select the seven mid-quantiles -- and need no scratch (NULL); longer recordings run the
 * series / select / affine kernels with scratch = n_chain * 7 * (n_frame + 1) floats.  Same results as the separate calls. */
int seqik_leg_affine_from_pose_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride,
                                   const float* consts, int include_claw, float* scratch, float* affine,
                                   int64_t n_chain, int64_t n_frame, void* stream);

/* The affine map of AlignPose.align_leg (alignment.py:471-485) as a standalone elementwise pass:
 * out[:,0] = template, out[:,i] = (pose[:,i] - fixed) * scale + template.   affine [n_chain][8] as above. */
int seqik_align_apply_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride,
                          const float* affine, float* out, int64_t n_chain, int64_t n_frame, void* stream);

/* Backward of seqik_align_apply_f32 (vector-Jacobian product), given grad_out = dL/dout.  New in this library: the reference
 * has no gradients, so this replaces nothing in it.
 *   pose, strides, affine: as for seqik_align_apply_f32;  grad_out [n_chain][n_frame][5][3] in (dense)
 *   grad_pose            NULL (skip), or [n_chain][n_frame][5][3] out (dense): 0 for key point 0 (it is replaced by the
 *                        template), aff[3] * grad_out for key points 1..4 (one float32 multiplication)
 *   grad_affine_partial  NULL (skip), or [n_chain][n_frame][8] out (dense): each leg-frame's contribution to dL/daffine (the
 *                        caller sums over frames).  With g_i = grad_out[c][t][i], d_i = ((p_ix - a0) g_ix + (p_iy - a1) g_iy)
 *                        + (p_iz - a2) g_iz and, per coordinate, S = ((g_1 + g_2) + g_3) + g_4, in float32 and in this order:
 *                          [0..2] = -(a3 S),  [3] = ((d_1 + d_2) + d_3) + d_4,  [4..6] = g_0 + S,  [7] = 0
 * Deterministic (no atomics); the bits do not depend on the launch path (dense and 16-byte aligned buffers stream through
 * the TMA tile pipeline, anything else through a plain kernel).  Sizes, NULL and stride errors are the forward's. */
int seqik_align_apply_backward_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride,
                                   const float* affine, const float* grad_out, float* grad_pose, float* grad_affine_partial,
                                   int64_t n_chain, int64_t n_frame, void* stream);

/* Backward of seqik_leg_affine_from_pose_f32 (vector-Jacobian product), given grad_affine = dL/daffine [n_chain][8].  New in
 * this library.  With H = grad_affine[c], m_s the seven mid-quantiles (coxa x, y, z, the four segment lengths), len = (m_3 +
 * m_4) + m_5 [+ m_6 with include_claw] and scale = affine[c][3]:
 *   grad_consts  NULL (skip), or [n_chain][4] out = (H4, H5, H6, H3 / len)
 *   grad_pose    [n_chain][n_frame][5][3] (dense, required): the statistics' contributions are ADDED to it, so a caller
 *                passes zeros or the output of seqik_align_apply_backward_f32.  dL/dm_s = H_s for the coxa series,
 *                -(H3 scale) / len for every length in len (the tarsus only with include_claw).  A mid-quantile
 *                0.5 ((v0 + (v1 - v0) f45) + (v2 + (v3 - v2) f55)) passes dL/dm to its order statistics with the weights
 *                0.5 (1 - f45), 0.5 f45, 0.5 (1 - f55), 0.5 f55 (ranks and weights of seqik_mid_quantile_f32; coinciding
 *                ranks add).  The order statistic of rank r sits in frame t_r; a coxa series sends its share to
 *                pose[t_r][0][coordinate], a length series j sends +share s / |s| to key point j+1 and -share s / |s| to key
 *                point j of frame t_r (s the segment vector; a squared length of exactly 0 contributes 0).
 *   Tie rule: keys are the forward's order keys (-0 below +0), the lengths compared on their float32 SQUARED lengths
 *   (dx dx + dy dy) + dz dz on every path; t_r is the (r - #{keys < key_r})-th frame, in ascending frame order, among the
 *   frames whose key equals key_r: argsort(keys, stable)[r].
 *   The mid-quantiles and len are recomputed from the selected keys with the forward's float32 arithmetic.  One thread per
 *   chain adds the contributions in a fixed order (series 0..6, rank position 0..3; end point before base point), so the
 *   result is deterministic.  Error bound against the float64 VJP at the same frames (u = 2^-24): per float of grad_pose
 *   64 u N A, N the contributions it receives and A the sum of their absolute values; 16 u |dL/dconsts| for grad_consts.
 *   scratch: NULL for recordings of up to 1024 frames (one CTA per chain), else n_chain * 7 * (n_frame + 12) 32-bit words.
 * Sizes, NULL, stride and empty-recording errors are the forward's. */
int seqik_leg_affine_backward_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride,
                                  const float* consts, int include_claw, const float* affine, const float* grad_affine,
                                  float* grad_pose, float* grad_consts, uint32_t* scratch,
                                  int64_t n_chain, int64_t n_frame, void* stream);

/* Antenna series of AlignPose.align_head (alignment.py:489-555).
 *   head [n_trial][n_frame][2][3] (base, tip), thorax [n_trial][n_frame][n_thorax_kp][3] (first and last
 *   key point are averaged, alignment.py:385-390).  Per trial, series [n_trial][5][n_frame]:
 *   rows 0-2 base xyz and row 3 d = |base - thorax_mid| at the "stationary" frames i with
 *   d[i+2] - 2 d[i+1] + d[i] < threshold (find_stationary_indices, alignment.py:425-434), +inf elsewhere;
 *   row 4 = |tip - base| at every frame.  counts [n_trial][5] int32: valid entries per row. */
int seqik_head_series_f32(const float* head, const float* thorax, int64_t n_thorax_kp, float threshold,
                          float* series, int32_t* counts, int64_t n_trial, int64_t n_frame, void* stream);
/* Same with FP64 key points (the dict API hands float64 arrays over).  Both variants evaluate the distances and the
 * stationarity test in FP64: one frame flipping in or out of the stationary set moves the quantiles by ~1e-4. */
int seqik_head_series_f64(const double* head, const double* thorax, int64_t n_thorax_kp, double threshold,
                          float* series, int32_t* counts, int64_t n_trial, int64_t n_frame, void* stream);

/* Head affine rows (alignment.py:515-553): stats [n_trial][5] (seqik_mid_quantile_f32 of the head
 *   series), consts [n_trial][5] = (template {side}_Antenna_base xyz, body_size Antenna_mid_thorax,
 *   body_size Antenna); affine [n_trial][8] out = (origin xyz, scale_base, template xyz, scale_tip) */
int seqik_head_affine_f32(const float* stats, const float* consts, float* affine, int64_t n_trial, void* stream);

/* out[:,0] = (base - origin) * scale_base + template; out[:,1] = (tip - origin) * scale_tip + template
 * (alignment.py:547-553).  head, out [n_trial][n_frame][2][3]. */
int seqik_head_apply_f32(const float* head, const float* affine, float* out, int64_t n_trial, int64_t n_frame,
                         void* stream);

/* Backward of seqik_head_apply_f32 (vector-Jacobian product), given grad_out = dL/dout.  New in this library: the reference
 * has no gradients, so this replaces nothing in it.
 *   head, affine: as for seqik_head_apply_f32;  grad_out [n_trial][n_frame][2][3] in.  With a = affine[trial], G_b and G_t
 *   the frame's dL/d(aligned base) and dL/d(aligned tip), P_b = base - origin and P_t = tip - origin (the forward's float32
 *   subtractions) and x . y = (x0 y0 + x1 y1) + x2 y2, in float32 and in this order:
 *   grad_head            NULL (skip), or [n_trial][n_frame][2][3] out: (a3 G_b, a7 G_t), one float32 multiplication each
 *                        (the affine contract of seqik_head_angles_backward_f32)
 *   grad_affine_partial  NULL (skip), or [n_trial][n_frame][8] out: each frame's contribution to dL/daffine (the caller sums
 *                        over frames): [0..2] = -((a3 G_b) + (a7 G_t)),  [3] = P_b . G_b,  [4..6] = G_b + G_t,  [7] = P_t . G_t
 * All arrays dense.  Deterministic (no atomics); the bits do not depend on the launch path (16-byte aligned buffers stream
 * through the TMA tile pipeline, anything else and the last partial tile through a plain kernel).  Size and NULL errors are
 * the forward's. */
int seqik_head_apply_backward_f32(const float* head, const float* affine, const float* grad_out, float* grad_head,
                                  float* grad_affine_partial, int64_t n_trial, int64_t n_frame, void* stream);

/* Backward of the head statistics -- seqik_head_series_f32/_f64, seqik_mid_quantile_f32 with the counts, seqik_head_affine_f32
 * -- (vector-Jacobian product), given grad_affine = dL/daffine [n_trial][8].  New in this library.
 *   head, thorax, n_thorax_kp: as for seqik_head_series_*, float32 (_f32) or float64 (_f64), dense
 *   series, counts: what seqik_head_series_* wrote for the same inputs.  The stationary set is NOT decided again: it is
 *           piecewise constant in the key points and is held fixed as the forward chose it
 *   consts, affine: the forward's consts (checked, not read: the gradient does not depend on them) and result rows
 *   grad_head    [n_trial][n_frame][2][3] (required), grad_thorax NULL (skip the thorax terms) or
 *                [n_trial][n_frame][n_thorax_kp][3], in the input type: the statistics' contributions are ADDED to them
 *   grad_consts  NULL (skip), or [n_trial][5] out
 *   scratch: NULL for recordings of up to 1024 frames (one CTA per trial), else n_trial * 5 * (n_frame + 12) 32-bit words.
 * With H = grad_affine[trial], a = affine[trial] and s_j the five mid-quantiles (base x, y, z, d, |tip - base|), recomputed
 * from the selected keys with the forward's float32 arithmetic:
 *   dL/ds = (H0, H1, H2, -(H3 a3) / s3, -(H7 a7) / s4),   grad_consts = (H4, H5, H6, H3 / s3, H7 / s4).
 * Series j has m = counts[trial][j] values (the stationary frames for j = 0..3, every frame for j = 4); its mid-quantile
 * passes dL/ds_j to its four order statistics with the weights of seqik_leg_affine_backward_f32 for m values, a share being
 * weight * dL/ds_j in float32.  Tie rule: keys are the order keys of the float32 series values; the rank-r statistic sits in
 * frame argsort(row keys, stable)[r].  The +inf padding sorts last and is never selected: finite inputs are the contract.
 * With sh = the share rounded to the input type T, a frame t receives, in T:
 *   j = 0..2: base[t][j] += sh
 *   j = 3:    u = (b - 0.5 (t0 + t_last)) / d in float64 (b, t0 = thorax[t][0], t_last = thorax[t][k-1]; the arithmetic of
 *             the series kernel) rounded to T, c = sh u:  base[t] += c, then thorax[t][0] -= 0.5 c, then thorax[t][k-1] -= 0.5 c
 *             (for k = 1 both go to the same point)
 *   j = 4:    v = (tip - base) / |tip - base| in float64 rounded to T, c = sh v:  tip[t] += c, then base[t] -= c
 *   a distance or length of exactly 0 contributes 0; a series with m = 0 scatters nothing (its s_j is NaN, and so is the
 *   grad_consts entry that divides by it).
 * One thread per trial adds in a fixed order (series 0..4, sorted rank position 0..3, the points in the order above, x, y, z),
 * so the result is deterministic.  Error bound against the float64 VJP at the same frames (u = 2^-24), in either type: per
 * element of grad_head / grad_thorax 64 u N A, N the contributions it receives and A the sum of their absolute values;
 * 16 u |dL/dconsts| for grad_consts.  Size, NULL and n_thorax_kp errors are the forward's; an empty recording is an error. */
int seqik_head_affine_backward_f32(const float* head, const float* thorax, int64_t n_thorax_kp, const float* series,
                                   const int32_t* counts, const float* consts, const float* affine, const float* grad_affine,
                                   float* grad_head, float* grad_thorax, float* grad_consts, uint32_t* scratch,
                                   int64_t n_trial, int64_t n_frame, void* stream);
int seqik_head_affine_backward_f64(const double* head, const double* thorax, int64_t n_thorax_kp, const float* series,
                                   const int32_t* counts, const float* consts, const float* affine, const float* grad_affine,
                                   double* grad_head, double* grad_thorax, float* grad_consts, uint32_t* scratch,
                                   int64_t n_trial, int64_t n_frame, void* stream);

/* Shape-preserving cubic (pchip) resampling of uniformly sampled series onto a finer or coarser uniform grid: the hand-off
 * of joint angles to a simulation time step.  Replaces utils.interpolate_signal / interpolate_joint_angles
 * (seqikpy/utils.py:332-359) = scipy.interpolate.pchip_interpolate(arange(0, n*ts, ts), y, arange(0, n*ts, new_ts)),
 * including the extrapolation of the last cubic piece over the samples of the new grid that lie past the last knot.
 *   in  [n_block][n][width], out [n_block][m][width], m = ceil(n * original_ts / new_ts) (the length of numpy's arange);
 *   width = interleaved channels (7 for an angles tensor [n_chain][n_frame][7], 1 for plain series [n_series][n]).
 * Values must be finite (scipy raises otherwise; the reference's retry zeroes +-inf samples and the last sample first:
 * the host wrapper does the same). */
int seqik_pchip_resample_f32(const float* in, float* out, int64_t n_block, int64_t n, int64_t m, int64_t width,
                             double original_ts, double new_ts, void* stream);
int seqik_pchip_resample_f64(const double* in, double* out, int64_t n_block, int64_t n, int64_t m, int64_t width,
                             double original_ts, double new_ts, void* stream);

/* Backward of seqik_pchip_resample_f32/_f64 (vector-Jacobian product): grad_in = dL/din given grad_out = dL/dout.  New in
 * this library: the reference has no gradients, so this replaces nothing in it.
 *   in [n_block][n][width], grad_out [n_block][m][width] in, grad_in [n_block][n][width] out; sizes, limits and error
 *   codes are those of the forward (n >= 2, positive steps, width <= 256; n_block = 0 or width = 0 returns OK).
 *   grad_in is written in full, zeros included (it may be uninitialised).  in must hold the values the forward was
 *   given (finite; the host wrapper zeroes +-inf as for the forward and gives the replaced samples gradient 0).
 * The VJP is taken at the samples the forward evaluated: the same sample-to-interval assignment (the float64 interval
 * search) and the same offsets s from the left knot (float64; in float32 the forward's fmaf(u - u_lo, (float)new_ts, s0)).
 * A sample in interval k is y_k + d_k s + c1 s^2 + c0 s^3 with h = original_ts, m_k = (y_{k+1} - y_k) / h,
 * c1 = (3 m_k - 2 d_k - d_{k+1}) / h and c0 = (d_k + d_{k+1} - 2 m_k) / h^2.  The knot slopes d are differentiated on the
 * branch the forward took, its decisions recomputed with its arithmetic (in float32 with its __fdividef): an interior
 * d = 2ab / (a + b) of the neighbouring secants, or 0 (gradient 0) where they differ in sign or one is 0; an end slope
 * (3 m0 - m1) / 2 (partials 3/2 and -1/2), or zeroed (gradient 0), or clamped to 3 m0 (d/dm0 = 3, d/dm1 = 0); for n = 2
 * d_0 = d_1 = m_0.
 * Float summation order: per interval the moments M_p = sum g s^p (p = 0..3) in ascending sample order; then per knot
 * dL/dd_i = (right term of interval i-1) + (left term of interval i), times the slope partials; per interval
 * dL/dm_k = direct term + (knot k) + (knot k+1) [+ (knot 0) for k = 1] [+ (knot n-1) for k = n-3]; and
 * dL/dy_i = M0[i] + (dL/dm_{i-1} - dL/dm_i) * (1 / h).  Deterministic (no atomics); the result does not depend on the
 * width's launch path, the pointers' alignment, or whether grad_out is staged in shared memory or read directly. */
int seqik_pchip_resample_backward_f32(const float* in, const float* grad_out, float* grad_in, int64_t n_block, int64_t n,
                                      int64_t m, int64_t width, double original_ts, double new_ts, void* stream);
int seqik_pchip_resample_backward_f64(const double* in, const double* grad_out, double* grad_in, int64_t n_block,
                                      int64_t n, int64_t m, int64_t width, double original_ts, double new_ts, void* stream);

/* Strided copy between host (pinned) and device buffers: `height` rows of `width_bytes`, row pitches in bytes.
 * direction 1 = host to device, 2 = device to host.  Plumbing for the chunked host pipeline (a frame range of a
 * chain-major array is a 2-D block); a thin wrapper over cudaMemcpy2DAsync so that callers need no CUDA binding. */
int seqik_memcpy2d_async(void* dst, int64_t dst_pitch_bytes, const void* src, int64_t src_pitch_bytes,
                         int64_t width_bytes, int64_t height, int direction, void* stream);

/* HOST-side helper of the joints-only wire format (SEQIK_FLAG_FK_JOINTS over the host link, the reference's layout in host
 * memory): rebuilds fk [n_chain][n_frame][9][3] (leg_inverse_kinematics.py:71-77: rows 0-3 = origin, 4-5 = Coxa-Femur joint,
 * 6-8 = the other joints) for frames [t0, t1) from joints [n_chain][n_frame][4][3] and row 0 of the HOST pose.  All pointers
 * are HOST pointers here; strides in floats; chains are split over n_threads host threads; synchronous. */
int seqik_fk_expand_host_f32(const float* joints, int64_t j_chain_stride, int64_t j_frame_stride,
                             const float* pose, int64_t p_chain_stride, int64_t p_frame_stride,
                             float* fk, int64_t f_chain_stride, int64_t f_frame_stride,
                             int64_t n_chain, int64_t t0, int64_t t1, int n_threads);

/* DEVICE side of the same wire format: out [n_chain][..][3] (chain stride out_chain_stride floats, frame stride 3) receives
 * key point 0 of frames [t0, t1) of pose [n_chain][..][>= 3].  Shipped next to the joint rows it lets the host rebuild rows
 * 0-3 from 12 contiguous bytes per leg-frame (pass it to seqik_fk_expand_host_f32 as `pose` with p_frame_stride = 3) instead
 * of walking the 60-byte-per-frame host pose: 88 instead of 136 result bytes per leg-frame on the link. */
int seqik_origin_rows_f32(const float* pose, int64_t pose_chain_stride, int64_t pose_frame_stride, float* out,
                          int64_t out_chain_stride, int64_t n_chain, int64_t t0, int64_t t1, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SEQIK_H_ */
