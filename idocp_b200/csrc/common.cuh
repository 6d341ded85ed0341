// common.cuh -- device-side problem description and HBM layout of a batch of OCP instances.
#pragma once
#include "octet.cuh"

#ifdef IDOCP_B200_EMU
#define IDOCP_DYN_SMEM(type, name) type* name = reinterpret_cast<type*>(emu::g_block->smem.data())
#else
#define IDOCP_DYN_SMEM(type, name) extern __shared__ __align__(16) unsigned char name##_raw[]; \
  type* name = reinterpret_cast<type*>(name##_raw)
#endif

namespace idocp_b200 {

constexpr int NC = 6;         // constraint components: pos lo/up, vel lo/up, torque lo/up
constexpr int MODEL_STRIDE = 24;  // doubles per joint in the model table

// per-joint model table (one row per lane, row 7 = padding joint with zero mass):
//  [0..8] placement R (row-major)  [9..11] placement p  [12] mass  [13..15] com  [16..21] inertia
struct DevProblem {
  int N;
  double T, dt;
  double q_ref[8], v_ref[8], u_ref[8];
  double q_weight[8], v_weight[8], a_weight[8], u_weight[8], qf_weight[8], vf_weight[8];
  double q_min[8], q_max[8], v_max[8], u_max[8];
  double barrier, fraction_rate;
  double gravity;
  double model[8 * MODEL_STRIDE];
  // TimeVaryingTaskSpace6DCost on the end-effector frame (task_space_cost.cuh): frame placement in the last
  // joint's frame [R row-major (9), p (3)] and the weights in the reference's internal order, i.e. applied
  // to diff_6d = [linear; angular]: w6 = [rotation_weight, position_weight]
  // (src/cost/time_varying_task_space_6d_cost.cpp:43-58)
  int task_enabled;
  double ee[12];
  double task_w6[6], task_wf6[6];
  // JointAccelerationLowerLimit / JointAccelerationUpperLimit (src/constraints/joint_acceleration_*_limit.cpp): amin <= a <= amax
  int acc_enable[2];
  double a_min[8], a_max[8];
};

// ---------------------------------------------------------------------------------------------
// HBM layout.  A SLOT is one 64-byte vector (8 doubles: 7 joints + pad) of one instance.  Four
// consecutive instances form a GROUP (= the 4 octets of one warp); every array is
//     [stage][group][slot][4 instances][8 lanes]
// so that (i) one warp-wide load/store of a slot is 256 contiguous, aligned bytes, (ii) all slots
// of one (stage, group) record are contiguous (a few KB: DRAM-page friendly), and (iii) inside a
// kernel a slot is addressed as  record_base + slot * 32  with a compile-time constant offset.
// ---------------------------------------------------------------------------------------------
constexpr int SLOT = 32;  // doubles per (slot, group)

// stage state X: solution + interior-point state                      [N+1 stages]
enum XSlot { X_LMD = 0, X_GMM, X_Q, X_V, X_A, X_U, X_BETA, X_SLACK = 7, X_DUAL = 13, X_NUM = 19 };
// condensed KKT system KQ written by k_linearize: six 7x7 blocks (slot = row, lane = column)
// and the residual [Fq,Fv,la,lq,lv]                                   [N stages]
enum KQSlot { KQ_AA = 0, KQ_AQ = 7, KQ_AV = 14, KQ_QQ = 21, KQ_QV = 28, KQ_VV = 35,
              KQ_FQ = 42, KQ_FV, KQ_LA, KQ_LQ, KQ_LV, KQ_NUM = 47 };
// factor data W: Riccati gains (rows of Kq, Kv; k), Riccati matrices (columns of Pqq,Pqv,Pvv;
// sq,sv) and the expansion data of the condensed inverse dynamics (ID, lu, Quu diag, rows of
// dID/dq and dID/dv, column of M)                                    [N stages]
// (Pvq = Pqv^T is NOT stored: k_expand transposes Pqv through shared memory -- 7 slots less to write and re-read)
enum WSlot { W_KQ = 0, W_KV = 7, W_K = 14, W_PQQ = 15, W_PQV = 22, W_PVV = 29, W_SQ = 36, W_SV = 37,
             W_ID = 38, W_LU = 39, W_QUU = 40, W_DQ = 41, W_DV = 48, W_M = 55, W_NUM = 62 };
// Newton direction D                                                  [N+1 stages]
enum DSlot { D_LMD = 0, D_GMM, D_Q, D_V, D_A, D_U, D_BETA, D_NUM = 7 };

struct Layout {
  int B;     // instances
  int Bp;    // padded to a multiple of 4
  int G;     // groups = Bp / 4
  int N;     // stages with controls; X and D have N+1 stages
  double* X;
  double* X2;        // ping-pong partner of X (k_linearize<.., FUSED>: old iterate in X, new iterate in X2; the host swaps them)
  double* KQ;
  double* W;
  double* D;
  double* smin;       // [2][N][Bp] per-stage fraction-to-boundary minima (primal, dual)
  double* steps;      // [3][Bp] primal step applied, dual step, fraction-to-boundary primal step
  double* kkt_stage;  // [N+1][Bp] squared KKT norms per stage
  double* kkt_err;    // [Bp]
  int* status;        // [Bp]
  double* task_ref;   // [N+1][12] host-sampled SE3 reference per stage index (R row-major, p); see capi.cu
  double* XA;         // [N][G][XA_NUM slots]: slack (lower, upper), dual (lower, upper) of the two acceleration-limit components;
                      // nullptr unless one of them is enabled (the X record and the hot kernels stay as they are otherwise)
  // per-instance cost references (idocp_b200_set_instance_reference / _task_reference); nullptr in shared mode, where the
  // kernels read DevProblem::q_ref / v_ref / u_ref and task_ref.  Read only by the IREF kernel instantiations.
  double* iref;       // [G][IREF_NUM slots]: q_ref, v_ref, u_ref of every instance in the slot layout of X
  double* itask;      // [N+1][Bp][12]: task-space reference of every (stage row, instance), rows as task_ref
};
constexpr int XA_NUM = 4;
enum IrefSlot { IREF_Q = 0, IREF_V, IREF_U, IREF_NUM };

// The ConfigurationSpaceCost reference (slot IREF_Q / _V / _U) of this lane's joint in instance group g: the instance's own
// in per-instance mode (IREF and L.iref set), the problem's otherwise
template <bool IREF, int FIELD>
__device__ __forceinline__ double cfg_ref(const DevProblem& P, const Layout& L, int g, int lane) {
  if (IREF && L.iref) return L.iref[(static_cast<size_t>(g) * IREF_NUM + FIELD) * SLOT + (threadIdx.x & 31)];
  return FIELD == IREF_Q ? P.q_ref[lane] : (FIELD == IREF_V ? P.v_ref[lane] : P.u_ref[lane]);
}
// row `row` of the task-space reference table of instance b: its own table (IREF and L.itask set) or the shared one
template <bool IREF>
__device__ __forceinline__ const double* task_ref_row(const Layout& L, int row, int b) {
  if (IREF && L.itask) return L.itask + (static_cast<size_t>(row) * L.Bp + b) * 12;
  return L.task_ref + static_cast<size_t>(row) * 12;
}

// element index of (stage, instance b, slot, joint j) in an array with `ns` slots per record
__host__ __device__ __forceinline__ size_t elem_index(int ns, int G, int stage, int b, int slot, int j) {
  return ((static_cast<size_t>(stage) * G + (b >> 2)) * ns + slot) * SLOT + (b & 3) * OCT + j;
}
// this thread's pointer into the record of (stage, group g): add slot * SLOT to address a slot
__device__ __forceinline__ double* rec_ptr(double* base, int ns, int G, int stage, int g) {
  return base + (static_cast<size_t>(stage) * G + g) * (static_cast<size_t>(ns) * SLOT) + (threadIdx.x & 31);
}

// constraint activity by time stage (reference constraints/constraints_data.hpp:18-43)
__device__ __forceinline__ bool pos_active(int time_stage) { return time_stage >= 2; }
__device__ __forceinline__ bool vel_active(int time_stage) { return time_stage >= 1; }

}  // namespace idocp_b200
