// incrementState_IMUCam (reference src/orcvio.cpp:4468-4567) as a CTA-wide device routine shared by
// every kernel that ends in a state increment (k_pinfo, k_zupt).
#pragma once
#include "kernels.h"

namespace ob {

// dxs: delta_x (D = 22 + 6N) in shared memory, already visible to the whole CTA.
// apply_log: optional slot that receives 1.0 / 0.0 (large-update guard, :4479-4494).
// Must be called by every thread of the CTA (contains a barrier).  Returns the guard's verdict.
//
// A dependent FP64 operation costs ~35 cycles on this GPU, so the scalar exp maps are pure latency: the IMU
// increment (thread 0) and the N clone increments (threads 32 .. 32 + N, another warp) run side by side, and
// every participating thread evaluates the guard and the extrinsic increment for itself instead of waiting
// for thread 0 to publish them.
__device__ __forceinline__ bool cta_increment_state(const double* dxs, double* imu, double* clones, int N, int flags,
                                                    double* apply_log) {
  const int tid = threadIdx.x;
  const int cbase = (blockDim.x >= 64) ? 32 : 0;          // first clone thread
  const int ci = tid - cbase;
  const bool is_clone = (ci >= 0 && ci < N);
  double rbc[9], tcb[3];
  for (int i = 0; i < 9; ++i) rbc[i] = imu[IM_RBC + i];
  for (int i = 0; i < 3; ++i) tcb[i] = imu[IM_TCB + i];
  __syncthreads();                                         // old extrinsics are in registers before thread 0 writes
  const double nv = sqrt((dxs[3] * dxs[3] + dxs[4] * dxs[4]) + dxs[5] * dxs[5]);
  const double np = sqrt((dxs[6] * dxs[6] + dxs[7] * dxs[7]) + dxs[8] * dxs[8]);
  const bool apply = !((nv > 1.0 || np > 1.5) && (flags & FL_DISCARD_LARGE));
  if (tid == 0) {
    if (!apply) imu[IM_DISCARDS] += 1.0;
    if (apply_log) *apply_log = apply ? 1.0 : 0.0;
  }
  if (!apply || !(tid == 0 || is_clone)) return apply;
  const bool left = (flags & FL_LARVIO) || (flags & FL_LEFT);
  // extrinsics / td (:4513-4520); dx is exactly zero there unless estimated
  double Rb[9], tcn[3];
  {
    double dq[3] = {dxs[15] / 2.0, dxs[16] / 2.0, dxs[17] / 2.0};
    double n2 = (dq[0] * dq[0] + dq[1] * dq[1]) + dq[2] * dq[2];
    double qw, qs = 1.0;
    if (n2 <= 1) qw = sqrt(1 - n2);
    else { qw = 1; qs = 1.0 / sqrt(1 + n2); }
    double Rq[9];
    quat_wxyz_to_R(qw * qs, dq[0] * qs, dq[1] * qs, dq[2] * qs, Rq);
    m3_mulT(rbc, Rq, Rb);
    for (int i = 0; i < 3; ++i) tcn[i] = tcb[i] + dxs[18 + i];
  }
  if (tid == 0) {
    double Rt[9], Rn[9];
    so3_exp(dxs, Rt);
    if (left) m3_mul(Rt, imu + IM_R, Rn);
    else m3_mul(imu + IM_R, Rt, Rn);
    for (int i = 0; i < 9; ++i) imu[IM_R + i] = Rn[i];
    for (int i = 0; i < 3; ++i) {
      imu[IM_V + i] += dxs[3 + i];
      imu[IM_P + i] += dxs[6 + i];
      imu[IM_BG + i] += dxs[9 + i];
      imu[IM_BA + i] += dxs[12 + i];
    }
    for (int i = 0; i < 9; ++i) imu[IM_RBC + i] = Rb[i];
    for (int i = 0; i < 3; ++i) imu[IM_TCB + i] = tcn[i];
    imu[IM_TD] += dxs[21];
  }
  if (is_clone) {
    double* c = clones + (size_t)ci * CL_STRIDE;
    const double* d = dxs + ORCVIO_LEG + 6 * ci;
    double Rt[9], Rn[9];
    so3_exp(d, Rt);
    if (left) m3_mul(Rt, c + CL_R, Rn);
    else m3_mul(c + CL_R, Rt, Rn);
    for (int i = 0; i < 9; ++i) c[CL_R + i] = Rn[i];
    for (int i = 0; i < 3; ++i) c[CL_P + i] += d[3 + i];
    double Rc[9], t[3];
    m3_mulT(Rn, Rb, Rc);               // R_b2w * R_b2c^T
    m3_vec(Rn, tcn, t);
    for (int i = 0; i < 9; ++i) c[CL_RC + i] = Rc[i];
    for (int i = 0; i < 3; ++i) c[CL_PC + i] = c[CL_P + i] + t[i];
  }
  return apply;
}

}  // namespace ob
