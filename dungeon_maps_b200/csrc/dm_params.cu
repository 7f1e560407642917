// Host-side packing of the kernels' per-sample parameter blocks, in C.  The Python layer (_params.py) builds the
// same blocks with torch / numpy — correct, but 0.1-0.25 ms of interpreter time per call, which is what a caller
// with a fresh pose every frame pays (bench.py rotates poses: the ego-flow step went from 0.19 ms, kernel-bound, to
// 0.29 ms, host-bound).  Nothing here touches the device, and nothing here calls sin / cos: the yaw rotation is formed
// from sin / cos values the caller computed with the reference's own torch-CPU ops (utils.py:325-326, the last ulp
// matters; of the raw yaw — the |a| <= 0.001 clamp of utils.py:323-324 is applied here), by the float32 operations of
// utils.py:318-327 in the reference's order:
//     R = (I + sin(a) S) + (1 - cos(a)) S²        S, S² built by the caller exactly as utils.py:303-318 does.
// tests/test_abi.py checks these blocks byte for byte against _params.py and the oracle.
#include <cmath>
#include <cstring>

#include "dm_common.cuh"

namespace dm {

void yaw_matrix(const DmPoseCfg& c, float yaw, float s, float cos_a, float* R) {
  // utils.py:323-324: |angle| <= 0.001 rotates by exactly 0 — sin(0) = 0, cos(0) = 1, whatever the caller computed
  if (!(fabsf(yaw) > 0.001f)) { s = 0.0f; cos_a = 1.0f; }
  const float one_minus_cos = 1.0f - cos_a;
  for (int k = 0; k < 9; ++k) {
    const float eye = (k == 0 || k == 4 || k == 8) ? 1.0f : 0.0f;
    const float a = s * c.yaw_skew[k];
    const float e = eye + a;
    const float q = one_minus_cos * c.yaw_skew_sq[k];
    R[k] = e + q;
  }
}

void put_step(float* w, int kind, const float* R, const float* t, int fused) {
  memset(w, 0, sizeof(DmStep));
  if (kind == DM_STEP_NONE) return;
  if (R) memcpy(w, R, 9 * sizeof(float));
  if (t) memcpy(w + 9, t, 3 * sizeof(float));
  int32_t* iw = reinterpret_cast<int32_t*>(w);
  iw[12] = kind;
  iw[13] = fused;
}

bool local_step_is_fast(const DmPoseCfg& c) {
  const float* R = c.pitch_R;
  return c.fused && R[0] == 1.0f && R[1] == 0.0f && R[2] == 0.0f && R[3] == 0.0f && R[6] == 0.0f;
}

bool yaw_step_is_fast(const float* R) {
  return R[4] == 1.0f && R[1] == 0.0f && R[3] == 0.0f && R[5] == 0.0f && R[7] == 0.0f;
}

}  // namespace dm

using namespace dm;

extern "C" int dm_pack_proj_samples(const DmPoseCfg* cfg, const float* pose, const float* sin_yaw, const float* cos_yaw,
                                    const float* width_offset, const float* height_offset, int32_t to_global,
                                    int32_t b, DmProjSample* out, int32_t* fast_steps) {
  if (!cfg || !width_offset || !height_offset || !out || b < 0) return DM_EINVAL;
  if (to_global && (!pose || !sin_yaw || !cos_yaw)) return DM_EINVAL;
  int fast = local_step_is_fast(*cfg) ? (to_global ? 2 : 1) : 0;
  const float tl[3] = {0.0f, cfg->cam_height, 0.0f};  // maps.py:795-797
  for (int i = 0; i < b; ++i) {
    float* sp = reinterpret_cast<float*>(out + i);
    memset(sp, 0, sizeof(DmProjSample));
    put_step(sp, DM_STEP_ROT_THEN_ADD, cfg->pitch_R, tl, cfg->fused);
    if (to_global) {
      float Ry[9];
      yaw_matrix(*cfg, pose[3 * i + 2], sin_yaw[i], cos_yaw[i], Ry);
      const float ty[3] = {pose[3 * i + 0], 0.0f, pose[3 * i + 1]};  // maps.py:889-891
      put_step(sp + 16, DM_STEP_ROT_THEN_ADD, Ry, ty, cfg->fused);
      if (fast == 2 && !yaw_step_is_fast(Ry)) fast = 0;
    }
    sp[32] = width_offset[i];
    sp[33] = height_offset[i];
  }
  if (fast_steps) *fast_steps = fast;
  return DM_OK;
}

extern "C" int dm_pack_flow_samples(const DmPoseCfg* cfg, const float* pose, const float* sin_yaw, const float* cos_yaw,
                                    int32_t b, DmFlowSample* out) {
  if (!cfg || !pose || !sin_yaw || !cos_yaw || !out || b < 0) return DM_EINVAL;
  const float tl[3] = {0.0f, cfg->cam_height, 0.0f};    // maps.py:795-797
  const float tb[3] = {0.0f, -cfg->cam_height, 0.0f};   // maps.py:843-845
  for (int i = 0; i < b; ++i) {
    float* sp = reinterpret_cast<float*>(out + i);
    float Ry[9];
    yaw_matrix(*cfg, pose[3 * i + 2], sin_yaw[i], cos_yaw[i], Ry);
    const float ty[3] = {pose[3 * i + 0], 0.0f, pose[3 * i + 1]};
    put_step(sp, DM_STEP_ROT_THEN_ADD, cfg->pitch_R, tl, cfg->fused);          // camera_to_local_space
    put_step(sp + 16, DM_STEP_ROT_THEN_ADD, Ry, ty, cfg->fused);               // local_to_global_space(trans_pose)
    put_step(sp + 32, DM_STEP_ADD_THEN_ROT, cfg->pitch_back_R, tb, cfg->fused);  // local_to_camera_space
  }
  return DM_OK;
}

extern "C" int dm_pack_ego_samples(const DmPoseCfg* cfg, const float* pose, const float* sin_yaw, const float* cos_yaw,
                                   const float* src_width_offset, const float* src_height_offset,
                                   const float* width_offset, const float* height_offset, int32_t b, float* out) {
  if (!cfg || !pose || !sin_yaw || !cos_yaw || !src_width_offset || !src_height_offset || !width_offset ||
      !height_offset || !out || b < 0)
    return DM_EINVAL;
  for (int i = 0; i < b; ++i) {
    float* sp = out + (size_t)i * DM_EGO_SAMPLE_WORDS;
    float Ry[9];
    yaw_matrix(*cfg, pose[3 * i + 2], sin_yaw[i], cos_yaw[i], Ry);
    const float ty[3] = {pose[3 * i + 0], 0.0f, pose[3 * i + 1]};  // maps.py:889-891
    put_step(sp, DM_STEP_ROT_THEN_ADD, Ry, ty, cfg->fused);           // local_to_global_space
    sp[16] = src_width_offset[i];
    sp[17] = src_height_offset[i];
    sp[18] = width_offset[i];
    sp[19] = height_offset[i];
  }
  return DM_OK;
}
