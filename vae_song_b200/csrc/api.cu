// api.cu -- extern "C" entry points of libb200vae.so for the ICNN path (validation + dispatch).
#include <mutex>
#include <unordered_map>

#include "icnn.cuh"

namespace b200vae {
int g_last_cuda_error = 0;
long long g_launch_count = 0;

int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
      n = 148;
  }
  return n;
}

// ---- saved GEMM2 accumulators (training, 3xTF32) ------------------------------------------------------------------------
// With a for_backward workspace and both masks requested, the pair forward kernel also stores its GEMM2 accumulators
// (gx1 / s2, [Bp][Hq] fp32) at the end of the workspace; the backward then skips recomputing that GEMM (icnn_tc3.cu, SV
// kernels).  Which workspace holds a valid save -- and for which (z, B, d, H) -- is tracked HERE on the host, in call
// order (= stream order for one stream; a CUDA-graph capture records the same decision it replays): prepare invalidates,
// a saving forward validates, the backward uses the save only on an exact match and otherwise recomputes.
struct SavedAcc { const void* z; int B, d, H; };
static std::mutex g_save_mu;
static std::unordered_map<const void*, SavedAcc> g_saved;
static void save_forget(const void* ws) {
  std::lock_guard<std::mutex> lk(g_save_mu);
  g_saved.erase(ws);
}
static void save_record(const void* ws, const void* z, int B, int d, int H) {
  std::lock_guard<std::mutex> lk(g_save_mu);
  if (g_saved.size() > 1024) g_saved.clear();
  g_saved[ws] = SavedAcc{z, B, d, H};
}
static bool save_matches(const void* ws, const void* z, int B, int d, int H) {
  std::lock_guard<std::mutex> lk(g_save_mu);
  auto it = g_saved.find(ws);
  return it != g_saved.end() && it->second.z == z && it->second.B == B && it->second.d == d && it->second.H == H;
}

// ---- workspace layout (icnn.cuh) ----------------------------------------------------------------------------------------
static int bwd_splits(int B, int Hp) {
  // output-stationary dP0 kernel of the FP32 path: (Hp/128)^2 tiles x splits CTAs; aim for >= ~3 waves of 148 SMs
  int tiles = (Hp / 128) * (Hp / 128);
  int want = (148 * 3 + tiles - 1) / tiles;
  int maxs = (B + 127) / 128;          // at least one 128-row slab per split
  int s = want < maxs ? want : maxs;
  if (s < 1) s = 1;
  if (s > 64) s = 64;
  return s;
}

WsLayout icnn_ws_layout(int B, int d, int H, int precision, bool for_backward) {
  WsLayout L = {};
  L.B = B; L.d = d; L.H = H;
  L.Hp = round_up(H, 128); L.Hq = round_up(H, 256); L.K1 = L.Hq + 16; L.NP = L.Hq / 256; L.Bp = round_up(B, 256);
  L.n_mtiles = (B + 127) / 128;
  L.splits = bwd_splits(B, L.Hp);
  const size_t Hp = L.Hp, Hq = L.Hq, Bp = L.Bp, NP = L.NP, tiles = Bp / 256;
  const bool tc = precision != B200VAE_PREC_FP32;
  size_t o = 0;
  auto take = [&o](size_t n) { const size_t at = o; o += (n + 63) / 64 * 64; return at; };   // 256 B aligned regions
  L.P0 = take(Hp * Hp);
  L.P0T = take(Hp * Hp);
  L.P1 = take(Hp);
  L.A0p = take(Hp * (d + 1));
  L.A1p = take(Hp * (d + 1));
  L.A2p = take(16 > d + 1 ? 16 : d + 1);
  if (tc) {
    L.A0q = take(4 * Hq); L.A1q = take(4 * Hq); L.P1q = take(Hq);
    L.B1ahi = take(Hq * L.K1); L.B1alo = take(Hq * L.K1); L.B2ghi = take(Hq * Hq); L.B2glo = take(Hq * Hq);
    L.A0g = take(4 * Hq); L.E1 = take(4 * Hq); L.sumV = take(64); L.cnt = take(2 * kTc3MaxTiles);
    L.scr1 = take(Bp * NP * 2 * 4); L.scr2 = take(Bp * NP * 2 * 4); L.imask = take(Bp * (Hq / 32));
    const size_t units = 2 * tiles * NP;
    L.cscr = take((units < (size_t)kTc3MaxClusters ? units : (size_t)kTc3MaxClusters) * 2 * k3ScrFloatsPerCta);
  }
  if (for_backward) {
    L.colpart = take((size_t)L.n_mtiles * Hp * (2 * d + 3));
    L.a2part = take((size_t)L.n_mtiles * (d + 1));
    L.dP0part = take((size_t)L.splits * Hp * Hp);
    if (tc) {
      L.dp0_splits = dp0_splits(B, L.Hq, sm_count() / 2);
      L.partA = take(tiles * 8 * (d + 1) * Hq); L.partB = take(tiles * 8 * (d + 1) * Hq);
      L.a2part_tc = take(tiles * d);
      L.dP0part_tc = take((size_t)L.dp0_splits * Hq * Hq);
      L.dzpart = take(Bp * NP * 2 * 4);
      if (precision == B200VAE_PREC_TF32X3 || precision == B200VAE_PREC_F16X3) L.accsave = take(Bp * Hq);
    }
  }
  L.end = o;
  return L;
}
static size_t ws_bytes_of(const WsLayout& L) { return L.end * sizeof(float) + 256; }   // + alignment of the base

static bool params_ok(const b200vae_icnn_params* p) {
  return p && p->A0w && p->A0b && p->A1w && p->A1b && p->A2w && p->A2b && p->W0 && p->W1 && aligned4(p->A0w) &&
         aligned4(p->W0);
}
// every entry point's shape / precision check: FP32 takes d <= 4, H <= 4096; the tensor-core precisions d <= 3, H <= 1024
static int shape_ok(int B, int d, int H, int precision) {
  if (B <= 0 || d <= 0 || H <= 0) return B200VAE_ESHAPE;
  if (precision == B200VAE_PREC_FP32) return (d <= 4 && H <= 4096) ? B200VAE_OK : B200VAE_EUNSUP;
  if (precision != B200VAE_PREC_TF32 && precision != B200VAE_PREC_TF32X3 && precision != B200VAE_PREC_F16X3)
    return B200VAE_EUNSUP;                                     // 2 is reserved
  return (d <= 3 && round_up(H, 256) <= kTc3MaxHq) ? B200VAE_OK : B200VAE_EUNSUP;
}
}  // namespace b200vae

using namespace b200vae;

extern "C" size_t b200vae_icnn_workspace_bytes(int B, int d, int H, int precision, int for_backward) {
  if (shape_ok(B, d, H, precision)) return 0;
  return ws_bytes_of(icnn_ws_layout(B, d, H, precision, for_backward != 0));
}

static float* ws_base(const void* ws) {
  return reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
}

extern "C" int b200vae_icnn_prepare(const b200vae_icnn_params* p, int d, int H, int weight_mode, int precision,
                                    void* ws, size_t ws_bytes, void* stream) {
  int rc = shape_ok(1, d, H, precision);
  if (rc) return rc;
  if (!params_ok(p) || !ws) return B200VAE_EALIGN;
  if (weight_mode != B200VAE_WEIGHT_EXP && weight_mode != B200VAE_WEIGHT_CLAMP) return B200VAE_EUNSUP;
  const WsLayout L = icnn_ws_layout(1, d, H, precision, false);    // prepare writes only regions that do not depend on B
  if (ws_bytes < ws_bytes_of(L)) return B200VAE_EWS;
  save_forget(ws_base(ws));
  rc = simt_prepare(p, L, weight_mode, ws_base(ws), (cudaStream_t)stream);
  if (rc || precision == B200VAE_PREC_FP32) return rc;
  return tc3_prepare(L, precision, ws_base(ws), (cudaStream_t)stream);
}

extern "C" int b200vae_icnn_decode_fwd(const float* z, int B, int d, int H, int weight_mode, float kappa, float* psi,
                                       float* xhat, uint32_t* mask1, uint8_t* mask2, int precision, const void* ws,
                                       size_t ws_bytes, void* stream) {
  (void)weight_mode;
  if (!z || !ws || !aligned4(z)) return B200VAE_EALIGN;
  int rc = shape_ok(B, d, H, precision);
  if (rc) return rc;
  if (ws_bytes < b200vae_icnn_workspace_bytes(B, d, H, precision, 0)) return B200VAE_EWS;
  const WsLayout L = icnn_ws_layout(B, d, H, precision, true);     // the forward's regions sit where they do without backward
  if (precision == B200VAE_PREC_FP32)
    return simt_fwd(z, L, kappa, psi, xhat, mask1, mask2, ws_base(ws), (cudaStream_t)stream);
  float* accsave = nullptr;
  if (mask1 && mask2 && xhat && L.accsave && ws_bytes >= ws_bytes_of(L)) accsave = ws_base(ws) + L.accsave;
  save_forget(ws_base(ws));
  rc = tc3_fwd(z, L, kappa, psi, xhat, mask1, mask2, precision, ws_base(ws), accsave, (cudaStream_t)stream);
  if (rc == B200VAE_OK && accsave) save_record(ws_base(ws), z, B, d, H);
  return rc;
}

extern "C" int b200vae_icnn_decode_bwd(const float* z, const float* v, const float* gpsi, const uint32_t* mask1,
                                       const uint8_t* mask2, int B, int d, int H, const b200vae_icnn_params* p,
                                       int weight_mode, float kappa, const b200vae_icnn_grads* grads, float* dz,
                                       int precision, void* ws, size_t ws_bytes, void* stream) {
  if (!z || !mask1 || !mask2 || !ws || !params_ok(p)) return B200VAE_EALIGN;
  if (!v && !gpsi) return B200VAE_ESHAPE;
  int rc = shape_ok(B, d, H, precision);
  if (rc) return rc;
  const WsLayout L = icnn_ws_layout(B, d, H, precision, true);
  if (ws_bytes < ws_bytes_of(L)) return B200VAE_EWS;
  if (precision != B200VAE_PREC_FP32 && !gpsi) { // tensor-core backward (gpsi path stays on the FP32 kernels)
    const float* accsave = nullptr;
    if (L.accsave && save_matches(ws_base(ws), z, B, d, H)) accsave = ws_base(ws) + L.accsave;
    return tc_bwd(z, v, mask1, mask2, L, p, weight_mode, kappa, grads, dz, precision, ws_base(ws), accsave, 0,
                  (cudaStream_t)stream);
  }
  return simt_bwd(z, v, gpsi, mask1, mask2, L, p, weight_mode, kappa, grads, dz, ws_base(ws), (cudaStream_t)stream);
}

extern "C" int b200vae_icnn_decode_bwd_params(const float* z, const float* v, const uint32_t* mask1, const uint8_t* mask2,
                                              int B, int d, int H, const b200vae_icnn_params* p, int weight_mode,
                                              const b200vae_icnn_grads* grads, int precision, void* ws, size_t ws_bytes,
                                              void* stream) {
  if (!z || !v || !mask1 || !mask2 || !ws || !grads || !params_ok(p)) return B200VAE_EALIGN;
  int rc = shape_ok(B, d, H, precision);
  if (rc) return rc;
  if (precision == B200VAE_PREC_FP32) return B200VAE_EUNSUP;
  const WsLayout L = icnn_ws_layout(B, d, H, precision, true);
  if (ws_bytes < ws_bytes_of(L)) return B200VAE_EWS;
  return tc_bwd(z, v, mask1, mask2, L, p, weight_mode, 0.f, grads, nullptr, precision, ws_base(ws), nullptr, 2,
                (cudaStream_t)stream);
}

static size_t jac_scratch_of(const WsLayout& L) {
  return (size_t)L.Bp * L.NP * 2 * tc3_jac_slots(L.d) * sizeof(float4);
}

extern "C" size_t b200vae_icnn_jac_scratch_bytes(int B, int d, int H, int precision) {
  if (shape_ok(B, d, H, precision) || precision == B200VAE_PREC_FP32) return 0;
  return jac_scratch_of(icnn_ws_layout(B, d, H, precision, false));
}

extern "C" int b200vae_icnn_decode_jac(const float* z, int B, int d, int H, float kappa, float* psi, float* xhat, float* jac,
                                       uint32_t* mask1, uint8_t* mask2, int precision, const void* ws, size_t ws_bytes,
                                       void* jac_scratch, size_t jac_scratch_bytes, void* stream) {
  int rc = shape_ok(B, d, H, precision);
  if (rc) return rc;
  if (!z || !ws || !jac || !xhat || !aligned4(z)) return B200VAE_EALIGN;
  if (ws_bytes < b200vae_icnn_workspace_bytes(B, d, H, precision, 0)) return B200VAE_EWS;
  const WsLayout L = icnn_ws_layout(B, d, H, precision, false);
  if (precision == B200VAE_PREC_FP32)
    return simt_fwd_jac(z, L, kappa, psi, xhat, mask1, mask2, jac, ws_base(ws), (cudaStream_t)stream);
  if (!jac_scratch || (reinterpret_cast<uintptr_t>(jac_scratch) & 15)) return B200VAE_EALIGN;
  if (jac_scratch_bytes < jac_scratch_of(L)) return B200VAE_EWS;
  // no save_forget / save_record: this variant never writes the saved accumulators, so a save stays valid across it
  return tc3_fwd_jac(z, L, kappa, psi, xhat, mask1, mask2, jac, reinterpret_cast<float4*>(jac_scratch), precision,
                     ws_base(ws), (cudaStream_t)stream);
}

static int inverse_shape_ok(int B, int d) {
  if (B <= 0 || d <= 0) return B200VAE_ESHAPE;
  return d <= 4 ? B200VAE_OK : B200VAE_EUNSUP;
}

extern "C" size_t b200vae_brenier_inverse_state_bytes(int B, int d) {
  return inverse_shape_ok(B, d) ? 0 : inverse_state_bytes(B);
}

extern "C" int b200vae_brenier_inverse_init(const float* x, const float* z0, int B, int d, float tol_rel, float tol_abs,
                                            void* state, size_t state_bytes, float* z_trial, float* z, int* status,
                                            float* err_bound, void* stream) {
  int rc = inverse_shape_ok(B, d);
  if (rc) return rc;
  if (!x || !state || !z_trial || !z || !status || !err_bound || !aligned16(state) || !aligned4(x) ||
      (z0 && !aligned4(z0)))
    return B200VAE_EALIGN;
  if (state_bytes < inverse_state_bytes(B)) return B200VAE_EWS;
  return brenier_inverse_init(x, z0, B, d, tol_rel, tol_abs, state, z_trial, z, status, err_bound, (cudaStream_t)stream);
}

extern "C" int b200vae_brenier_newton_step(const float* x, const float* xhat, const float* jac, int B, int d, float kappa,
                                           int round, int final_round, void* state, size_t state_bytes, float* z_trial,
                                           float* z, int* status, float* err_bound, void* stream) {
  int rc = inverse_shape_ok(B, d);
  if (rc) return rc;
  if (round < 0) return B200VAE_ESHAPE;
  if (!x || !xhat || !jac || !state || !z_trial || !z || !status || !err_bound || !aligned16(state) || !aligned4(x) ||
      !aligned4(xhat) || !aligned4(jac))
    return B200VAE_EALIGN;
  if (state_bytes < inverse_state_bytes(B)) return B200VAE_EWS;
  return brenier_newton_step(x, xhat, jac, B, d, kappa, round, final_round, state, z_trial, z, status, err_bound,
                             (cudaStream_t)stream);
}

extern "C" int b200vae_last_cuda_error(void) { return g_last_cuda_error; }
extern "C" const char* b200vae_version(void) { return "b200vae 0.2 (sm_100a)"; }
extern "C" long long b200vae_launch_count(void) { return g_launch_count; }
