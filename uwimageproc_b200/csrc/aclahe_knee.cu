// aclahe_knee.cu - the knee search of ParametrosACLAHE on the device: one thread per (frame, block size) runs the curve fit,
// spline and curvature of csrc/aclahe_knee.h on entries 1..49 of the frame's entropy row, the clip limit of the frame is
// the largest of its five knees (ACLAHE.py:92-96).  This translation unit is built with --fmad=false: the header's double
// arithmetic must round like the reference's (no contraction into FMA).
#include "aclahe_knee.h"
#include "common.cuh"

constexpr int KN_GRIDS = 5;
constexpr int KN_FRAMES_PER_CTA = 32;

// the clip curve (0.5 .. 24.5) is the same for every frame: fitted once per call; xd[0] = x', xd[1] = x'' (NaN if the fit
// fails, which makes every knee fail like the reference's exception would)
__global__ void knee_x_kernel(double* __restrict__ xd) {
  if (threadIdx.x != 0) return;
  if (!knee::clip_curve_derivs(xd, xd + knee::NE))
    for (int i = 0; i < 2 * knee::NE; i++) xd[i] = __longlong_as_double(0x7ff8000000000000ll);
}

// ent: [grid][frame][n_clips] (the sweep's device layout); cl[f] = max of the knees, -1 when a fit fails
__global__ void __launch_bounds__(KN_GRIDS * KN_FRAMES_PER_CTA) knee_kernel(const float* __restrict__ ent, int n, int n_clips,
                                                                            const double* __restrict__ xd, int* __restrict__ cl) {
  __shared__ int s_knee[KN_FRAMES_PER_CTA][KN_GRIDS];
  const int fl = threadIdx.x / KN_GRIDS, gi = threadIdx.x % KN_GRIDS;
  const int f = blockIdx.x * KN_FRAMES_PER_CTA + fl;
  int k = -1;
  if (f < n && !(xd[0] != xd[0])) {
    float y[knee::M];
    const float* row = ent + ((size_t)gi * n + f) * n_clips;
    for (int i = 0; i < knee::M; i++) y[i] = row[1 + i];   // graficar: columns 2..50 of the 51-column table
    k = knee::knee_of(y, xd, xd + knee::NE);
  }
  s_knee[fl][gi] = k;
  __syncthreads();
  if (gi == 0 && f < n) {
    int c = 0;
    for (int j = 0; j < KN_GRIDS; j++) c = (s_knee[fl][j] < 0 || c < 0) ? -1 : max(c, s_knee[fl][j]);
    cl[f] = c;
  }
}

int k_aclahe_knees(uwip_ctx* ctx, const float* d_ent, int n, int n_clips, double* d_xd, int* d_cl) {
  UWIP_REQUIRE(ctx, n_clips >= 1 + knee::M, "the knee search needs 50 entropies per grid");
  UWIP_LAUNCH(ctx, "aclahe_knee_x", knee_x_kernel, 1, 32, 0, d_xd);
  UWIP_LAUNCH(ctx, "aclahe_knee", knee_kernel, cdiv(n, KN_FRAMES_PER_CTA), KN_GRIDS * KN_FRAMES_PER_CTA, 0, d_ent, n, n_clips,
              (const double*)d_xd, d_cl);
  return UWIP_OK;
}
