// Lens-network (codes/config/latent-bokeh) additions to the NAFNet kernels of nafnet.cu.  Kept out of common.cuh, which is
// one of the sources the tcgen05 conv kernel compiles from (build.py conv_tc_sha256 names its profiles).
#pragma once
#include "common.cuh"

namespace irsde {

// per-image affine after the FFN SimpleGate of the lens network: row (b * img_stride) of the camera table [rows][S] holds
// (cam_scale[c], cam_shift[c]) of a block at `off`; img_stride 0 = one lens row shared by the batch
struct CamMod {
  const float* cam;  // null: plain SimpleGate
  int S, off, img_stride, pix_per_img;
};
// g = SimpleGate(x) * (cam_scale + 1) + cam_shift over B images of npix / B pixels each
template <typename T>
void launch_simple_gate(const T* x, int x_pitch, T* out, int o_pitch, long long npix, int c, cudaStream_t st, const CamMod& cam,
                        int B);
// rows x k scalars -> SimpleGate(Linear(SimpleGate(Linear(cat_k [sin, cos](scalar))))) [rows][2w]; k = 1 is
// launch_naf_time_gate, k = 3 the lens network's camera embedding (cam_mlp)
void launch_naf_time_gate_k(const float* times, int rows, int k, int width, const float* w1, const float* b1, const float* w2,
                            const float* b2, float* tgate, cudaStream_t st);

}  // namespace irsde
