// vss_render_emu.cpp — TEST HARNESS: runs the product's per-pixel picture code (csrc/vss_render.cuh, the
// exact source the vss_render kernel compiles) on the host, so the picture can be checked against the numpy
// restatement (oracle/vss_render.py) in a GPU-less build. The loop mirrors k_render in csrc/vss_step.cu: one
// 16-pixel segment at a time, packed into the same 48 bytes.
// Not part of the product: libvss_b200.so has no host execution path.
#include <cstdint>
#include <cstring>

#include "../../rsoccer_isaac_cleanrl_b200/csrc/vss_render.cuh"

using namespace vss;

extern "C" {

// Frames (num_fields, height, width, 3) of fields [first, first + num_fields) of the SoA state (60 x ld).
// Returns -1 for a size the kernel rejects (height / width not a multiple of 16 in [64, 4096]).
__attribute__((visibility("default"))) int emu_render(const vss_params* p, const float* state, long long ld,
                                                      long long first, int num_fields, int height, int width,
                                                      uint8_t* rgb) {
  if (height % 16 || width % 16 || height < 64 || height > 4096 || width < 64 || width > 4096) return -1;
  const RenderFrame g = render_frame(*p, height, width);
  for (int fr = 0; fr < num_fields; ++fr) {
    float f[RENDER_WORDS];
    for (int k = 0; k < RENDER_WORDS; ++k) f[k] = state[(long long)render_word(k) * ld + first + fr];
    for (int i = 0; i < height; ++i)
      for (int j0 = 0; j0 < width; j0 += 16) {
        uint32_t w[12];
        render_segment(g, f, i, j0, w);
        memcpy(rgb + (((long long)fr * height + i) * width + j0) * 3, w, sizeof(w));
      }
  }
  return 0;
}

}  // extern "C"
