// api.cu — library-level C ABI: identification, status strings, launch counter, and the plugin-shaped
// enqueue / supportsFormatCombination mirrors for MSDA (reference: multiScaleDeformableAttnPlugin.cpp:71-189).
#include "common.cuh"

namespace b200 {
std::atomic<unsigned long long> g_launch_count{0};
}

using namespace b200;

extern "C" {

const char *b200_bev_ops_version(void) { return "b200_bev_ops 0.1.0 sm_100a"; }

const char *b200_status_string(int status) {
  switch (status) {
    case B200_OK: return "ok";
    case B200_ERR_UNSUPPORTED: return "unsupported dtype/format/shape";
    case B200_ERR_BAD_PARAM: return "bad parameter";
    case B200_ERR_LAUNCH: return "CUDA launch error";
    default: return "unknown status";
  }
}

unsigned long long b200_launch_count(void) { return g_launch_count.load(std::memory_order_relaxed); }

// IPluginV2DynamicExt::enqueue of the reference, argument for argument (…Plugin.cpp:71-140). Shape unpacking is the
// reference's: batch/spatial/heads/channels from value dims, L from shapes.d[0], G from ref.d[3]/2, Q from
// offsets.d[1], P from weights.d[3]/L; scales from the tensor descriptors (:75-88).
int b200_msda_enqueue(const b200_tensor_desc *in, const b200_tensor_desc *out, const void *const *inputs,
                      void *const *outputs, void *workspace, void *stream, int use_h2) {
  // The reference asks for 0 workspace bytes (…Plugin.cpp:64-69). A host that lends b200_msda_enqueue_workspace_size()
  // bytes gets the second-generation INT8 kernels (msda_v2.cu); workspace == NULL keeps the round-1 kernels.
  if (!in || !out || !inputs || !outputs) return B200_ERR_BAD_PARAM;
  const int batch = in[0].dims.d[0], spatial = in[0].dims.d[1], heads = in[0].dims.d[2], ch = in[0].dims.d[3];
  const int levels = in[1].dims.d[0];
  if (levels <= 0) return B200_ERR_BAD_PARAM;
  const int G = in[2].dims.d[3] / 2, Q = in[3].dims.d[1], P = in[4].dims.d[3] / levels;
  const int32_t *shapes = static_cast<const int32_t *>(inputs[1]);
  switch (in[0].type) {
    case 0:  // kFLOAT
      return b200_msda_f32(static_cast<const float *>(inputs[0]), shapes, static_cast<const float *>(inputs[2]),
                           static_cast<const float *>(inputs[3]), static_cast<const float *>(inputs[4]), batch,
                           spatial, heads, ch, levels, Q, P, G, static_cast<float *>(outputs[0]), stream);
    case 1:  // kHALF
      if (use_h2 && ch % 2 == 0)
        return b200_msda_f16_h2(inputs[0], shapes, inputs[2], inputs[3], inputs[4], batch, spatial, heads, ch, levels,
                                Q, P, G, outputs[0], stream);
      return b200_msda_f16(inputs[0], shapes, inputs[2], inputs[3], inputs[4], batch, spatial, heads, ch, levels, Q, P,
                           G, outputs[0], stream);
    case 2: {  // kINT8; reference points stay fp16 or fp32 (…Plugin.cpp:168-176)
      if (in[2].type != 0 && in[2].type != 1) return B200_ERR_UNSUPPORTED;
      const size_t ws = workspace ? b200_msda_i8_workspace_size(batch, spatial, heads, ch, levels, P, G) : 0;
      if (ws) {
        const int st = b200_msda_i8_ws(static_cast<const int8_t *>(inputs[0]), in[0].scale, shapes, inputs[2],
                                       in[2].type == 1, static_cast<const int8_t *>(inputs[3]), in[3].scale,
                                       static_cast<const int8_t *>(inputs[4]), in[4].scale, batch, spatial, heads, ch,
                                       levels, Q, P, G, static_cast<int8_t *>(outputs[0]), out[0].scale, workspace, ws,
                                       nullptr, stream);
        if (st != B200_ERR_UNSUPPORTED) return st;
      }
      return b200_msda_i8(static_cast<const int8_t *>(inputs[0]), in[0].scale, shapes, inputs[2], in[2].type == 1,
                          static_cast<const int8_t *>(inputs[3]), in[3].scale, static_cast<const int8_t *>(inputs[4]),
                          in[4].scale, batch, spatial, heads, ch, levels, Q, P, G, static_cast<int8_t *>(outputs[0]),
                          out[0].scale, stream);
    }
    default:
      return B200_ERR_UNSUPPORTED;
  }
}

// getWorkspaceSize mirror for the MSDA plugin shell: dimensions only, like the TensorRT call.
size_t b200_msda_enqueue_workspace_size(const b200_tensor_desc *in) {
  if (!in) return 0;
  const int levels = in[1].dims.d[0];
  if (levels <= 0) return 0;
  if (in[0].type != 2) return 0;  // kINT8 only
  return b200_msda_i8_workspace_size(in[0].dims.d[0], in[0].dims.d[1], in[0].dims.d[2], in[0].dims.d[3], levels,
                                     in[4].dims.d[3] / levels, in[2].dims.d[3] / 2);
}

int b200_msda_supports_format(int pos, const b200_tensor_desc *io, int nb_inputs, int nb_outputs) {
  if (!io || nb_inputs != 5 || nb_outputs != 1) return 0;
  const int levels = io[1].dims.d[0] > 0 ? io[1].dims.d[0] : 1;
  const int channels = io[0].dims.d[3], point_num = io[4].dims.d[3] / levels;
  const bool int8_ok = (channels % 4 == 0) && (point_num % 4 == 0);
  const bool linear = io[pos].format == 0;
  switch (pos) {
    case 0: return linear && (io[0].type == 0 || io[0].type == 1 || (io[0].type == 2 && int8_ok));
    case 1: return linear && io[1].type == 3;
    case 2:
      if (io[0].type == 0 || io[0].type == 1) return linear && io[2].type == io[0].type;
      return linear && (io[2].type == 0 || io[2].type == 1);
    case 3:
    case 4: return linear && io[pos].type == io[0].type;
    case 5: return io[5].type == io[0].type && io[5].format == io[0].format;
    default: return 0;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// GridSampler{2D,3D}TRT[2]: IPluginV2DynamicExt::enqueue / supportsFormatCombination of the reference, argument for
// argument (gridSamplerPlugin.cpp:110-155, :168-194). inputs: input, grid; attributes: interpolation_mode, padding_mode,
// align_corners (:277-288). Dispatch: fp32 / fp16 linear, fp16 kCHW2 (…TRT2), int8 kCHW4 with the descriptors' scales.
int b200_grid_sampler_enqueue(const b200_tensor_desc *in, const b200_tensor_desc *out, const void *const *inputs,
                              void *const *outputs, void *workspace, void *stream, int interpolation_mode,
                              int padding_mode, int align_corners) {
  (void)workspace;  // 0 bytes (gridSamplerPlugin.cpp:102-108)
  if (!in || !out || !inputs || !outputs) return B200_ERR_BAD_PARAM;
  const int nb = in[0].dims.nbDims;
  if (nb != 4 && nb != 5) return B200_ERR_BAD_PARAM;
  int id[5], gd[5], od[5];
  for (int i = 0; i < nb; ++i) id[i] = in[0].dims.d[i], gd[i] = in[1].dims.d[i], od[i] = out[0].dims.d[i];
  // The launcher writes N x C from the input and the spatial extent from the grid, whatever the output descriptor says:
  // an output that disagrees would be written past its end, so it is rejected before anything is launched.
  if (in[1].dims.nbDims != nb || out[0].dims.nbDims != nb || od[0] != id[0] || od[1] != id[1]) return B200_ERR_BAD_PARAM;
  for (int i = 2; i < nb; ++i)
    if (od[i] != gd[i]) return B200_ERR_BAD_PARAM;
  switch (in[0].type) {
    case 0:
      return b200_grid_sample_f32(static_cast<float *>(outputs[0]), static_cast<const float *>(inputs[0]),
                                  static_cast<const float *>(inputs[1]), od, id, gd, nb, interpolation_mode, padding_mode,
                                  align_corners, stream);
    case 1:
      if (in[0].format == 1 /* kCHW2 */) {
        if (nb != 4) return B200_ERR_UNSUPPORTED;
        return b200_grid_sample_f16_chw2(outputs[0], inputs[0], inputs[1], od, id, gd, nb, interpolation_mode,
                                         padding_mode, align_corners, stream);
      }
      return b200_grid_sample_f16(outputs[0], inputs[0], inputs[1], od, id, gd, nb, interpolation_mode, padding_mode,
                                  align_corners, stream);
    case 2:
      if (nb != 4) return B200_ERR_UNSUPPORTED;
      return b200_grid_sample_i8_chw4(static_cast<int8_t *>(outputs[0]), out[0].scale,
                                      static_cast<const int8_t *>(inputs[0]), in[0].scale,
                                      static_cast<const int8_t *>(inputs[1]), in[1].scale, od, id, gd, nb,
                                      interpolation_mode, padding_mode, align_corners, stream);
    default:
      return B200_ERR_UNSUPPORTED;
  }
}

// io[0] input, io[1] grid, io[2] output. use_h2 = the …TRT2 flavour (FP16 as kCHW2 packets).
int b200_grid_sampler_supports_format(int pos, const b200_tensor_desc *io, int nb_inputs, int nb_outputs, int use_h2) {
  if (!io || nb_inputs != 2 || nb_outputs != 1 || pos < 0 || pos > 2) return 0;
  const b200_tensor_desc &d = io[pos], &x = io[0];
  if (pos != 0) return d.type == x.type && d.format == x.format;
  if (x.dims.nbDims == 5) return (d.type == 0 || d.type == 1) && d.format == 0;  // 5-D: fp32 / fp16 linear (:187-189)
  if (d.type == 2) return d.format == 3;                                         // int8: kCHW4
  if (d.type == 1) return d.format == (use_h2 ? 1 : 0);                          // fp16: kCHW2 for …TRT2
  return d.type == 0 && d.format == 0;
}

// ------------------------------------------------------------------------------------------------------------------
// ModulatedDeformableConv2dTRT[2]: enqueue of the reference (…Conv2dPlugin.cpp:117-199). inputs: x, offset, mask,
// weight[, bias]. stride / padding / dilation are the plugin attributes' int[2]; element [0] goes to the launcher's *_w
// slot and [1] to *_h exactly as the reference's call does (:152-160). workspace: b200_dcn_enqueue_workspace_size.
// The launcher derives (Ho, Wo) from those attributes and the kernel size weight.d[2] x weight.d[3]; TensorRT sizes the
// output from the graph, which may read the attributes the other way round. b200_dcn_enqueue checks the output, offset,
// mask and weight descriptors against the launcher's geometry and returns B200_ERR_BAD_PARAM if they disagree, instead
// of letting the kernel read and write past those buffers (the reference does not check).
static bool dims_are(const b200_tensor_desc &t, int d0, int d1, int d2, int d3) {
  return t.dims.nbDims == 4 && t.dims.d[0] == d0 && t.dims.d[1] == d1 && t.dims.d[2] == d2 && t.dims.d[3] == d3;
}

size_t b200_dcn_enqueue_workspace_size(const b200_tensor_desc *in, const int32_t *stride, const int32_t *padding,
                                       const int32_t *dilation, int groups, int deform_groups) {
  if (!in || !stride || !padding || !dilation) return 0;
  const int32_t *x = in[0].dims.d, *w = in[3].dims.d;
  if (in[0].type == 2)
    return b200_dcn_i8_workspace_size(x[0], x[1], x[2], x[3], w[0], w[3], w[2], stride[0], stride[1], padding[0], padding[1],
                                      dilation[0], dilation[1], groups, deform_groups);
  if (in[0].type == 1 && in[0].format == 1)
    return b200_dcn_f16_chw2_workspace_size(x[0], x[1], x[2], x[3], w[0], w[3], w[2], stride[0], stride[1], padding[0],
                                            padding[1], dilation[0], dilation[1], groups, deform_groups);
  return b200_dcn_workspace_size(in[0].type == 1, x[0], x[1], x[2], x[3], w[3], w[2], stride[0], stride[1], padding[0],
                                 padding[1], dilation[0], dilation[1]);
}

int b200_dcn_enqueue(const b200_tensor_desc *in, const b200_tensor_desc *out, const void *const *inputs,
                     void *const *outputs, void *workspace, void *stream, int nb_inputs, const int32_t *stride,
                     const int32_t *padding, const int32_t *dilation, int groups, int deform_groups) {
  if (!in || !out || !inputs || !outputs || !stride || !padding || !dilation) return B200_ERR_BAD_PARAM;
  if (nb_inputs != 4 && nb_inputs != 5) return B200_ERR_BAD_PARAM;
  const int32_t *x = in[0].dims.d, *w = in[3].dims.d;
  const void *bias = nb_inputs == 5 ? inputs[4] : nullptr;
  const int s0 = stride[0], s1 = stride[1], p0 = padding[0], p1 = padding[1], d0 = dilation[0], d1 = dilation[1];
  if (in[0].dims.nbDims != 4 || s0 <= 0 || s1 <= 0 || groups <= 0) return B200_ERR_BAD_PARAM;
  const int kh = w[2], kw = w[3], taps = deform_groups * kh * kw;
  const int Ho = (x[2] + 2 * p1 - (d1 * (kh - 1) + 1)) / s1 + 1;
  const int Wo = (x[3] + 2 * p0 - (d0 * (kw - 1) + 1)) / s0 + 1;
  if (!dims_are(out[0], x[0], w[0], Ho, Wo) || !dims_are(in[1], x[0], 2 * taps, Ho, Wo) ||
      !dims_are(in[2], x[0], taps, Ho, Wo) || !dims_are(in[3], w[0], x[1] / groups, kh, kw))
    return B200_ERR_BAD_PARAM;
  switch (in[0].type) {
    case 0:
      return b200_dcn_f32(static_cast<const float *>(inputs[0]), static_cast<const float *>(inputs[3]),
                          static_cast<const float *>(bias), static_cast<const float *>(inputs[1]),
                          static_cast<const float *>(inputs[2]), static_cast<float *>(outputs[0]), workspace, x[0], x[1],
                          x[2], x[3], w[0], kw, kh, s0, s1, p0, p1, d0, d1, groups, deform_groups, x[0], nullptr, stream);
    case 1:
      if (in[0].format == 1)
        return b200_dcn_f16_chw2(inputs[0], inputs[3], bias, inputs[1], inputs[2], outputs[0], workspace, x[0], x[1], x[2],
                                 x[3], w[0], kw, kh, s0, s1, p0, p1, d0, d1, groups, deform_groups, x[0], nullptr, stream);
      return b200_dcn_f16(inputs[0], inputs[3], bias, inputs[1], inputs[2], outputs[0], workspace, x[0], x[1], x[2], x[3],
                          w[0], kw, kh, s0, s1, p0, p1, d0, d1, groups, deform_groups, x[0], nullptr, stream);
    case 2:
      return b200_dcn_i8(static_cast<const int8_t *>(inputs[0]), in[0].scale, static_cast<const int8_t *>(inputs[3]),
                         in[3].scale, bias, nb_inputs == 5 && in[4].type == 1, static_cast<const int8_t *>(inputs[1]),
                         in[1].scale, static_cast<const int8_t *>(inputs[2]), in[2].scale,
                         static_cast<int8_t *>(outputs[0]), out[0].scale, workspace, x[0], x[1], x[2], x[3], w[0], kw,
                         kh, s0, s1, p0, p1, d0, d1, groups, deform_groups, x[0], nullptr, stream);
    default:
      return B200_ERR_UNSUPPORTED;
  }
}

}  // extern "C"
