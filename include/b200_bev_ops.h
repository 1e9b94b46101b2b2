/*
 * b200_bev_ops.h — C ABI of libb200_bev_ops.so: BEVFormer's attention-sampling hot path for NVIDIA B200 (sm_100a).
 *
 * This is the drop-in boundary for the three TensorRT plugins of DerryHub/BEVFormer_tensorrt that sit on that path.
 * Every entry point replaces one launcher of the reference (the level directly under IPluginV2DynamicExt::enqueue)
 * and keeps its argument order and meaning; `file:line` below are relative to the reference repository.
 *
 * Conventions (all entry points)
 *   - All data pointers are DEVICE pointers owned by the caller (TensorRT / PyTorch); nothing is allocated, freed
 *     or retained. `stream` is a cudaStream_t passed as void*; launches are asynchronous on it, no syncs.
 *   - Return value: B200_OK (0) on success; non-zero status otherwise. Never aborts/exits the process (the reference
 *     ASSERT()s -> abort(), TensorRT/common/helper.h:43-49, and printf()s launch errors, …Kernel.cu:1124-1127).
 *     B200_ERR_UNSUPPORTED == 1 matches enqueue()'s "return 1" for an unsupported dtype (…Plugin.cpp:136-139).
 *   - No CPU fallback exists: without a CUDA device the launch fails and the status says so.
 */
#ifndef B200_BEV_OPS_H
#define B200_BEV_OPS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  B200_OK = 0,
  B200_ERR_UNSUPPORTED = 1, /* dtype / format / shape combination not implemented */
  B200_ERR_BAD_PARAM = 2,   /* null pointer, non-positive dimension, size overflow, misalignment */
  B200_ERR_LAUNCH = 3       /* CUDA reported an error at launch (cudaGetLastError) */
};

/* Library / build identification: "b200_bev_ops <version> sm_100a". */
const char *b200_bev_ops_version(void);
/* Text for a status code. */
const char *b200_status_string(int status);
/* Number of kernels this library has launched since load (bench.py's gpu_launches claim is counted here). */
unsigned long long b200_launch_count(void);

/* ------------------------------------------------------------------------------------------------------------
 * Multi-scale deformable attention (plugin MultiScaleDeformableAttnTRT / …TRT2)
 *
 *   value            [batch, spatial_size, num_heads, channels]      levels concatenated along spatial_size
 *   spatial_shapes   int32 [num_levels, 2] (h, w), device memory
 *   reference_points [batch, num_query, 1, 2*points_per_group]       normalised (x, y) per group (Z anchor)
 *   sampling_offsets [batch, num_query, num_heads, num_levels*num_point*2]   pixels of that level, (x, y) innermost
 *   attn_weight      [batch, num_query, num_heads, num_levels*num_point]     PRE-softmax logits
 *   out              [batch, num_query, num_heads, channels]
 *
 * Semantics = the reference FP32 kernel (…/multiScaleDeformableAttnKernel.cu:611-688, :133-178): softmax over
 * all num_levels*num_point logits, loc = fma(ref, size, off) - 0.5 (bit-exact index arithmetic), zero-padded bilinear
 * taps. The FP16 entry stores FP16 but evaluates indices and accumulates in FP32 (the reference's __half kernels do
 * the coordinate math in half precision, :740-756; that loss is deliberately not reproduced).
 * ---------------------------------------------------------------------------------------------------------- */

/* replaces ms_deformable_im2col_cuda<float>   — …/multiScaleDeformableAttnKernel.h:12-19, .cu:1106-1128 */
int b200_msda_f32(const float *value, const int32_t *spatial_shapes, const float *reference_points,
                  const float *sampling_offsets, const float *attn_weight, int batch, int spatial_size, int num_heads,
                  int channels, int num_levels, int num_query, int num_point, int points_per_group, float *out,
                  void *stream);

/* replaces ms_deformable_im2col_cuda<__half>  — …Kernel.h:12-19 (T=__half), .cu:1130-1149; pointers are __half* */
int b200_msda_f16(const void *value, const int32_t *spatial_shapes, const void *reference_points,
                  const void *sampling_offsets, const void *attn_weight, int batch, int spatial_size, int num_heads,
                  int channels, int num_levels, int num_query, int num_point, int points_per_group, void *out,
                  void *stream);

/* replaces ms_deformable_im2col_cuda_h2        — …Kernel.h:21-27, .cu:1151-1169. Same memory layout as _f16
 * (__half2 is a reinterpretation); needs even `channels` like the reference (…Plugin.cpp:240-245). */
int b200_msda_f16_h2(const void *value, const int32_t *spatial_shapes, const void *reference_points,
                     const void *sampling_offsets, const void *attn_weight, int batch, int spatial_size,
                     int num_heads, int channels, int num_levels, int num_query, int num_point, int points_per_group,
                     void *out, void *stream);

/* replaces ms_deformable_im2col_cuda_int8<float> / <__half2> — …Kernel.h:29-38, .cu:1172-1218.
 * value / offsets / attn_weight / out are int8 with per-tensor scales (real = q * scale, TensorRT PTQ convention,
 * …Plugin.cpp:75-77); reference_points are float (ref_is_half == 0) or __half (ref_is_half != 0).
 * Needs channels % 4 == 0 and num_point % 4 == 0 like the reference (…Plugin.cpp:151-156).
 * Arithmetic: in-register dequantisation, FP32 evaluation, one requantisation of the result with
 * round-half-away-from-zero and saturation (T2int8, .cu:51-55). */
int b200_msda_i8(const int8_t *value, float scale_value, const int32_t *spatial_shapes, const void *reference_points,
                 int ref_is_half, const int8_t *sampling_offsets, float scale_offset, const int8_t *attn_weight,
                 float scale_weight, int batch, int spatial_size, int num_heads, int channels, int num_levels,
                 int num_query, int num_point, int points_per_group, int8_t *out, float scale_out, void *stream);

/* Fused spatial-cross-attention sampling (beyond the reference's plugin set; SURVEY.md §8(f)-1): MSDA followed by the
 * bev_mask-weighted sum over cameras that SpatialCrossAttention applies to the plugin output
 * (det2trt/models/modules/spatial_cross_attention.py:270 — slots = (queries * bev_mask).sum(0)):
 *     accum[q, m*channels + c] += bev_mask[b, q] * MSDA(value, …)[b, q, m, c]        (fp32 accumulator, += semantics)
 * The per-camera output [batch, num_query, heads, channels] is never written; cameras that do not see a query add
 * nothing. bev_mask: float [batch, num_query]; accum: float [num_query, num_heads*channels], zeroed by the caller.
 * Needs channels == 32, num_point % 4 == 0, points_per_group in {1,2,4} (returns B200_ERR_UNSUPPORTED otherwise). */
int b200_msda_sca_f32(const float *value, const int32_t *spatial_shapes, const float *reference_points,
                      const float *sampling_offsets, const float *attn_weight, const float *bev_mask, int batch,
                      int spatial_size, int num_heads, int channels, int num_levels, int num_query, int num_point,
                      int points_per_group, float *accum, void *stream);
int b200_msda_sca_f16(const void *value, const int32_t *spatial_shapes, const void *reference_points,
                      const void *sampling_offsets, const void *attn_weight, const float *bev_mask, int batch,
                      int spatial_size, int num_heads, int channels, int num_levels, int num_query, int num_point,
                      int points_per_group, float *accum, void *stream);

/* Camera-shared form of the same fused op. SpatialCrossAttention repeats the BEV query for every camera before the
 * sampling_offsets / attention_weights Linear layers (spatial_cross_attention.py:254 `query.repeat(num_cams, 1, 1)`), so
 * the [batch, ...] offsets and logits the plugin receives are `batch` identical copies. Here they are passed once:
 *     sampling_offsets [num_query, heads, levels*points*2],  attn_weight [num_query, heads, levels*points]
 *     value [batch, keys, heads, channels], reference_points [batch, num_query, 1, 2*G], bev_mask [batch, num_query]
 *     slots[q, m*channels + c] = sum_b bev_mask[b, q] * MSDA(value[b], ref[b], offsets, logits)[q, m, c]   (plain store)
 * One item per (query, head): the softmax is evaluated once, the cameras that see the query are looped in registers and
 * every slot is written exactly once (no atomics, no pre-zeroed accumulator; queries no camera sees get zeros). The
 * two Linear layers upstream shrink by `batch`x and 5/6 of the offsets/logits bytes disappear. Same shape limits. */
int b200_msda_sca_shared_f32(const float *value, const int32_t *spatial_shapes, const float *reference_points,
                             const float *sampling_offsets, const float *attn_weight, const float *bev_mask,
                             int batch, int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                             int num_point, int points_per_group, float *slots, void *stream);
int b200_msda_sca_shared_f16(const void *value, const int32_t *spatial_shapes, const void *reference_points,
                             const void *sampling_offsets, const void *attn_weight, const float *bev_mask, int batch,
                             int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                             int num_point, int points_per_group, float *slots, void *stream);

/* ---- Second-generation INT8 MSDA path (csrc/msda_v2.cu): channels == 32, 16 <= num_levels*num_point <= 32 ----
 * Same operator, same semantics and argument meaning as b200_msda_i8, with one addition to the signature: the caller
 * lends a WORKSPACE (TensorRT: IPluginV2DynamicExt::getWorkspaceSize / enqueue's `workspace`; the reference's plugin
 * asks for 0 bytes, …Plugin.cpp:64-69). Its size depends on tensor DIMENSIONS only (a bound: 3 * spatial_size 64-byte
 * entries per camera and head — at base shapes 97 MB of it are touched); spatial_shapes stays the device tensor the
 * reference plugin receives, the packed-stack plan is evaluated on the device.
 * Two launches per call: (1) a pack pre-pass re-lays `value` into per-(camera, head) column-pair entries with the two
 * image rows interleaved per channel (value tiles staged through shared memory by TMA bulk copies); (2) the gather:
 * persistent CTAs bound to one (camera, head) slab of the packed stack, the coarsest levels of the slab resident in
 * shared memory (TMA bulk copies; b200_msda_set_i8_resident_bytes, default 128 KiB); a bilinear sample is one 128-byte
 * run, one 16-byte load per lane (shared memory for resident levels, L1/L2 otherwise), accumulated with dp2a against
 * 16-bit fixed-point tap weights in int32, one requantisation (T2int8). Index arithmetic is the round-1 kernel's
 * (FP32, bit-exact).
 * `trace_records` (optional, may be NULL): the gather kernel's own sampling-index records, as in b200_msda_i8_trace.
 * Returns B200_ERR_UNSUPPORTED for shapes outside the envelope (callers fall back to b200_msda_i8). */
int b200_msda_set_i8_resident_bytes(int bytes); /* returns the previous setting */
size_t b200_msda_i8_workspace_size(int batch, int spatial_size, int num_heads, int channels, int num_levels, int num_point,
                                   int points_per_group); /* 0 = shape outside the envelope */
int b200_msda_i8_ws(const int8_t *value, float scale_value, const int32_t *spatial_shapes,
                    const void *reference_points, int ref_is_half, const int8_t *sampling_offsets, float scale_offset,
                    const int8_t *attn_weight, float scale_weight, int batch, int spatial_size, int num_heads,
                    int channels, int num_levels, int num_query, int num_point, int points_per_group, int8_t *out,
                    float scale_out, void *workspace, size_t workspace_bytes, int32_t *trace_records, void *stream);

/* Multi-GPU SCA (SURVEY.md §8(e); not in the reference, which runs spatial_cross_attention.py:270's camera sum on one
 * GPU): reduce-scatter of the fp32 BEV accumulator inside a camera group, over NVLink PEER MEMORY — no NCCL call.
 * The `group_size` ranks of a camera group hold partial sums partials[r][rows*width] (their own cameras only, written
 * by b200_msda_sca_*) for the same query tile; this rank owns floats [first_elem, first_elem + num_elems) of the tile.
 * The kernel (1) publishes step `epoch` into every peer's flag row flags[r][my_index] (release, system scope) and waits
 * until flags[my_index][r] >= epoch for all peers (acquire) — stream order guarantees the local partial is final when
 * the kernel starts; (2) out[i] = sum_r partials[r][first_elem + i], peers read directly over NVLink; (3) zero-fills
 * `zero_next` (the local partial buffer of the NEXT step; partials are double-buffered by step parity).
 *   partials / flags: HOST arrays of `group_size` DEVICE pointers (peer-mapped: torch symmetric memory / cudaIpc);
 *   flags[r] is uint32[10], zero-initialised; epoch starts at 1 and increases by 1 per step on every rank;
 *   out: float (out_is_half == 0) or __half [num_elems]; element counts are multiples of 4. */
int b200_sca_peer_reduce(const void *const *partials, void *const *flags, int group_size, int my_index,
                         unsigned int epoch, long long first_elem, long long num_elems, void *out, int out_is_half,
                         float *zero_next, long long zero_elems, void *stream);
/* The same kernel with the step number kept ON THE DEVICE (flags[my_index][8] counts completed steps; the last block of
 * a launch advances it), so that every step's launch has identical parameters and the whole step — sampling launch +
 * this launch — can be captured once into a CUDA graph and replayed. Step s (1, 2, ...) reduces partials_even when
 * s is odd and partials_odd when s is even (the buffers alternate), and zero-fills the OTHER local buffer (zero_elems
 * floats; 0 = do not zero). flags[r] is uint32[10], zero-initialised. */
int b200_sca_peer_reduce_auto(const void *const *partials_even, const void *const *partials_odd, void *const *flags,
                              int group_size, int my_index, long long first_elem, long long num_elems, void *out,
                              int out_is_half, long long zero_elems, void *stream);
/* The overlapped form of the same exchange: a rank first samples the tile rows its PEERS own (launch 1), then its own rows
 * (launch 2). b200_sca_peer_pull_auto — on a side stream, ordered after launch 1 — publishes the step, waits for the
 * peers and pulls THEIR launch-1 results for this rank's slice into `staging` (floats [num_elems], local memory) while
 * launch 2 runs; b200_sca_peer_add_auto — on the main stream after launch 2 and after the pull — writes
 * out = own partial + staging and zero-fills the next step's buffer. Buffers, flags and the device-side step counter are
 * those of b200_sca_peer_reduce_auto. */
int b200_sca_peer_pull_auto(const void *const *partials_even, const void *const *partials_odd, void *const *flags,
                            int group_size, int my_index, long long first_elem, long long num_elems, float *staging,
                            void *stream);
int b200_sca_peer_add_auto(const void *partial_even, const void *partial_odd, void *flags_local, int my_index,
                           long long first_elem, long long num_elems, const float *staging, void *out, int out_is_half,
                           long long zero_elems, void *stream);



/* Trace entries: b200_msda_f32 / _f16 / _i8 with the production kernel's trace switch on (the same kernel template,
 * compiled with one extra store): besides `out` they write, for every (batch, query, head, level*point), the
 * sampling-index record {in_range, h_low, w_low, tap_mask} (4 x int32; all-zero when the point is out of range) that
 * THE GATHER KERNEL ITSELF computed on its way to the taps. `records` must hold batch*num_query*num_heads*num_levels*
 * num_point*4 int32; it is zero-filled on `stream` first. These are what the bit-exact index parity tests compare with
 * the oracle (reference arithmetic: …Kernel.cu:657-674, :138-172). */
int b200_msda_f32_trace(const float *value, const int32_t *spatial_shapes, const float *reference_points,
                        const float *sampling_offsets, const float *attn_weight, int batch, int spatial_size,
                        int num_heads, int channels, int num_levels, int num_query, int num_point,
                        int points_per_group, float *out, int32_t *records, void *stream);
int b200_msda_f16_trace(const void *value, const int32_t *spatial_shapes, const void *reference_points,
                        const void *sampling_offsets, const void *attn_weight, int batch, int spatial_size,
                        int num_heads, int channels, int num_levels, int num_query, int num_point,
                        int points_per_group, void *out, int32_t *records, void *stream);
int b200_msda_i8_trace(const int8_t *value, float scale_value, const int32_t *spatial_shapes,
                       const void *reference_points, int ref_is_half, const int8_t *sampling_offsets,
                       float scale_offset, const int8_t *attn_weight, float scale_weight, int batch, int spatial_size,
                       int num_heads, int channels, int num_levels, int num_query, int num_point, int points_per_group,
                       int8_t *out, float scale_out, int32_t *records, void *stream);

/* Stand-alone diagnostic: the same records from a small index-only kernel (no value / logits needed; shares the
 * point_record() device function with the generic fallback kernel). dtype: 0 = float inputs, 1 = __half inputs. */
int b200_msda_debug_indices(int dtype, const int32_t *spatial_shapes, const void *reference_points,
                            const void *sampling_offsets, int batch, int num_heads, int num_levels, int num_query,
                            int num_point, int points_per_group, int32_t *records, void *stream);

/* Selects the FP16 accumulate flavour for b200_msda_f16*. 0 (default) = exact: taps widened to FP32, FP32 weights,
 * packed FP32 FMA (FFMA2) — meets the 1e-3 max-abs parity bar everywhere. 1 = mixed: FP16 tap x FP16 weight -> FP32
 * accumulator (fma.rn.f32.f16, FHFMA); ~15 % fewer issue slots but the FP16 rounding of the weights adds up to ~3e-4
 * on O(1) outputs, so it is opt-in. Returns the previous setting. */
int b200_msda_set_f16_mode(int mode);

/* Selects the kernel behind b200_msda_f16 / _f16_h2 / _f16_trace. 0 (default) = the gather kernel (csrc/msda.cu) for
 * every shape; 1 = the resident-tail kernel (csrc/msda_res.cu: CTAs bound to one (batch, head), the coarsest pyramid
 * levels staged in shared memory by TMA, taps of those levels served from shared memory) whenever channels == 32,
 * num_levels*num_point <= 32, num_point % 4 == 0 — measured slower on B200 (DESIGN.md §4.1c), hence opt-in. Same
 * results either way (same index arithmetic, FP32 accumulation).
 * b200_msda_set_resident_bytes: shared memory the resident kernel may use for the tail (default 128 KiB). Both return
 * the previous setting. */
int b200_msda_set_f16_path(int path);
int b200_msda_set_resident_bytes(int bytes);

/* Launch shape of the FP32 / FP16 plugin op (b200_msda_f32 / _f16 / _f16_h2 and their _trace twins): units = 1 is one
 * block of items per CTA; 2 or 4 is the batched launch — every warp first scans the visibility of `units` of its item
 * groups with all their offset / reference-point loads in flight together, answers the invisible ones with zeros and
 * runs the sampling body on the rest (csrc/msda.cu, UPW). strided = 0: the units of a CTA are neighbouring blocks of
 * items; 1: they lie a whole grid apart (evens out CTA run times when visibility comes in long runs). Results are
 * bit-identical for every setting. Any other `units` (e.g. 0) only queries. The initial value is the environment
 * variable B200_MSDA_BATCH ("1", "2", "4", "2s", "4s") if set, else the library default. Returns the previous setting
 * as units | strided << 8. */
int b200_msda_set_batch_units(int units, int strided);

/* Gather depth of the same plugin op (one-unit grid, untraced launches): 0 (default) = 3 CTAs of 8 warps per SM, the 4 tap
 * loads of one sampling point in flight per warp; 1 = 2 CTAs per SM (128-register budget): the 16 tap loads of a 4-point
 * chunk in flight per warp; 2 = the same with that order written out in the source; 3 = 128-thread CTAs, 5 per SM (20 warps,
 * 96 registers), two points = 8 loads issued together — fewer warps, more loads per warp, for inputs on which the kernel is
 * latency-bound. Same bits for every variant (the FMA order does not change). Any other value (e.g. -1) only queries.
 * Initial value: environment variable B200_MSDA_VARIANT ("0" .. "3"), else 0. Returns the
 * previous setting. A batched launch (units > 1 above) combines with variant 1 (batched scan at 2 CTAs per SM) and takes
 * precedence over variants 2 and 3. The fused forms
 * (b200_msda_sca_* / b200_msda_sca_shared_*) have one alternative: any non-zero variant runs them at 2 CTAs per SM. */
int b200_msda_set_gather_variant(int variant);

/* ------------------------------------------------------------------------------------------------------------
 * Plugin-shaped entry: the argument list of IPluginV2DynamicExt::enqueue
 * (…/multiScaleDeformableAttnPlugin.cpp:71-140) with a POD mirror of nvinfer1::PluginTensorDesc, so a TensorRT
 * plugin shell (csrc/trt_plugin/, compiled only where NvInfer.h exists) or any other host can forward verbatim.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t nbDims;
  int32_t d[8];
} b200_dims; /* layout of nvinfer1::Dims */

typedef struct {
  b200_dims dims;
  int32_t type;   /* nvinfer1::DataType: 0 kFLOAT, 1 kHALF, 2 kINT8, 3 kINT32 */
  int32_t format; /* nvinfer1::TensorFormat: 0 kLINEAR, 1 kCHW2 (fp16x2), 2 kHWC8, 3 kCHW4 (int8x4) */
  float scale;
} b200_tensor_desc; /* layout of nvinfer1::PluginTensorDesc */

/* inputs: value, spatial_shapes, reference_points, sampling_offsets, attn_weight; outputs: out.
 * use_h2 selects the …TRT2 flavour. Returns 0 ok / 1 unsupported dtype, as the reference does. */
int b200_msda_enqueue(const b200_tensor_desc *input_desc, const b200_tensor_desc *output_desc,
                      const void *const *inputs, void *const *outputs, void *workspace, void *stream, int use_h2);

/* getWorkspaceSize mirror: bytes b200_msda_enqueue wants in `workspace` for the second-generation INT8 kernels
 * (0 for FP32 / FP16 and for shapes outside their envelope). enqueue(workspace == NULL) runs the round-1 kernels. */
size_t b200_msda_enqueue_workspace_size(const b200_tensor_desc *input_desc);

/* Mirror of supportsFormatCombination (…Plugin.cpp:148-189): 1 if descriptor `pos` of in_out[0..5] is acceptable. */
int b200_msda_supports_format(int pos, const b200_tensor_desc *in_out, int nb_inputs, int nb_outputs);


/* ------------------------------------------------------------------------------------------------------------
 * Grid sampler (plugins GridSampler2DTRT / GridSampler2DTRT2 / GridSampler3DTRT / GridSampler3DTRT2)
 *
 *   input  [N, C, Hi, Wi]       (5-D: [N, C, Di, Hi, Wi])
 *   grid   [N, 2, Ho, Wo]       channel-first: x plane then y plane (5-D: [N, 3, Do, Ho, Wo]); range [-10, 10]
 *   output [N, C, Ho, Wo]
 *   *_dims: HOST int arrays of length nb_dims (4 or 5), as the reference launchers take them.
 *   interp: 0 bilinear, 1 nearest, 2 bicubic (2-D only);  padding: 0 zeros, 1 border, 2 reflection
 *   (enum order of gridSamplerKernel.h:11-12).
 * Semantics = the reference FP32 kernel (TensorRT/plugin/grid_sampler/gridSamplerKernel.cu:666-795, helpers :82-92,
 * :157-162, :226-247, :342-393), evaluated in FP32 for every storage type.
 * ---------------------------------------------------------------------------------------------------------- */

/* replaces grid_sample<float>   — gridSamplerKernel.h:14-18, .cu:1933-1964 */
/* Opt-in tile kernel for 2-D bilinear sampling: 0 (default) = the generic kernel; 1 / 2 = the source window of an 8 x 32
 * output tile is staged in shared memory by TMA (1: one bulk copy per packet row, 2: one 2-D tensor copy per channel
 * packet), with a per-tile fallback to scattered loads when the window does not fit and a per-call fallback when the
 * layout does not meet TMA's 16-byte rules (input pointer, row pitch). Same results bit for bit; measured equal (mode 2)
 * or slower (mode 1) than the generic kernel at the prev-BEV warp. Returns the previous setting. */
int b200_grid_sample_set_tile_path(int mode);
int b200_grid_sample_f32(float *output, const float *input, const float *grid, const int *output_dims,
                         const int *input_dims, const int *grid_dims, int nb_dims, int interp, int padding,
                         int align_corners, void *stream);

/* replaces grid_sample<__half>  — same launcher, T=__half, kLINEAR tensors (gridSamplerPlugin.cpp:171-186) */
int b200_grid_sample_f16(void *output, const void *input, const void *grid, const int *output_dims,
                         const int *input_dims, const int *grid_dims, int nb_dims, int interp, int padding,
                         int align_corners, void *stream);

/* replaces grid_sample<__half2> — .cu:1969-2008: tensors in TensorRT kCHW2 format
 * (input/output [N, ceil(C/2), H, W, 2]; the 2-channel grid is one (x, y) __half2 per output pixel). 2-D only. */
int b200_grid_sample_f16_chw2(void *output, const void *input, const void *grid, const int *output_dims,
                              const int *input_dims, const int *grid_dims, int nb_dims, int interp, int padding,
                              int align_corners, void *stream);

/* replaces grid_sample_int8     — gridSamplerKernel.h:20-26, .cu:2010-2043: tensors in kCHW4 format
 * (input/output [N, ceil(C/4), H, W, 4] int8; grid (x, y, pad, pad) int8 per output pixel), per-tensor scales,
 * real = q * scale. In-register dequantisation, FP32 math, one requantisation (T2int8). 2-D only. */
int b200_grid_sample_i8_chw4(int8_t *output, float scale_o, const int8_t *input, float scale_i, const int8_t *grid,
                             float scale_g, const int *output_dims, const int *input_dims, const int *grid_dims,
                             int nb_dims, int interp, int padding, int align_corners, void *stream);

/* ------------------------------------------------------------------------------------------------------------
 * Rotate (plugins RotateTRT / RotateTRT2; det2trt/models/functions/rotate.py:7-124)
 *
 *   input / output [C, H, W]   (input_dims = HOST int[3] {C, H, W}, as the plugin passes inputDesc[0].dims.d)
 *   angle  [1] degrees, counter-clockwise; center [2] = (x, y) in pixels: DEVICE pointers (plugin inputs 1, 2)
 *   interp: 0 bilinear, 1 nearest (RotateInterpolation, TensorRT/plugin/rotate/rotateKernel.h:12); zero padding.
 *
 * Semantics = the reference FP32 kernel (rotateKernel.cu:128-210) — its index arithmetic is reproduced operation for
 * operation (b200_rotate_debug_indices exposes it to the tests). FP16 / INT8 images are converted in registers;
 * matrix, coordinates and blending stay FP32 (the reference computes them in half precision, :213-260, :416-456).
 * ---------------------------------------------------------------------------------------------------------- */
/* replaces rotate<float>        — rotateKernel.h:14-16, .cu:708-719 */
int b200_rotate_f32(float *output, const float *input, const float *angle, const float *center,
                    const int *input_dims, int interp, void *stream);

/* replaces rotate<__half>       — same launcher, T=__half: image, angle and center are __half, kLINEAR */
int b200_rotate_f16(void *output, const void *input, const void *angle, const void *center, const int *input_dims,
                    int interp, void *stream);

/* replaces rotate_h2            — rotateKernel.h:18-20, .cu:721-732: image in kCHW2 ([ceil(C/2), H, W, 2] __half) */
int b200_rotate_f16_h2(void *output, const void *input, const void *angle, const void *center, const int *input_dims,
                       int interp, void *stream);

/* replaces rotate_int8<float|__half> — rotateKernel.h:22-26, .cu:734-748: image in kCHW4 ([ceil(C/4), H, W, 4] int8),
 * per-tensor scales (real = q * scale); angle / center are float (angle_is_half = 0) or __half (1), as
 * rotatePlugin.cpp:101-111 dispatches on inputDesc[1].type. */
int b200_rotate_i8(int8_t *output, float scale_o, const int8_t *input, float scale_i, const void *angle,
                   const void *center, int angle_is_half, const int *input_dims, int interp, void *stream);

/* B200 extension: channels-last image [H, W, C] (input_dims still {C, H, W}). prev_bev is stored [H*W, C] at the call
 * site (det2trt/models/modules/transformer.py:296-304); this entry rotates it in place of permute -> RotateTRT ->
 * permute. dtype 0: float image/angle/center, 1: __half. Needs C % 4 == 0 (fp32) / C % 8 == 0 (fp16) and 16-byte
 * aligned buffers, else B200_ERR_UNSUPPORTED. */
int b200_rotate_hwc(void *output, const void *input, const void *angle, const void *center, int dtype,
                    const int *input_dims, int interp, void *stream);

/* Test hook: source_xy[H*W*2] = (ix, iy), the fractional source pixel of every output pixel, from FP32 angle/center. */
int b200_rotate_debug_indices(const float *angle, const float *center, const int *input_dims, float *source_xy,
                              void *stream);


/* ------------------------------------------------------------------------------------------------------------
 * BEV pillar points -> per-camera reference points and visibility weights (the encoder prologue that feeds spatial
 * cross-attention; eager PyTorch in the reference, ONNX elementwise nodes in its engines — no plugin):
 *   BEVFormerEncoderTRTP.get_reference_points_3d  det2trt/models/modules/encoder.py:168-194
 *   BEVFormerEncoderTRTP.point_sampling_trt        det2trt/models/modules/encoder.py:196-259
 *
 *   reference_points      [1, D, bev_h*bev_w, 3] in [0,1] (what get_reference_points_3d returns), or NULL to generate
 *                         that pillar grid analytically (Z = pc_range[5] - pc_range[2], encoder.py:281-289)
 *   pc_range              HOST double[6] = (x0, y0, z0, x1, y1, z1)
 *   lidar2img             DEVICE float [num_cams, 4, 4]
 *   reference_points_cam  [num_cams, 1, Q, D, 2]  (u, v) normalised by (image_w, image_h) — the MSDA reference_points
 *   bev_mask              [num_cams, Q, 1]        seen / max(sum over cameras of seen, 1e-4)
 *   dtype                 0: float tensors, 1: __half tensors (reference_points in, both outputs; math stays FP32 and
 *                         coordinates of points behind a camera saturate to +-65504 instead of overflowing to inf)
 * num_cams <= 16, num_points_in_pillar <= 8, reference_points_cam 16-byte aligned, else B200_ERR_UNSUPPORTED.
 * ---------------------------------------------------------------------------------------------------------- */
int b200_bev_point_sampling(const void *reference_points, const double *pc_range, const float *lidar2img,
                            int num_cams, int image_h, int image_w, int bev_h, int bev_w, int num_points_in_pillar,
                            int dtype, void *reference_points_cam, void *bev_mask, void *stream);

/* ------------------------------------------------------------------------------------------------------------
 * Modulated deformable convolution, DCNv2 (plugins ModulatedDeformableConv2dTRT / …TRT2)
 *
 *   input  [batch, channels, height, width]
 *   weight [channels_out, channels/group, kernel_h, kernel_w]     bias [channels_out] or NULL
 *   offset [batch, deformable_group*2*kernel_h*kernel_w, Ho, Wo]  per tap: dh then dw (mmcv order,
 *                                                                 modulatedDeformableConv2dKernel.cu:297-301)
 *   mask   [batch, deformable_group*kernel_h*kernel_w, Ho, Wo]    already sigmoid-ed
 *   output [batch, channels_out, Ho, Wo],  Ho = (height + 2*pad_h - (dilation_h*(kernel_h-1)+1))/stride_h + 1
 *   workspace: device scratch of b200_dcn_workspace_size(...) bytes (the plugin's getWorkspaceSize,
 *              …Conv2dPlugin.cpp:73-115, should return this instead of its single-image column size).
 *   cublas_handle: the reference's slot (…Conv2dPlugin.cpp:286-290), kept for signature compatibility and IGNORED — no
 *   library GEMM runs on this path (dcn_fused.cu: tcgen05 implicit GEMM; dcn_generic.cu: fused FP32-pipe implicit GEMM)
 *              to use the library's own handle.
 * Argument order = the reference launcher ModulatedDeformConvForwardCUDAKernel<T> (…Conv2dKernel.h:11-19).
 * FP16 accumulates the GEMM in FP32 (the reference accumulates in FP16, common/cuda_helper.cu:101-110).
 * ---------------------------------------------------------------------------------------------------------- */
size_t b200_dcn_workspace_size(int dtype /* 0 f32, 1 f16 */, int batch, int channels, int height, int width,
                               int kernel_w, int kernel_h, int stride_w, int stride_h, int pad_w, int pad_h,
                               int dilation_w, int dilation_h);

/* FP16 runs as one fused implicit GEMM on tcgen05 tensor cores (csrc/dcn_fused.cu) when groups == deformable_groups == 1,
 * channels % 64 == 0 and channels_out in {128, 256, 512}; otherwise (and for FP32) as the generic fused implicit GEMM on
 * the FP32 pipe (csrc/dcn_generic.cu: any groups / deformable groups / kernel size). No library GEMM on either path.
 * b200_dcn_set_fused(0) forces the second path (A/B measurements), a negative argument only queries; returns the
 * previous setting. */
int b200_dcn_set_fused(int enabled);

/* replaces ModulatedDeformConvForwardCUDAKernel<float> — …Conv2dKernel.cu:695-760 */
int b200_dcn_f32(const float *input, const float *weight, const float *bias, const float *offset, const float *mask,
                 float *output, void *workspace, int batch, int channels, int height, int width, int channels_out,
                 int kernel_w, int kernel_h, int stride_w, int stride_h, int pad_w, int pad_h, int dilation_w,
                 int dilation_h, int group, int deformable_group, int im2col_step, void *cublas_handle, void *stream);

/* Deployment helpers for the fused FP16 path (beyond the reference's launcher set): weights are constants at inference
 * time and feature maps may already be channels-last, so both pre-passes of b200_dcn_f16 can be hoisted out of the call.
 *   b200_dcn_pack_weights_f16: weight [Co, C, kh, kw] -> packed [Co][C/64][kh*kw][64] (same byte size), once per layer.
 *   b200_dcn_f16_ex: flags bit 0 = `input` is NHWC [batch, H, W, channels]; bit 1 = `weight` is already packed.
 *   Fused path only (see b200_dcn_set_fused): returns B200_ERR_UNSUPPORTED for other shapes. */
int b200_dcn_pack_weights_f16(const void *weight, void *packed, int channels_out, int channels, int kernel_h, int kernel_w,
                              void *stream);
int b200_dcn_f16_ex(const void *input, const void *weight, const void *bias, const void *offset, const void *mask,
                    void *output, void *workspace, int batch, int channels, int height, int width, int channels_out,
                    int kernel_w, int kernel_h, int stride_w, int stride_h, int pad_w, int pad_h, int dilation_w,
                    int dilation_h, int group, int deformable_group, int flags, void *stream);

/* replaces ModulatedDeformConvForwardCUDAKernel_int8<float> / <__half> — …Conv2dKernel.h:21-29, .cu:897-978.
 * input int8 kCHW4 [batch, channels/4, H, W, 4], weight int8 kCHW4 [channels_out, channels/4, kh, kw, 4], offset / mask
 * int8 kLINEAR, output int8 kLINEAR, per-tensor scales (real = q*scale); bias float (bias_is_half == 0), __half, or NULL.
 * Arithmetic: in-register dequantisation (int8 values are exact in FP16), FP16 tensor-core products with FP32
 * accumulation, one requantisation T2int8((acc*scale_i*scale_w + bias)/scale_o) — the reference requantises the
 * sampled columns to int8 first (:536-545). Shapes of the fused path (groups == deformable_groups == 1,
 * channels % 64 == 0, channels_out in {128, 256, 512}) run on tensor cores in one kernel; any other shape with
 * channels % 4 == 0 and (channels / group) % 4 == 0 dequantises into the workspace and runs the generic hand-written FP16
 * kernel (csrc/dcn_generic.cu, FP32 accumulation), one requantisation at the end. workspace: b200_dcn_i8_workspace_size(...) bytes,
 * 256-byte aligned. */
size_t b200_dcn_i8_workspace_size(int batch, int channels, int height, int width, int channels_out, int kernel_w,
                                  int kernel_h, int stride_w, int stride_h, int pad_w, int pad_h, int dilation_w,
                                  int dilation_h, int group, int deformable_group);
int b200_dcn_i8(const int8_t *input, float scale_i, const int8_t *weight, float scale_w, const void *bias, int bias_is_half,
                const int8_t *offset, float scale_off, const int8_t *mask, float scale_mask, int8_t *output, float scale_o,
                void *workspace, int batch, int channels, int height, int width, int channels_out, int kernel_w,
                int kernel_h, int stride_w, int stride_h, int pad_w, int pad_h, int dilation_w, int dilation_h, int group,
                int deformable_group, int im2col_step, void *cublas_handle, void *stream);

/* replaces ModulatedDeformConvForwardCUDAKernel<__half> / <__half2> — …Conv2dKernel.cu:762-895 (kLINEAR tensors) */
int b200_dcn_f16(const void *input, const void *weight, const void *bias, const void *offset, const void *mask,
                 void *output, void *workspace, int batch, int channels, int height, int width, int channels_out,
                 int kernel_w, int kernel_h, int stride_w, int stride_h, int pad_w, int pad_h, int dilation_w,
                 int dilation_h, int group, int deformable_group, int im2col_step, void *cublas_handle, void *stream);

/* FP16 in TensorRT's kCHW2 packets — what the …TRT2 plugin negotiates (…Conv2dPlugin.cpp:222-250: input, offset and
 * weight as __half2 packets [N, ceil(C/2), H, W, 2]; mask, bias and output linear). Replaces
 * ModulatedDeformConvForwardCUDAKernel<__half2> (…Conv2dKernel.cu:828-895). The packets are unpacked into the workspace
 * (sized by b200_dcn_f16_chw2_workspace_size) and the FP16 path above runs. */
size_t b200_dcn_f16_chw2_workspace_size(int batch, int channels, int height, int width, int channels_out, int kernel_w,
                                        int kernel_h, int stride_w, int stride_h, int pad_w, int pad_h, int dilation_w,
                                        int dilation_h, int group, int deformable_group);
int b200_dcn_f16_chw2(const void *input, const void *weight, const void *bias, const void *offset, const void *mask,
                      void *output, void *workspace, int batch, int channels, int height, int width, int channels_out,
                      int kernel_w, int kernel_h, int stride_w, int stride_h, int pad_w, int pad_h, int dilation_w,
                      int dilation_h, int group, int deformable_group, int im2col_step, void *cublas_handle, void *stream);

/* ------------------------------------------------------------------------------------------------------------
 * Plugin-shaped entries for the other two plugins (the argument list of IPluginV2DynamicExt::enqueue plus the plugin's
 * attributes), so that a TensorRT shell — or a test — forwards verbatim, as b200_msda_enqueue does for MSDA.
 * ---------------------------------------------------------------------------------------------------------- */
/* GridSampler{2D,3D}TRT[2] (gridSamplerPlugin.cpp:110-155): inputs = input, grid; dispatch on the input descriptor's
 * type / format (fp32, fp16 linear, fp16 kCHW2, int8 kCHW4 with the descriptors' scales). Needs no workspace. */
int b200_grid_sampler_enqueue(const b200_tensor_desc *input_desc, const b200_tensor_desc *output_desc,
                              const void *const *inputs, void *const *outputs, void *workspace, void *stream,
                              int interpolation_mode, int padding_mode, int align_corners);
/* supportsFormatCombination mirror (gridSamplerPlugin.cpp:168-194): in_out = {input, grid, output}. */
int b200_grid_sampler_supports_format(int pos, const b200_tensor_desc *in_out, int nb_inputs, int nb_outputs, int use_h2);

/* ModulatedDeformableConv2dTRT[2] (…Conv2dPlugin.cpp:117-199): inputs = x, offset, mask, weight[, bias] (nb_inputs 4 or
 * 5). stride / padding / dilation = the plugin attributes' int[2]; element [0] is handed to the launcher's *_w slot and
 * [1] to *_h exactly as the reference's enqueue does (:152-160). Dispatch: fp32, fp16 linear, fp16 kCHW2, int8 kCHW4.
 * Before launching anything, b200_dcn_enqueue computes (Ho, Wo) as the launcher will (stride / padding / dilation [0]
 * for w and [1] for h, kernel weight.d[2] x weight.d[3]) and returns B200_ERR_BAD_PARAM unless output == (N, Co, Ho, Wo),
 * offset == (N, deform_groups*2*kh*kw, Ho, Wo), mask == (N, deform_groups*kh*kw, Ho, Wo) and
 * weight.d[1] == C / groups: a graph that reads the attributes as (h, w) is refused instead of being read and
 * written past its buffers. b200_grid_sampler_enqueue likewise requires output == (N, C) of the input followed by the
 * grid's spatial dims. */
size_t b200_dcn_enqueue_workspace_size(const b200_tensor_desc *input_desc, const int32_t *stride, const int32_t *padding,
                                       const int32_t *dilation, int groups, int deform_groups);
int b200_dcn_enqueue(const b200_tensor_desc *input_desc, const b200_tensor_desc *output_desc, const void *const *inputs,
                     void *const *outputs, void *workspace, void *stream, int nb_inputs, const int32_t *stride,
                     const int32_t *padding, const int32_t *dilation, int groups, int deform_groups);

#ifdef __cplusplus
} /* extern "C" */
#endif
#endif /* B200_BEV_OPS_H */
