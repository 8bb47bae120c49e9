/*
 * scn_b200.h -- C ABI of the B200-native SparseConvNet backbone path.
 *
 * This is the drop-in boundary: every entry point replaces one operation of the reference's
 * native extension `sparseconvnet.SCN` (pybind11; paths below are relative to
 * /root/reference/SparseConvNet/sparseconvnet/SCN/).  Dimension is fixed to 3 (Metadata_3),
 * dtype to float32 features / int32 rule indices, as on the reference's hot path
 * (cuda.cu:52-72 instantiates <float> only; Metadata/32bits.h:11).
 *
 * Conventions
 *  - all feature / weight / gradient pointers are DEVICE pointers (row-major float32);
 *  - `stream` is a cudaStream_t passed as void*; everything is enqueued on it, nothing runs on the
 *    legacy default stream and no blocking copy of rule tables ever happens (compare
 *    CUDA/RuleBookIterator.h:15-32);
 *  - spatial sizes / filter sizes / strides are `const long[3]` (the reference passes LongTensors);
 *  - every function returns 0 on success, non-zero on failure with a message in scn_last_error()
 *    (the reference raises C++ exceptions through pybind -> RuntimeError; the Python wrapper does
 *    the same from the status code);
 *  - two-phase sizing: the caller learns the number of output rows from scn_get_nactive /
 *    scn_convolution_prepare, allocates, and passes the pointer (the reference resizes a caller
 *    supplied empty tensor, e.g. CPU/Convolution.cpp:55);
 *  - a scn_metadata is used from one thread / one stream at a time, like the reference's
 *    Metadata (lazy caches are unguarded, Metadata.cpp:434-441).
 */
#ifndef SCN_B200_H
#define SCN_B200_H
#ifdef __cplusplus
extern "C" {
#endif

typedef struct scn_metadata scn_metadata;

const char *scn_last_error(void);
int scn_version(void);

/* n_rulebook_bits()  -- pybind.cpp:234 */
int scn_n_rulebook_bits(void);

/* Metadata_3() / destructor -- pybind.cpp:12-32, Metadata/Metadata.h:44-163 */
int scn_metadata_create(scn_metadata **out, void *stream);
void scn_metadata_destroy(scn_metadata *m);

/* Metadata::inputLayer  (pybind InputLayer_updateOutput, pybind.cpp:154-158; Metadata.cpp:405-417;
 * Metadata/IOLayersRules.h:18-125).  coords: int64 [nrows][ncols], ncols 3 or 4 (x,y,z[,batch]),
 * host or device memory.  Builds the level-0 grid and the input rule table; returns the number
 * of active voxels and the largest number of input rows merged into one voxel. */
int scn_input_layer_build(scn_metadata *m, const long spatial_size[3], const long *coords, int coords_on_device,
                          long nrows, int ncols, int batch_size, int mode, long *n_active, int *max_active);
/* 1 (and the counts) when scn_input_layer_build has run on this Metadata, else 0 */
int scn_input_layer_built(scn_metadata *m, long *n_active, int *max_active);
/* InputLayer_ForwardPass / InputLayer_fp  (CPU/IOLayers.cpp:11-29, CUDA/IOLayers.cu:31-41) */
int scn_input_layer_forward(scn_metadata *m, const float *in_features, float *out_features, int n_planes);
/* scn_input_layer_forward that also writes the rows as 16-bit values (bfloat16; float16 in math mode 5) zero-padded to `padded`
 * channels (first convolution of a bf16 / fp16 program) */
int scn_input_layer_forward_padded_bf16(scn_metadata *m, const float *in_features, float *out_features, void *out_bf16, int n_planes, int padded);
/* InputLayer_updateGradInput (pybind.cpp:159-162; CPU/IOLayers.cpp:30-47) */
int scn_input_layer_backward(scn_metadata *m, float *d_in_features, const float *d_out_features, int n_planes);

/* OutputLayer_updateOutput / _updateGradInput (pybind.cpp:163-170; CPU/IOLayers.cpp:97-140): out [n input rows][n_planes] =
 * the feature row of each input row's voxel (no averaging); d_in [nActive][n_planes] = sum over the rows of a voxel. */
int scn_output_layer_forward(scn_metadata *m, const float *in_features, float *out_features, int n_planes);
int scn_output_layer_backward(scn_metadata *m, float *d_in_features, const float *d_out_features, int n_planes);

/* Metadata::getNActive (Metadata.cpp:67-69) */
int scn_get_nactive(scn_metadata *m, const long spatial_size[3], long *n_active);
/* Metadata::getSpatialLocations (pybind.cpp:17; Metadata.cpp:147-168): int64 [nActive][4] */
int scn_get_spatial_locations(scn_metadata *m, const long spatial_size[3], long *out, int out_on_device);

/* Metadata::getSubmanifoldRuleBook (Metadata.cpp:429-443): builds (once) and reports the total
 * number of rules over all filter offsets. */
int scn_submanifold_prepare(scn_metadata *m, const long spatial_size[3], const long filter_size[3], long *n_rules);
/* Hint (no reference counterpart; the reference builds every rulebook lazily and synchronously on the
 * calling thread, Metadata.cpp:429-510): build these rulebooks ahead on a worker thread + the build
 * stream while the caller keeps submitting feature kernels.  ops = n_ops x 13 longs: kind (1 submanifold,
 * 2 convolution, 3 deconvolution), a[3], b[3], filter[3], stride[3] with (a, b) = (size, -) / (in, out) /
 * (in, out) exactly as the corresponding *_forward call receives them.  Kinds 4 (submanifold, a = size) and
 * 5 (convolution, a = in, b = out) build the (in, out) rule lists a backward entry reads, after every
 * rulebook of kinds 1-3, in the order given.  Results are unaffected. */
int scn_metadata_prefetch(scn_metadata *m, int n_ops, const long *ops);
/* Metadata::getRuleBook (Metadata.cpp:484-510): builds (once) the strided rulebook AND the output
 * grid; reports the output grid's active count and the number of rules. */
int scn_convolution_prepare(scn_metadata *m, const long in_size[3], const long out_size[3], const long filter_size[3],
                            const long filter_stride[3], long *n_active_out, long *n_rules);

/* Rulebook access for parity checks (the reference keeps these as public members,
 * Metadata/Metadata.h:56-67).  kind 0 = input-layer table, 1 = submanifold, 2 = strided, 3 = SparseToDense (a = spatial size;
 * one list per batch item of (row, spatial offset) pairs in hash-iteration order, Metadata.cpp:469-483).
 * scn_rulebook_info fills n_lists and list_len[n_lists] (ints per list: 2*pairs; for kind 0:
 * list 0 = {mode,maxActive,nIn,nOut}, list 1 = nOut*(1+maxActive)).  scn_rulebook_copy copies
 * one list to HOST memory as the reference lays it out ((in,out) int32 pairs). */
int scn_rulebook_info(scn_metadata *m, int kind, const long a[3], const long b[3], const long c[3], int *n_lists, long *list_len);
int scn_rulebook_copy(scn_metadata *m, int kind, const long a[3], const long b[3], const long c[3], int list, int *dst);
/* Reference hash-iteration order of a grid (ids in ascending dense_hash_map bucket order,
 * batch items concatenated) -- host int32 [nActive]. */
int scn_iteration_order(scn_metadata *m, const long spatial_size[3], int *dst);

/* SubmanifoldConvolution_updateOutput (pybind.cpp:134-138; CPU/Convolution.cpp:117-150;
 * CUDA/Convolution.cpp:95-125).  weight [K][Cin][Cout] (= (K,1,Cin,Cout) with groups 1),
 * bias NULL or [Cout].  *macs = sum_k nRules_k*Cin*Cout, the value the reference returns.
 * in_bf16 (all three forward calls): NULL, or a device copy of `in` rounded to 16 bits (same
 * [rows][n_in] layout) that a preceding scn_batchnorm_forward / scn_add_features produced; it is
 * only read in math modes 2 and 5, where a NULL makes the call convert `in` itself.  Every "bf16"
 * argument of this header (in_bf16, out_bf16, lat_in_bf16) holds a 16-bit copy in the format of the
 * current math mode: float16 in mode 5, bfloat16 in every other mode.
 * weight_tag: 0, or a value that identifies the CONTENTS of `weight` (same pointer + same tag =
 * same values as in an earlier call): the tensor-core paths then reuse the operand image they
 * derived from it (rounded, swizzled copy) instead of rebuilding it on every call.
 * add_in: NULL, or [output rows][n_out] float32 added to the result (out = conv(in) + add_in): the
 * residual / lateral AddTable that follows the convolution in the network, fused into its epilogue.
 * out_bf16: NULL, or [output rows][n_out] 16-bit values (the mode's format) that receive the (summed) result rounded to nearest. */
int scn_submanifold_convolution_forward(scn_metadata *m, const long spatial_size[3], const long filter_size[3],
                                        const float *in, float *out, const float *weight, const float *bias,
                                        int n_in, int n_out, double *macs, const void *in_bf16, long long weight_tag,
                                        const float *add_in, void *out_bf16);
/* Convolution_updateOutput (pybind.cpp:54-59; CPU/Convolution.cpp:45-79) */
int scn_convolution_forward(scn_metadata *m, const long in_size[3], const long out_size[3], const long filter_size[3],
                            const long filter_stride[3], const float *in, float *out, const float *weight,
                            const float *bias, int n_in, int n_out, double *macs, const void *in_bf16, long long weight_tag,
                            const float *add_in, void *out_bf16);
/* Deconvolution_updateOutput (pybind.cpp:78-83; CPU/Deconvolution.cpp:7-41): reuses the rulebook of the
 * Convolution out_size -> in_size with the pair columns swapped. */
int scn_deconvolution_forward(scn_metadata *m, const long in_size[3], const long out_size[3], const long filter_size[3],
                              const long filter_stride[3], const float *in, float *out, const float *weight,
                              const float *bias, int n_in, int n_out, double *macs, const void *in_bf16, long long weight_tag,
                            const float *add_in, void *out_bf16);

/* *_backward (pybind.cpp:60-65,84-89,139-143; CPU/Convolution.cpp:81-115,152-185; CPU/Deconvolution.cpp:43-77):
 * d_in [nIn rows][Cin] is overwritten (scn_submanifold_convolution_backward: NULL = not wanted, skipped), d_weight [K][Cin][Cout]
 * is overwritten, d_bias NULL or [Cout]. */
int scn_submanifold_convolution_backward(scn_metadata *m, const long spatial_size[3], const long filter_size[3],
                                         const float *in, float *d_in, const float *d_out, const float *weight,
                                         float *d_weight, float *d_bias, int n_in, int n_out);
int scn_convolution_backward(scn_metadata *m, const long in_size[3], const long out_size[3], const long filter_size[3],
                             const long filter_stride[3], const float *in, float *d_in, const float *d_out,
                             const float *weight, float *d_weight, float *d_bias, int n_in, int n_out);
int scn_deconvolution_backward(scn_metadata *m, const long in_size[3], const long out_size[3], const long filter_size[3],
                               const long filter_stride[3], const float *in, float *d_in, const float *d_out,
                               const float *weight, float *d_weight, float *d_bias, int n_in, int n_out);

/* BatchNormalization_updateOutput (pybind.cpp:219-220; CPU/BatchNormalization.cpp:12-62).
 * mode 0 = train, 1 = eval with the given running stats, 2 = eval with
 * track_running_stats=False (batchNormalization.py:51-56: mean(0) / unbiased var(0) of this input).
 * weight / bias may be NULL.  leakiness 0 = ReLU, 1 = no activation.
 * out_bf16: NULL, or [n_rows][n_planes] 16-bit values (bfloat16; float16 in math mode 5) that receive `out`
 * rounded to nearest (the gather operand of a following convolution in math mode 2 / 5; n_planes % 4 == 0). */
int scn_batchnorm_forward(const float *in, float *out, long n_rows, int n_planes, float *save_mean, float *save_invstd,
                          float *running_mean, float *running_var, const float *weight, const float *bias, float eps,
                          float momentum, int mode, float leakiness, void *stream, void *out_bf16);
/* BatchNormalization_backward (pybind.cpp:221; CPU/BatchNormalization.cpp:64-107); d_out is rewritten in place. */
int scn_batchnorm_backward(const float *in, float *d_in, const float *out, float *d_out, long n_rows, int n_planes,
                           const float *save_mean, const float *save_invstd, const float *weight, float *d_weight,
                           float *d_bias, float leakiness, void *stream);

/* NetworkInNetwork_updateOutput / _updateGradInput / _accGradParameters (pybind.cpp:224-228; CPU/NetworkInNetwork.cpp:7-46):
 * out[n][n_out] = bias + in[n][n_in] @ weight[n_in][n_out]; d_in = d_out @ weight^T; d_weight = in^T @ d_out and
 * d_bias = column sums of d_out (both overwritten; d_bias may be NULL).  *macs = n_rows * n_in * n_out.  in_bf16 /
 * weight_tag as for the convolutions. */
int scn_network_in_network_forward(const float *in, float *out, const float *weight, const float *bias, long n_rows, int n_in, int n_out,
                                   double *macs, void *stream, const void *in_bf16, long long weight_tag);
int scn_network_in_network_backward_input(float *d_in, const float *d_out, const float *weight, long n_rows, int n_in, int n_out, void *stream);
int scn_network_in_network_backward_params(const float *in, const float *d_out, float *d_weight, float *d_bias, long n_rows, int n_in, int n_out,
                                           void *stream);

/* AddTable / add_feature_planes (sparseconvnet/tables.py:28-41, utils.py:61-66): out = a + b */
int scn_add_features(const float *a, const float *b, float *out, long n_elements, void *stream, void *out_bf16);

/* ---- recorded layer programs (no reference counterpart: the reference drives every layer from Python,
 * one pybind call per layer).  A program is the list of the calls above that one forward of a network
 * makes, recorded once by the host layer and replayed by ONE call: same kernels, same order, same
 * results, without ~100 Python round trips per forward.  Feature tensors are registers (0..n_regs-1);
 * their buffers are allocated on `stream` and freed after their last use, output registers stay valid
 * until the next run / destroy.  Op kinds and integer arguments:
 *   0 INPUT  : out, size[3], mode, batch_size, n_planes                      (scn_input_layer_build + _forward)
 *   1 SUBM   : in, out, size[3], filter[3], w, bias, n_in, n_out             (scn_submanifold_convolution_forward)
 *   2 CONV   : in, out, in_size[3], out_size[3], filter[3], stride[3], w, bias, n_in, n_out
 *   3 DECONV : same argument layout as CONV                                   (scn_deconvolution_forward)
 *   4 BN     : in, out, n_planes, weight, bias, running_mean, running_var, mode;  fargs eps, momentum, leakiness
 *   5 ADD    : a, b, out                                                      (scn_add_features)
 * w / bias / ... are indices into the params[] array given to scn_program_run (-1 = none). */
typedef struct scn_program scn_program;
int scn_program_create(scn_program **out);
void scn_program_destroy(scn_program *p);
int scn_program_add(scn_program *p, int kind, const long *iargs, int n_iargs, const double *fargs, int n_fargs);
int scn_program_finish(scn_program *p, int n_regs, const int *outputs, int n_outputs);
int scn_program_run(scn_program *p, scn_metadata *m, const long *coords, int coords_on_device, long nrows, int ncols,
                    const float *features, const void *const *params, const long long *weight_tags, int n_params,
                    void *stream, double *macs);
/* Training replay.  scn_program_set_training(p, 1): scn_program_run keeps every register (and every BatchNorm's saved mean / inverse
 * standard deviation) until the next run, writes nothing as bf16 only and runs the layers on the caller's Metadata in the
 * reference's numbering.  scn_program_backward then runs the backward pass of that run, op by op in reverse, through the same
 * scn_*_backward entries the per-layer autograd Functions use (the reference: one autograd node per layer,
 * sparseconvnet/{submanifoldConvolution,convolution,deconvolution,batchNormalization}.py).  d_out[i] = gradient of output register
 * out_regs[i] (device, not modified); param_grads[j] = device buffer for parameter j's gradient (overwritten) or NULL; param_live[j]
 * (host, may be NULL) = 1 when parameter j received one -- ops that reach no output are skipped, as autograd skips them;
 * d_features = NULL or the gradient of the network input.  The Metadata of the run must still be alive. */
int scn_program_set_training(scn_program *p, int on);
int scn_program_backward(scn_program *p, int n_out, const int *out_regs, const float *const *d_out, const void *const *params, void *const *param_grads,
                         int n_params, float *d_features, int *param_live, void *const *param_events);
/* param_events: NULL, or one cudaEvent_t (or NULL) per parameter, recorded on the program's stream right behind the kernels that
 * write that parameter's gradient: a data-parallel caller lets the all-reduce of a gradient bucket wait for the event of the bucket's
 * last parameter only, so that the collective overlaps the rest of the backward pass (the reference: DistributedDataParallel's
 * bucketed all-reduce, tools/train_net_sparse3d.py:52-58). */
/* Internal row numbering (used by scn_program_run, never handed to callers): rows of every grid are numbered by spatial
 * index instead of the reference's first-touch order in dense_hash_map iteration order, which removes the hash-order
 * emulation from the critical path.  scn_rows_to_reference_order hands a feature matrix computed under such a Metadata
 * out in the reference numbering of an ordinary Metadata built from the same input. */
int scn_metadata_set_internal_numbering(scn_metadata *m, int on);
/* Makes the empty Metadata m the reference-numbered twin of `internal` (one batch item, input layer already built): on a worker
 * thread, m's input layer (grid of spatial_size) and the output grids of the given strided convolutions (ops: n_ops x 13 longs,
 * kind 2, in the order they follow from each other) take their block structure from internal's grids and compute only the
 * reference row ids.  Their rulebooks are built on first use.  `internal` must stay alive until scn_metadata_wait_jobs(m)
 * returns. */
int scn_metadata_build_reference_grids(scn_metadata *m, scn_metadata *internal, const long spatial_size[3], int n_ops, const long *ops);
/* blocks until the Metadata's worker jobs are done; its compute stream then waits for what they queued */
int scn_metadata_wait_jobs(scn_metadata *m);
/* batch items of the grid of this spatial size (0 when there is none) */
int scn_get_batch_size(scn_metadata *m, const long spatial_size[3], int *batch);
int scn_rows_to_reference_order(scn_metadata *ref, scn_metadata *internal, const long spatial_size[3], const float *src, float *dst, int cols);
/* the same for up to 8 feature matrices in one launch (sizes: n_maps x 3) */
int scn_rows_to_reference_order_multi(scn_metadata *ref, scn_metadata *internal, int n_maps, const long *sizes, const float *const *src, float *const *dst,
                                      const int *cols);
/* The inverse for gradients (training replay): dst[internal row of site x] = src[reference row of site x] for every site of
 * the grid `size`; dst [rows][cols] is written completely (the two numberings are bijections of the same site set). */
int scn_rows_from_reference_order(scn_metadata *ref, scn_metadata *internal, const long size[3], const float *src, float *dst, int cols);
/* Build half of a run, callable ahead of scn_program_run for the NEXT input while the GPU still computes the current
 * one (streaming many buildings through one network): input layer + the worker threads that build every rulebook the
 * program requests.  coords_on_device: 0 host, 1 device (ordered after the caller's stream), 2 device and complete.
 * scn_program_run on a Metadata prepared this way skips its own build. */
int scn_program_prepare(scn_program *p, scn_metadata *m, const long *coords, int coords_on_device, long nrows, int ncols);
/* Training step i+1 prepared while step i still runs (program in training mode): builds ahead what scn_program_run would build
 * before the first layer of a training step on the empty Metadata m -- the internally numbered Metadata with its input layer and
 * plan hints, and the reference-numbered twin on m -- or, where that step runs on m itself (several batch items,
 * SCN_TRAIN_INTERNAL=0, input modes 0), scn_program_prepare on m.  The rule lists the backward pass will read are hinted after the
 * plans (scn_metadata_prefetch kinds 4 / 5; an unprepared step builds them on demand).  Does not wait for the GPU work queued before
 * (call scn_program_throttle and scn_set_pool_growth(1) around creating m, as for scn_program_prepare).  The program keeps at most two
 * prepared steps: a third drops the oldest, whose m then remains an ordinary Metadata; dropping waits on the host for that step's
 * reference numbering to finish, which waits on the GPU only when the Metadata memory pool has grown past its bound.  A
 * scn_program_run of this program on m computes exactly what it computes on an unprepared Metadata.  m must stay alive until that
 * run, until it is dropped, or until the program is destroyed. */
int scn_program_prepare_training(scn_program *p, scn_metadata *m, const long *coords, int coords_on_device, long nrows, int ncols);
/* Drops every step prepared by scn_program_prepare_training (with its internally numbered Metadata); their Metadata m remain ordinary
 * Metadata.  For a caller that stops training for a while (evaluation), so that the prepared steps do not hold their memory. */
int scn_program_drop_prepared(scn_program *p);
/* Blocks until at most one forward of this program is still running on the GPU (call before scn_metadata_create of the
 * Metadata to prepare: it then reuses the memory of the forward that just finished). */
int scn_program_throttle(scn_program *p);
/* 1 while a Metadata is created / prepared AHEAD of its forward: its memory may then come from fresh chunks instead of
 * waiting for chunks a still-running forward owns (bounded pool growth); 0 (default) otherwise. */
int scn_set_pool_growth(int on);
int scn_program_output(scn_program *p, int reg, long *rows, int *cols, const float **ptr);
/* output register -> caller's device buffer [rows][cols], in the row numbering of the caller's Metadata `m` */
int scn_program_output_copy(scn_program *p, scn_metadata *m, int reg, const long spatial_size[3], float *dst);
/* every output register of the last run at once (n <= 8; sizes: n x 3): one gather launch */
int scn_program_outputs_copy(scn_program *p, scn_metadata *m, int n, const int *regs, const long *sizes, float *const *dst);
/* device-to-device copy on `stream` (hands an output register to a caller-owned tensor) */
int scn_copy_device(void *dst, const void *src, long bytes, void *stream);

/* SparseToDense_updateOutput / _updateGradInput (pybind.cpp: SparseToDense_*; CPU/SparseToDense.cpp:34-101): out = zero-filled
 * [batch][n_planes][X][Y][Z] float32 with out[b][c][x][y][z] = in[row of the site][c]; d_in[row][c] = d_out[b][c][x][y][z]
 * (every row of the grid is written).  Both run on the Metadata's compute stream. */
int scn_sparse_to_dense_forward(scn_metadata *m, const long spatial_size[3], const float *in, float *out, int n_planes);
int scn_sparse_to_dense_backward(scn_metadata *m, const long spatial_size[3], float *d_in, const float *d_out, int n_planes);

/* ---- first consumers of the backbone's maps (SURVEY.md section 8f rank 1): the RPN head and its anchors.
 * RPNHead.forward for ONE feature map (maskrcnn_benchmark/modeling/rpn/rpn_sparse3d.py:81-131): t = relu(conv(x)), logits =
 * cls_logits(t), reg = bbox_pred(t); the three layers are 1x1 Conv2d on [1, C, n, 1] = GEMMs over the n feature rows.  Weights in
 * Conv2d layout [out][in] (kernel 1x1), biases may be NULL.  logits [n][n_cls], reg [n][n_reg] -- the memory the reference's
 * permute(0,2,1,3).reshape(1, n, A, sep) / (1, n, A, 7 sep) views.  One kernel, exact fp32. */
int scn_rpn_head_forward(const float *feats, long n_rows, int n_planes, const float *w_conv, const float *b_conv, const float *w_cls, const float *b_cls,
                         int n_cls, const float *w_reg, const float *b_reg, int n_reg, float *logits, float *reg, void *stream);
/* AnchorGenerator.grid_anchors for one map (anchor_generator_sparse3d.py:88-104): anchors[(row * A + a)][7] =
 * [loc_xyz / voxel_scale * stride, 0, 0, 0, 0] + base_anchors[a]; locations = DEVICE int64 [n][4] as scn_get_spatial_locations
 * (out_on_device = 1) returns them, base_anchors = device float32 [A][7] (generate_anchors_3d, :213-250). */
int scn_rpn_grid_anchors(const long *locations, long n_rows, float voxel_scale, const float stride[3], const float *base_anchors, int n_anchors, float *anchors,
                         void *stream);

/* ROIAlignRotated3D on a SPARSE feature map (SURVEY.md section 8f rank 3): what maskrcnn_benchmark/layers/roi_align_rotated_3d.py:56-86
 * computes by densifying the map (sparse_3d_to_dense_2d) and running csrc/cuda/ROIAlignRotated3D_cuda.cu:89-172 / :238-346 on it,
 * evaluated straight from the sparse grid.  feats [nActive][n_planes]; extent = the occupied extent the reference crops the dense
 * tensor to (max coordinate + 1 per dimension = its height, width, zsize); rois = device float32 [n_rois][8] (batch, center_w,
 * center_h, center_z, w, h, z, theta in degrees); out [n_rois][n_planes][ph][pw][pz]; d_feats [nActive][n_planes] is overwritten
 * (zero where no sample touches a site).  Both run on the Metadata's compute stream. */
int scn_roi_align_rotated_3d_forward(scn_metadata *m, const long spatial_size[3], const float *feats, int n_planes, const int extent[3], const float *rois,
                                     long n_rois, float spatial_scale, int pooled_h, int pooled_w, int pooled_z, int sampling_ratio, float *out);
/* (accumulates with float atomics in every mode: not reproducible bit for bit, see scn_set_deterministic) */
int scn_roi_align_rotated_3d_backward(scn_metadata *m, const long spatial_size[3], float *d_feats, int n_planes, const int extent[3], const float *rois,
                                      long n_rois, float spatial_scale, int pooled_h, int pooled_w, int pooled_z, int sampling_ratio, const float *d_out);

/* ---- the steps either side of the path (SURVEY.md section 8f rank 4): RPN post-processing and the input voxeliser.  All pointers
 * are DEVICE pointers unless stated otherwise; everything runs on `stream`.
 *
 * torch.topk(values, k, sorted=True) (inference_3d.py:101-104, box_torch_ops.py:495-499): the k largest values in descending order and
 * their indices; apply_sigmoid = 1 ranks sigmoid(values) (objectness.sigmoid().topk) and returns the sigmoid values.  Ties: lower
 * index first (torch leaves the order of equal values unspecified). */
int scn_top_k_descending(const float *values, long n, int apply_sigmoid, long k, float *out_values, long *out_indices, void *stream);
/* BoxCoder3D.decode (maskrcnn_benchmark/modeling/box_coder_3d.py:38-65 -> second_box_decode, second/pytorch/core/box_torch_ops.py:51-88):
 * boxes[i] = decode(encodings[j] / weights, anchors[j]), j = indices[i] (or i when indices is NULL); sizes clamped to `clip`, smooth_dim
 * 1 = (t + 1) * a, 0 = exp(t) * a; yaw wrapped into [-pi/2, pi/2) by limit_period(., 0.5, pi).  weights = HOST float[7]. */
int scn_box_decode_3d(const float *encodings, const float *anchors, const long *indices, long n, const float weights[7], float clip, int smooth_dim, float *boxes,
                      void *stream);
/* boxes_iou_3d (utils3d/rotate_nms_3d_torch.py:22-84): iou[t][a] = rotated BEV IoU (rotate_iou_gpu_eval, second/core/non_max_suppression/
 * nms_gpu.py:548-667, criterion -1 / 0 / 1 / 2 / other = intersection area; identical rectangles forced to 1) times the IoU of the z
 * extents (only_xy = 0).  Boxes are yx_zb rows [x, y, z_bottom, size_y, size_x, size_z, yaw]; aug_thickness = HOST float[4] = minimum
 * size_y / size_z of the targets, then of the anchors (NULL = no augmentation). */
int scn_boxes_iou_3d(const float *targets, long n_targets, const float *anchors, long n_anchors, const float aug_thickness[4], int criterion, int only_xy, float *iou,
                     void *stream);
/* rotate_nms_3d (second/pytorch/core/box_torch_ops.py:489-514 -> rotate_nms_3d_cc, second/core/non_max_suppression/nms_cpu.py:32-44):
 * top pre_max_size boxes by score, greedy suppression in score order (a kept box removes every later box whose 3-D IoU with it is
 * positive and whose BEV polygon IoU reaches iou_threshold), first post_max_size survivors.  keep = device long[>= min(n, post_max_size)]
 * receives indices into `boxes`, n_keep = device long[1] their count.  At most 16384 candidates after pre_max_size. */
int scn_rotate_nms_3d(const float *boxes, const float *scores, long n, long pre_max_size, long post_max_size, float iou_threshold, long *keep, long *n_keep,
                      void *stream);
/* Input voxeliser (data3d/suncg_utils/suncg_dataset.py:115-177): a = xyz @ matrix + offset (float64), rows with any coordinate outside
 * [0, full_scale) dropped (order kept), locs = trunc(a) as int64 [kept][loc_cols] (loc_cols 4 appends batch_index), feats_out = feats with
 * columns 0..2 replaced by a / scale when xyz_in_feats.  matrix (row-major 3x3, as numpy's a @ m), offset, full_scale = HOST doubles;
 * n_kept = HOST long, written after a stream synchronisation.  scn_voxelize_extent returns min / max of xyz @ matrix per coordinate
 * (the `offset = -a.min(0)` of :131-134) to HOST doubles. */
int scn_voxelize_extent(const float *xyz, long n, const double matrix[9], double extent_min[3], double extent_max[3], void *stream);
int scn_voxelize(const float *xyz, const float *feats, long n, int n_feat, const double matrix[9], const double offset[3], double scale, const double full_scale[3],
                 int xyz_in_feats, long batch_index, int loc_cols, long *locs, float *feats_out, long *n_kept, void *stream);

/* Selects the arithmetic of the gather-GEMM kernels for this process: 0 = fp32 CUDA cores
 * (exact-fp32 anchor), 1 = tcgen05 tensor cores, TF32 inputs / fp32 accumulate (default where the
 * channel counts allow), 2 = tcgen05 BF16 inputs / fp32 accumulate, 3 = tcgen05 "3xTF32": each fp32
 * operand split into two exact TF32 values hi + lo, three TF32 products (hi*lo, lo*hi, hi*hi) in one fp32
 * accumulator, fp32-class accuracy, 5 = tcgen05 FP16 inputs / fp32 accumulate wherever mode 2 has BF16 inputs
 * (everything else as in mode 2): 11 significant bits instead of 8, range +-65504 -- conversions round to nearest
 * even with IEEE overflow (a larger value becomes +-inf and propagates) and keep subnormals.  Code 4 is not a mode.
 * The tensor-core kernels take convolutions with up to 1024 input channels and, in multiples of 32, up to 1024 output
 * channels (layers wider than 256 run as column slabs of <= 256).  In modes 1 and 3 every convolution the tensor-core kernel
 * cannot take, and every weight gradient, runs on the exact fp32 CUDA-core kernels -- except, in mode 3, the weight gradients of
 * up to 256 x 256 channels (Cin <= 32, a multiple of 32 up to 128, or 256; Cout a multiple of 32 up to 256; up to 64 filter
 * offsets -- so not Cin 160, 192 or 224): these run on the
 * tensor cores with each fp32 operand split exactly into three bf16 parts (six products, fp32-class accuracy); in modes 2 and 5
 * the weight gradients of up to 1024 x 1024 channels (multiples of 32 beyond 256) run on the tensor cores too. */
int scn_set_math_mode(int mode);
int scn_get_math_mode(void);
/* Deterministic mode for this process (0 = off, the default): with 1, every float result of the calls above except
 * scn_roi_align_rotated_3d_backward is bitwise reproducible from run to run for a fixed build, GPU model, math mode and
 * inputs.  Launches that would accumulate floats with atomics (split filter offsets, BatchNorm statistics, weight and bias
 * gradients) write per-work-item partial sums to fixed slots of a per-stream workspace instead and add them in index
 * order.  Read by every launch, so a change applies from the next call on, recorded programs included.  The Python
 * package follows torch.are_deterministic_algorithms_enabled(). */
int scn_set_deterministic(int on);
int scn_get_deterministic(void);
/* 1 when the tcgen05 kernels are compiled in and the device is sm_100 */
int scn_tensor_core_path_available(void);
/* number of kernels this library has launched since load (for bench.py's gpu_launches) */
long scn_kernel_launch_count(void);
/* developer counters.  Metadata memory pool: 0 = chunks taken from the driver, 1 = waits for a chunk still in use, 2 = pool
 * size in MiB.  Which code path ran (monotonic since load; the parity tests assert on their deltas): 3 = tensor-core launches
 * that carried a lateral 1x1x1 stage, 4 = launches whose epilogue accumulated BatchNorm statistics, 5 = program registers
 * written as bf16 only, 6 = laterals run as a separate convolution + add (fallback), 7 = tcgen05 convolution launches,
 * 8 = BatchNorm ops applied from epilogue statistics, 9 = launches that split the filter offsets over CTAs (atomic
 * epilogue), 10 = CUDA-core convolution launches, 11 = backward passes run by scn_program_backward, 12 = bf16 operand copies the
 * weight-gradient kernel took from its caller (forward shadow / shared d_out copy) instead of converting again, 13 = weight-gradient
 * launches driven by the output-stationary plan, 14 = float-atomic launches: launches whose float result depends on the order in
 * which atomics land (0 in deterministic mode except for scn_roi_align_rotated_3d_backward), 17 = host -> device copies of
 * input-layer coordinates, 18 = tensor-core launches with fp16 operands (convolutions and weight gradients, math mode 5), 19 = rule
 * lists a convolution's backward entry found already built (hinted ahead by a training run), 20 = training runs that took a Metadata
 * prepared by scn_program_prepare_training, 21 = CUDA-core weight-gradient
 * launches of the sparse convolutions (k_dw, one per non-empty rule list; NetworkInNetwork's dense weight gradient is not counted),
 * 22 = tensor-core weight-gradient launches with split operands (math mode 3, one per channel block of <= 128 x <= 128). */
long scn_debug_counter(int which);
/* Hands the library's idle device memory back to the driver: Metadata chunks not owned by a live Metadata, cached weight operand
 * images, per-stream scratch buffers (the library recycles these itself instead of returning them; torch.cuda.empty_cache() cannot
 * see them).  Synchronises the device first.  Returns the number of bytes released, -1 on a CUDA error.  Live Metadata objects and
 * recorded programs keep their memory (destroy them first). */
long scn_release_cached_memory(void);

/* Fusion requests for the next call this thread makes to scn_submanifold_convolution_forward, scn_convolution_forward or
 * scn_deconvolution_forward, and to no other entry: that call takes the pending requests when it is entered, whether or not it
 * can honour them (the fusions of a recorded program: the FPN's lateral 1x1x1 convolution and the statistics of a following
 * BatchNorm folded into a convolution; no reference counterpart:
 * the reference runs NetworkInNetwork / SubmanifoldConvolution(1), AddTable and BatchNormalization as separate passes,
 * fpn_net.py:166-176, CPU/BatchNormalization.cpp:12-62).
 *  lateral: out = conv(in) [+ add_in] + lat_in[row] @ lat_weight ([n_in][n_out], one filter offset), lat_in_bf16 = 16-bit
 *           copy of lat_in in the mode's format (needed in math modes 2 and 5);
 *  stats:   sums = [8 replicas][2][128] doubles, zeroed by the caller; the launch adds per-channel sum (first 128) and sum
 *           of squares (second 128) of the rows it stores, spread over the replicas (deterministic mode: written into replica
 *           0 after the launch, in a fixed order).
 * A call that cannot honour a request (CUDA-core path, packed rows, split offsets, > 128 channels) drops it;
 * scn_fuse_result reports what the last of those three calls took and disarms both requests. */
int scn_fuse_next_lateral(const float *lat_in, const void *lat_in_bf16, const float *lat_weight, long long weight_tag, int n_in, long rows);
int scn_fuse_next_stats(double *sums);
int scn_fuse_result(int *lateral_taken, int *stats_taken);

#ifdef __cplusplus
}
#endif
#endif
