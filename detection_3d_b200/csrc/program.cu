// Recorded layer programs: the sequence of native calls one forward of a network makes, replayed by
// ONE C-ABI call.  The reference drives every layer from Python (sparseconvnet/*.py -> one pybind
// call per layer); on B200 the ~100 layer calls of the Detection_3D backbone cost more host time
// (Python + ctypes, ~60 us each) than the GPU needs for the small pyramid levels.  A program is
// nothing but the same calls of include/scn_b200.h issued from C++: same kernels, same order,
// same results; feature tensors live in registers whose buffers the executor allocates on the
// caller's stream and frees after their last use.
#include "../../include/scn_b200.h"
#include "conv.cuh"
#include <algorithm>
#include <stdlib.h>
#include <array>
#include <deque>
#include <utility>
#include <vector>

namespace {

constexpr long kHalfOnlyRows = 32768; // from here on a convolution never splits its filter offsets over CTAs (its epilogue stores final values)
enum Kind { K_INPUT = 0, K_SUBM = 1, K_CONV = 2, K_DECONV = 3, K_BN = 4, K_ADD = 5 };
struct Op {
  int kind;
  long a[24];
  double f[4];
};
struct Reg {
  float *p = nullptr;
  void *p16 = nullptr; // 16-bit copy (math mode 2: bfloat16, 5: fp16; written by BatchNorm / add)
  long rows = 0;
  int cols = 0;
  int pad16 = 0; // > 0: p16 holds the rows zero-padded to this many channels (network input in bf16 / fp16 mode)
};

} // namespace

// Register buffers come from slots the program keeps across runs (best fit, single stream => a slot
// freed after its register's last use can be handed to the next register right away).  The CUDA
// stream-ordered pool was measured to take 2-7 ms for the 300-600 MB level-0 buffers here.
struct Slot { void *p; size_t cap; bool busy; };

struct scn_program {
  std::vector<Slot> slots;
  std::vector<Op> ops;
  int nRegs = 0;
  std::vector<int> lastUse;     // op index after which a register's buffers can be freed
  std::vector<char> isOutput;
  std::vector<std::array<long, 3>> outSize; // spatial size of the grid every register lives on
  std::vector<Reg> regs;
  float *bnScratch = nullptr;   // saveMean / saveInvStd of inference-mode BatchNorm (unused downstream)
  int nStats = 0;               // convolutions whose epilogue accumulates the statistics of the BatchNorm that follows
  double *stats = nullptr;      // nStats x [kBnReplicas][2][kFusedStatsC], zeroed at the start of every run
  std::vector<char> statsDone;
  scn_metadata *ms = nullptr;   // internally numbered Metadata of the current / last run (see scn_program_run)
  bool internal = false;        // the registers of the last run are in internal row order
  cudaEvent_t evEnd[2] = {nullptr, nullptr}; // end of the last two runs on `stream` (throttle of scn_program_prepare)
  long nRuns = 0;
  cudaStream_t stream = nullptr;
  // Training replay (scn_program_set_training): every register stays alive until the next run, nothing is written as bf16 only,
  // the layers run on the caller's Metadata (reference numbering), and every BatchNorm keeps its saveMean / saveInvStd for
  // scn_program_backward.
  bool train = false;
  std::vector<float *> bnSave;  // per op: [2][C] floats (train mode), from the slot pool
  scn_metadata *lastMd = nullptr; // Metadata the layers of the last training run ran on (the backward pass needs its rulebooks): the caller's, or `ms`
  scn_metadata *lastRef = nullptr; // the caller's Metadata of that run (reference numbering: the order gradients arrive in)
  // Training steps prepared ahead (scn_program_prepare_training), oldest first: the caller's Metadata and the internally numbered
  // one its run will take (nullptr: the run uses the caller's Metadata itself, which was prepared instead)
  std::deque<std::pair<scn_metadata *, scn_metadata *>> prepared;
};

static void *slot_get(scn_program *p, size_t bytes) {
  bytes = std::max<size_t>(bytes, 256);
  int best = -1;
  for (int i = 0; i < (int)p->slots.size(); i++) {
    const Slot &s = p->slots[i];
    if (!s.busy && s.cap >= bytes && s.cap <= 4 * bytes + (1u << 20) && (best < 0 || s.cap < p->slots[best].cap)) best = i;
  }
  if (best < 0) {
    Slot s{nullptr, (bytes + bytes / 8 + (1u << 20) - 1) & ~(size_t)((1u << 20) - 1), true}; // 12 % headroom: buildings differ a little
    if (cudaMalloc(&s.p, s.cap) != cudaSuccess) { scn::set_error("program: cudaMalloc failed"); return nullptr; }
    p->slots.push_back(s);
    return s.p;
  }
  p->slots[best].busy = true;
  return p->slots[best].p;
}
static void slot_put(scn_program *p, void *ptr) {
  for (Slot &s : p->slots) if (s.p == ptr) { s.busy = false; return; }
}
// Forgets a prepared training step: its twin job reads the internally numbered Metadata, which goes with it, so the host waits
// for that job first.  The job waits for nothing but build work -- except when the Metadata chunk pool has grown past its bound
// (alloc_in): a chunk the running step still owns is then waited for on the GPU.
static void drop_prepared(const std::pair<scn_metadata *, scn_metadata *> &e) {
  if (!e.second) return;
  scn_metadata_wait_jobs(e.first);
  scn_metadata_destroy(e.second);
}
static void release_regs(scn_program *p, bool outputsToo) {
  if (outputsToo) {
    for (float *&b : p->bnSave) if (b) { slot_put(p, b); b = nullptr; }
  }
  for (size_t i = 0; i < p->regs.size(); i++) {
    Reg &r = p->regs[i];
    if (!outputsToo && p->isOutput[i]) continue;
    if (r.p) slot_put(p, r.p);
    if (r.p16) slot_put(p, r.p16);
    r.p = nullptr;
    r.p16 = nullptr;
  }
}

extern "C" {

int scn_program_create(scn_program **out) {
  *out = new scn_program();
  return 0;
}
void scn_program_destroy(scn_program *p) {
  if (!p) return;
  release_regs(p, true);
  cudaDeviceSynchronize();
  for (Slot &s : p->slots) cudaFree(s.p);
  if (p->bnScratch) cudaFree(p->bnScratch);
  if (p->stats) cudaFree(p->stats);
  for (cudaEvent_t e : p->evEnd) if (e) cudaEventDestroy(e);
  if (p->ms) scn_metadata_destroy(p->ms);
  for (const auto &e : p->prepared) drop_prepared(e);
  delete p;
}
int scn_program_set_training(scn_program *p, int on) {
  SCN_CHECK(p, "null program");
  p->train = on != 0;
  return 0;
}
int scn_program_add(scn_program *p, int kind, const long *iargs, int n_iargs, const double *fargs, int n_fargs) {
  SCN_CHECK(p && kind >= K_INPUT && kind <= K_ADD && n_iargs <= 24 && n_fargs <= 4, "bad program op");
  Op op;
  op.kind = kind;
  for (int i = 0; i < 24; i++) op.a[i] = i < n_iargs ? iargs[i] : 0;
  for (int i = 0; i < 4; i++) op.f[i] = i < n_fargs ? fargs[i] : 0.0;
  op.a[18] = -1; // lateral 1x1x1 convolution folded into this convolution: its input register, weight parameter (a[19]), channels (a[20])
  op.a[21] = -1; // statistics slot shared by a convolution and the BatchNorm ops that read its output (scn_program_finish)
  op.a[23] = 0;
  op.a[22] = -1; // register added in the epilogue of a convolution (set by the fusion pass of scn_program_finish)
  p->ops.push_back(op);
  return 0;
}
int scn_program_finish(scn_program *p, int n_regs, const int *outputs, int n_outputs) {
  SCN_CHECK(p && n_regs > 0, "bad program");
  { // Fuse `ADD(conv_out, other)` into the convolution's epilogue (out = conv + other, one kernel and one pass
    // over the rows less): AddTable after a residual block, add_feature_planes after a Deconvolution.
    auto out_of = [](const Op &o) -> long { return o.kind == K_INPUT ? o.a[0] : (o.kind == K_ADD ? o.a[2] : o.a[1]); };
    std::vector<int> producer(n_regs, -1), consumers(n_regs, 0);
    std::vector<char> isOut(n_regs, 0);
    for (int i = 0; i < n_outputs; i++) if (outputs[i] >= 0 && outputs[i] < n_regs) isOut[outputs[i]] = 1;
    for (int i = 0; i < (int)p->ops.size(); i++) {
      const Op &o = p->ops[i];
      long r = out_of(o);
      SCN_CHECK(r >= 0 && r < n_regs, "register index");
      producer[r] = i;
      if (o.kind == K_ADD) { consumers[o.a[0]]++; consumers[o.a[1]]++; }
      else if (o.kind != K_INPUT) consumers[o.a[0]]++;
    }
    std::vector<char> dead(p->ops.size(), 0);
    for (int i = 0; i < (int)p->ops.size(); i++) {
      Op &add = p->ops[i];
      if (add.kind != K_ADD) continue;
      const long ra = add.a[0], rb = add.a[1];
      const int pa = producer[ra], pb = producer[rb];
      if (pa < 0 || pb < 0 || pa == pb) continue;
      const int host = std::max(pa, pb);               // the operand produced last; the other one exists by then
      const long hostReg = host == pa ? ra : rb, other = host == pa ? rb : ra;
      Op &h = p->ops[host];
      if (h.kind != K_SUBM && h.kind != K_CONV && h.kind != K_DECONV) continue;
      if (consumers[hostReg] != 1 || isOut[hostReg] || h.a[22] >= 0) continue;
      h.a[22] = other;
      h.a[1] = add.a[2]; // the convolution now writes the sum
      producer[add.a[2]] = host;
      dead[i] = 1;
    }
    std::vector<Op> kept;
    for (int i = 0; i < (int)p->ops.size(); i++) if (!dead[i]) kept.push_back(p->ops[i]);
    p->ops.swap(kept);
  }
  { // Lateral 1x1x1 convolutions: `conv(x) + NiN(y)` (the FPN's top-down step: Deconvolution + shortcut) becomes ONE kernel
    // that accumulates y[row] @ W_nin into the same TMEM accumulators as an extra stage, so the lateral tensor is never
    // written or read.  Pattern: a convolution with a fused addend whose producer is a bias-free 1x1x1 SubmanifoldConvolution
    // consumed by nothing else.
    auto out_of = [](const Op &o) -> long { return o.kind == K_INPUT ? o.a[0] : (o.kind == K_ADD ? o.a[2] : o.a[1]); };
    std::vector<int> producer(n_regs, -1), consumers(n_regs, 0);
    std::vector<char> isOut(n_regs, 0);
    for (int i = 0; i < n_outputs; i++) if (outputs[i] >= 0 && outputs[i] < n_regs) isOut[outputs[i]] = 1;
    for (int i = 0; i < (int)p->ops.size(); i++) {
      const Op &o = p->ops[i];
      producer[out_of(o)] = i;
      if (o.kind == K_ADD) { consumers[o.a[0]]++; consumers[o.a[1]]++; }
      else if (o.kind != K_INPUT) { consumers[o.a[0]]++; if (o.kind != K_BN && o.a[22] >= 0) consumers[o.a[22]]++; }
    }
    std::vector<char> dead(p->ops.size(), 0);
    static const bool on = !(getenv("SCN_LATERAL_FUSED") && atoi(getenv("SCN_LATERAL_FUSED")) == 0);
    for (int i = 0; on && i < (int)p->ops.size(); i++) {
      Op &h = p->ops[i];
      if ((h.kind != K_SUBM && h.kind != K_CONV && h.kind != K_DECONV) || h.a[22] < 0) continue;
      const long r = h.a[22];
      const int j = producer[r];
      if (j < 0 || j >= i || consumers[r] != 1 || isOut[r]) continue;
      const Op &nin = p->ops[j];
      if (nin.kind != K_SUBM || nin.a[5] != 1 || nin.a[6] != 1 || nin.a[7] != 1 || nin.a[9] >= 0) continue; // 1x1x1, no bias
      const long ninOutC = nin.a[11], hostOutC = h.kind == K_SUBM ? h.a[11] : h.a[17];
      if (ninOutC != hostOutC) continue;
      h.a[18] = nin.a[0]; h.a[19] = nin.a[8]; h.a[20] = nin.a[10];
      h.a[22] = -1;
      dead[j] = 1;
    }
    std::vector<Op> kept;
    for (int i = 0; i < (int)p->ops.size(); i++) if (!dead[i]) kept.push_back(p->ops[i]);
    p->ops.swap(kept);
  }
  { // BatchNorm statistics in the producing convolution's epilogue: BN(conv_out) with batch statistics (modes 0 / 2)
    // reads per-channel sums the convolution kernel accumulated while it still held the output values, and runs
    // only its apply pass.  Whether a given convolution launch can do it (tensor-core path, no offset splitting,
    // <= 128 channels) is decided at run time; otherwise the BatchNorm computes its own statistics as before.
    auto out_of = [](const Op &o) -> long { return o.kind == K_INPUT ? o.a[0] : (o.kind == K_ADD ? o.a[2] : o.a[1]); };
    std::vector<int> producer(n_regs, -1);
    for (int i = 0; i < (int)p->ops.size(); i++) producer[out_of(p->ops[i])] = i;
    p->nStats = 0;
    for (Op &bn : p->ops) {
      if (bn.kind != K_BN || bn.a[7] == 1 || bn.a[2] > scn::kFusedStatsC || bn.a[2] % 32 != 0) continue;
      const int j = producer[bn.a[0]];
      if (j < 0) continue;
      Op &c = p->ops[j];
      if (c.kind != K_SUBM && c.kind != K_CONV && c.kind != K_DECONV) continue;
      if (c.a[21] < 0) c.a[21] = p->nStats++;
      bn.a[21] = c.a[21];
    }
  }
  { // bf16 mode: a BatchNorm output that only feeds tensor-core convolutions gathering its bf16 copy is never read in fp32;
    // such BatchNorm ops (a[19] = 1) write the bf16 copy only.  Outputs, addends, laterals and anything whose channel counts
    // or geometry may take the TF32 / CUDA-core route keep their fp32 rows.
    std::vector<int> good(n_regs, 0), bad(n_regs, 0);
    for (int i = 0; i < n_outputs; i++) bad[outputs[i]] = 1;
    for (const Op &o : p->ops) {
      if (o.kind == K_INPUT) continue;
      if (o.kind == K_ADD) { bad[o.a[0]] = 1; bad[o.a[1]] = 1; continue; }
      if (o.kind == K_BN) { bad[o.a[0]] = 1; continue; }
      const long Cin = o.kind == K_SUBM ? o.a[10] : o.a[16], Cout = o.kind == K_SUBM ? o.a[11] : o.a[17];
      long K = 1;
      for (int d = 0; d < 3; d++) K *= o.kind == K_SUBM ? o.a[5 + d] : o.a[8 + d];
      // (wider layers run as column slabs of <= 256 that all gather the 16-bit copy when Cin is a multiple of 64)
      const bool tc = Cout % 32 == 0 && Cout >= 32 && K <= 63 &&
                      (Cout <= 256 ? (Cin % 64 == 0 || (Cin == 32 && Cout <= 128)) : (Cout <= 1024 && Cin % 64 == 0 && Cin <= 1024));
      // a deconvolution takes the tensor-core path when every fine site has exactly one parent: guaranteed by filter == stride
      const bool deconvTc = o.kind == K_DECONV && Cin % 64 == 0 && o.a[8] == o.a[11] && o.a[9] == o.a[12] && o.a[10] == o.a[13];
      if (tc && (o.kind != K_DECONV || deconvTc)) good[o.a[0]] = 1; else bad[o.a[0]] = 1;
      if (o.a[22] >= 0) bad[o.a[22]] = 1;
      if (o.a[18] >= 0) bad[o.a[18]] = 1; // whether a lateral is folded in (bf16 copy) or run on its own is decided at run time: keep the fp32 rows
    }
    for (Op &bn : p->ops) if (bn.kind == K_BN) bn.a[19] = (good[bn.a[1]] && !bad[bn.a[1]] && bn.a[2] % 32 == 0) ? 1 : 0;
    // the same for the OUTPUT of a convolution (a[23] = 1): the finest top-down sum deconv(x) + lateral is read only by the
    // merged 3^3 convolution.  Applied at run time to large levels only (no offset splitting there, see launch_conv_plan_tc).
    for (Op &c : p->ops)
      if (c.kind == K_SUBM || c.kind == K_CONV || c.kind == K_DECONV) {
        const long Cout = c.kind == K_SUBM ? c.a[11] : c.a[17];
        c.a[23] = (good[c.a[1]] && !bad[c.a[1]] && Cout % 32 == 0) ? 1 : 0;
      }
  }
  p->nRegs = n_regs;
  p->lastUse.assign(n_regs, -1);
  p->isOutput.assign(n_regs, 0);
  p->regs.assign(n_regs, Reg());
  auto use = [&](long r, int i) -> int {
    SCN_CHECK(r >= 0 && r < n_regs, "register index");
    p->lastUse[r] = i;
    return 0;
  };
  for (int i = 0; i < (int)p->ops.size(); i++) {
    const Op &op = p->ops[i];
    switch (op.kind) {
      case K_INPUT: SCN_TRY(use(op.a[0], i)); break;
      case K_ADD: SCN_TRY(use(op.a[0], i)); SCN_TRY(use(op.a[1], i)); SCN_TRY(use(op.a[2], i)); break;
      default:
        SCN_TRY(use(op.a[0], i));
        SCN_TRY(use(op.a[1], i));
        if (op.kind != K_BN && op.a[22] >= 0) SCN_TRY(use(op.a[22], i));
        if (op.kind != K_BN && op.a[18] >= 0) SCN_TRY(use(op.a[18], i));
        break;
    }
  }
  for (int i = 0; i < n_outputs; i++) {
    SCN_CHECK(outputs[i] >= 0 && outputs[i] < n_regs, "output register");
    p->isOutput[outputs[i]] = 1;
  }
  p->outSize.assign(n_regs, std::array<long, 3>{0, 0, 0});
  for (const Op &o : p->ops) { // grid of every register, propagated from its producer
    auto sz3 = [](const long *v) { return std::array<long, 3>{v[0], v[1], v[2]}; };
    switch (o.kind) {
      case K_INPUT: p->outSize[o.a[0]] = sz3(o.a + 1); break;
      case K_SUBM: p->outSize[o.a[1]] = sz3(o.a + 2); break;
      case K_CONV: case K_DECONV: p->outSize[o.a[1]] = sz3(o.a + 5); break;
      case K_BN: p->outSize[o.a[1]] = p->outSize[o.a[0]]; break;
      case K_ADD: p->outSize[o.a[2]] = p->outSize[o.a[0]]; break;
    }
  }
  return 0;
}

// Training: the (in, out) rule lists the backward pass will read (scn_*_convolution_backward), built on the plan worker after every
// plan, in the order the backward pass requests them.  Only ops whose output reaches a program output (the backward pass skips
// the others); the gradient of the network input is assumed not wanted.  Nothing depends on the features, so a step prepared
// ahead (scn_program_prepare_training) has its lists ready when its backward pass starts.  Only prepared steps get them: queued
// behind an unprepared step's own plans they cost its forward more than they save its backward (DESIGN.md section 8).
// SCN_TRAIN_LISTS_AHEAD (developer switch, read per call: tools/train_stream_bench.py alternates it in one process): 0 = built on
// demand only, 1 (default) = for prepared steps, 2 = for every replayed training step.
static bool lists_ahead(bool prepared) {
  const char *env = getenv("SCN_TRAIN_LISTS_AHEAD");
  const int mode = env ? atoi(env) : 1;
  return mode >= 2 || (mode == 1 && prepared);
}
static void rule_list_hints(const scn_program *p, std::vector<long> &hints) {
  std::vector<char> live(p->nRegs, 0);
  for (int r = 0; r < p->nRegs; r++) live[r] = p->isOutput[r];
  for (int i = (int)p->ops.size() - 1; i >= 0; i--) {
    const Op &o = p->ops[i];
    if (o.kind == K_INPUT) continue;
    if (o.kind == K_ADD) { if (live[o.a[2]]) live[o.a[0]] = live[o.a[1]] = 1; continue; }
    if (!live[o.a[1]]) continue;
    live[o.a[0]] = 1;
    if (o.kind == K_BN) continue;
    if (o.a[22] >= 0) live[o.a[22]] = 1;
    if (o.a[18] >= 0) live[o.a[18]] = 1;
    bool fromInput = false;
    for (const Op &q : p->ops) if (q.kind == K_INPUT && q.a[0] == o.a[0]) fromInput = true;
    const long *f = o.kind == K_SUBM ? o.a + 5 : o.a + 8, *st = o.kind == K_SUBM ? o.a + 5 : o.a + 11;
    const int Cin = (int)(o.kind == K_SUBM ? o.a[10] : o.a[16]), Cout = (int)(o.kind == K_SUBM ? o.a[11] : o.a[17]);
    if (!scn::backward_reads_lists(o.kind, f, st, Cin, Cout, !(fromInput && o.kind == K_SUBM))) continue;
    long h[13] = {0};
    if (o.kind == K_SUBM) { h[0] = 4; for (int d = 0; d < 3; d++) { h[1 + d] = o.a[2 + d]; h[7 + d] = o.a[5 + d]; } }
    else { // the deconvolution's backward reads the lists of the convolution fine -> coarse
      h[0] = 5;
      for (int d = 0; d < 3; d++) {
        h[1 + d] = o.kind == K_CONV ? o.a[2 + d] : o.a[5 + d];
        h[4 + d] = o.kind == K_CONV ? o.a[5 + d] : o.a[2 + d];
        h[7 + d] = o.a[8 + d];
        h[10 + d] = o.a[11 + d];
      }
    }
    bool seen = false; // (layers of one level share a rulebook)
    for (size_t j = 0; j < hints.size() && !seen; j += 13) seen = std::equal(h, h + 13, hints.begin() + j);
    if (!seen) hints.insert(hints.end(), h, h + 13);
  }
}
// The build half of a run: input layer (active sites of the finest grid) and, on the worker threads, every rulebook /
// plan the program will request.  scn_program_run calls it when the Metadata comes unprepared; a caller that streams
// buildings through the network calls it for building i+1 right after it has queued building i
// (coords_on_device = 2: device coordinates that are already complete), so that this build runs while the GPU
// computes building i.
// Streaming throttle: building i+2's Metadata is not started before forward i has finished on the GPU.  Two forwards in
// flight are what the overlap needs (one computing, one queued with its Metadata being built); a host that ran further
// ahead would only pile up Metadata memory.  Call it BEFORE creating the Metadata that scn_program_prepare will fill,
// so that the new Metadata finds the finished forward's memory free.
int scn_program_throttle(scn_program *p) {
  SCN_CHECK(p, "null program");
  if (p->nRuns >= 2 && p->evEnd[p->nRuns & 1]) SCN_CUDA(cudaEventSynchronize(p->evEnd[p->nRuns & 1]));
  return 0;
}
// prepared: a training step prepared ahead (scn_program_prepare_training), which also gets the rule lists of its backward pass
static int prepare_build(scn_program *p, scn_metadata *m, const long *coords, int coords_on_device, long nrows, int ncols, bool prepared) {
  SCN_CHECK(p && m && p->nRegs > 0, "program not finished");
  SCN_TRY(scn_program_throttle(p));
  for (const Op &op : p->ops) {
    if (op.kind != K_INPUT) continue;
    const long *a = op.a;
    long nActive = 0;
    int maxActive = 0;
    SCN_TRY(scn_input_layer_build(m, a + 1, coords, coords_on_device, nrows, ncols, (int)a[5], (int)a[4], &nActive, &maxActive));
    std::vector<long> hints; // the rulebooks this program is about to request, built ahead on the worker threads
    for (const Op &o : p->ops) {
      long h[13] = {0};
      if (o.kind == K_SUBM) { h[0] = 1; for (int d = 0; d < 3; d++) { h[1 + d] = o.a[2 + d]; h[7 + d] = o.a[5 + d]; } }
      else if (o.kind == K_CONV || o.kind == K_DECONV) { h[0] = o.kind == K_CONV ? 2 : 3; for (int d = 0; d < 12; d++) h[1 + d] = o.a[2 + d]; }
      else continue;
      hints.insert(hints.end(), h, h + 13);
    }
    if (p->train && lists_ahead(prepared)) rule_list_hints(p, hints);
    if (!hints.empty()) SCN_TRY(scn_metadata_prefetch(m, (int)(hints.size() / 13), hints.data()));
    return 0;
  }
  scn::set_error("program has no input layer");
  return -2;
}
int scn_program_prepare(scn_program *p, scn_metadata *m, const long *coords, int coords_on_device, long nrows, int ncols) {
  return prepare_build(p, m, coords, coords_on_device, nrows, ncols, false);
}

static const Op *input_op(const scn_program *p) {
  for (const Op &o : p->ops) if (o.kind == K_INPUT) return &o;
  return nullptr;
}
// Whether a run on an unprepared Metadata numbers its rows internally (see scn_program_run).  Training runs do too, so that every
// gather of the forward AND backward pass stays local; SCN_TRAIN_INTERNAL=0 keeps them on the caller's Metadata.
static bool uses_internal_numbering(const scn_program *p, const Op *inOp) {
  static const int internalOn = getenv("SCN_INTERNAL_IDS") ? atoi(getenv("SCN_INTERNAL_IDS")) : 1;
  static const int trainInternal = getenv("SCN_TRAIN_INTERNAL") ? atoi(getenv("SCN_TRAIN_INTERNAL")) : 1;
  return (!p->train || trainInternal) && internalOn && inOp && inOp->a[4] != 0;
}
// The internally numbered Metadata of a run on `m` (see scn_program_run): input layer and plan hints (prepare_build), and
// the reference-numbered twin started on `m`.  *out = nullptr when the input has several batch items: `m` then does everything.
static int start_internal(scn_program *p, scn_metadata *m, const Op *inOp, const long *coords, int coords_on_device, long nrows, int ncols,
                          void *stream, bool prepared, scn_metadata **out) {
  scn_metadata *ms = nullptr;
  SCN_TRY(scn_metadata_create(&ms, stream));
  int rc = scn_metadata_set_internal_numbering(ms, 1);
  if (rc == 0) rc = prepare_build(p, ms, coords, coords_on_device, nrows, ncols, prepared);
  int batch = 0;
  if (rc == 0) rc = scn_get_batch_size(ms, inOp->a + 1, &batch);
  if (rc || batch != 1) { // several batch items: the caller's Metadata does everything (reference numbering throughout)
    scn_metadata_destroy(ms);
    *out = nullptr;
    return rc;
  }
  // the strided convolutions whose output grid an output register lives on, or that lead there
  std::vector<std::array<long, 3>> need;
  for (int r = 0; r < p->nRegs; r++) if (p->isOutput[r]) need.push_back(p->outSize[r]);
  std::vector<long> hints;
  for (bool grew = true; grew;) {
    grew = false;
    for (const Op &o : p->ops) {
      if (o.kind != K_CONV) continue;
      const std::array<long, 3> in{o.a[2], o.a[3], o.a[4]}, out{o.a[5], o.a[6], o.a[7]};
      if (std::find(need.begin(), need.end(), out) != need.end() && std::find(need.begin(), need.end(), in) == need.end()) { need.push_back(in); grew = true; }
    }
  }
  for (const Op &o : p->ops) {
    if (o.kind != K_CONV) continue;
    const std::array<long, 3> out{o.a[5], o.a[6], o.a[7]};
    if (std::find(need.begin(), need.end(), out) == need.end()) continue;
    long h[13] = {0};
    h[0] = 2;
    for (int d = 0; d < 12; d++) h[1 + d] = o.a[2 + d];
    hints.insert(hints.end(), h, h + 13);
  }
  static const bool skipTwin = getenv("SCN_SKIP_TWIN") && atoi(getenv("SCN_SKIP_TWIN")); // developer timing experiment only: outputs stay in internal row order
  if (!skipTwin) rc = scn_metadata_build_reference_grids(m, ms, inOp->a + 1, (int)(hints.size() / 13), hints.data());
  if (rc) { scn_metadata_destroy(ms); ms = nullptr; }
  *out = ms;
  return rc;
}

// Training step i+1 prepared while step i still runs: what scn_program_run does before the first layer of an unprepared training
// step (the internally numbered Metadata with its input layer and plan hints, the reference-numbered twin on `m`), or -- where
// that step runs on `m` itself (several batch items, SCN_TRAIN_INTERNAL=0, input modes the internal numbering does not cover) --
// scn_program_prepare on `m`; either way with the rule lists of its backward pass.  Nothing here waits for the GPU work queued
// before: the builds run on the Metadata's build streams.  At most two steps are kept; a third drops the oldest (its `m` is then
// an ordinary reference-numbered Metadata, see drop_prepared).
int scn_program_prepare_training(scn_program *p, scn_metadata *m, const long *coords, int coords_on_device, long nrows, int ncols) {
  SCN_CHECK(p && m && p->nRegs > 0 && p->train, "scn_program_prepare_training needs a finished program in training mode");
  for (const auto &e : p->prepared) SCN_CHECK(e.first != m, "scn_program_prepare_training: this Metadata is prepared already");
  // (an empty Metadata is never one a pending backward pass reads: a run leaves its input layer built; the internal one is new)
  SCN_CHECK(!scn_input_layer_built(m, nullptr, nullptr), "scn_program_prepare_training needs an empty Metadata");
  const Op *inOp = input_op(p);
  SCN_CHECK(inOp, "program has no input layer");
  scn_metadata *ms = nullptr;
  if (uses_internal_numbering(p, inOp))
    SCN_TRY(start_internal(p, m, inOp, coords, coords_on_device, nrows, ncols, scn::metadata_stream(m), true, &ms));
  if (!ms) SCN_TRY(prepare_build(p, m, coords, coords_on_device, nrows, ncols, true));
  if (p->prepared.size() == 2) {
    drop_prepared(p->prepared.front());
    p->prepared.pop_front();
  }
  p->prepared.emplace_back(m, ms);
  return 0;
}

int scn_program_drop_prepared(scn_program *p) {
  SCN_CHECK(p, "null program");
  for (const auto &e : p->prepared) drop_prepared(e);
  p->prepared.clear();
  return 0;
}

// params[i] / tags[i]: device pointers of the recorded parameter tensors (and their content tags, see
// weight_tag in scn_*_convolution_forward), in the order the recorder numbered them.
int scn_program_run(scn_program *p, scn_metadata *m, const long *coords, int coords_on_device, long nrows, int ncols, const float *feats,
                    const void *const *params, const long long *tags, int n_params, void *stream, double *macs_out) {
  SCN_CHECK(p && m && p->nRegs > 0, "program not finished");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  release_regs(p, true); // outputs of the previous run
  if (p->stream && p->stream != s) SCN_CUDA(cudaStreamSynchronize(p->stream)); // slots are recycled in stream order
  p->stream = s;
  const int mode = scn_get_math_mode();
  // ---- Which Metadata do the layers run on?
  // A forward whose Metadata arrives unprepared runs on an INTERNALLY NUMBERED Metadata of its own (rows = spatial order):
  // the reference's hash-iteration order and first-touch numbering -- ~40 % of the grid-pyramid latency, all of it on the
  // critical path -- are not needed to compute anything, only to NAME the rows.  The caller's Metadata `m` is numbered beside
  // it on a worker thread (input layer + the strided convolutions that lead to the output grids: reference row ids over the
  // block structure of the internal grids, scn_metadata_build_reference_grids) and the output rows are handed out in that
  // numbering (scn_program_output_copy).  The layers' rulebooks on `m` are built on first use.  A Metadata prepared ahead
  // (scn_program_prepare) or an input mode / batch the internal numbering does not cover uses `m` for everything, as before.
  // A training step prepared ahead (scn_program_prepare_training) takes the pair built then.
  if (p->ms) { scn_metadata_destroy(p->ms); p->ms = nullptr; }
  p->internal = false;
  const Op *inOp = input_op(p);
  const bool train = p->train;
  bool preparedTrain = false;
  for (auto it = p->prepared.begin(); train && it != p->prepared.end(); ++it)
    if (it->first == m) {
      p->ms = it->second;
      p->prepared.erase(it);
      preparedTrain = true;
      ++scn::g_counters[scn::kCntTrainPrepared];
      break;
    }
  // (a prepared pair's `m` is still being numbered by its twin job: its input layer is not read here)
  const bool preparedAhead = preparedTrain || scn_input_layer_built(m, nullptr, nullptr) != 0; // its workers build everything
  scn_metadata *M = m;
  p->lastMd = train ? m : nullptr;
  p->lastRef = train ? m : nullptr;
  if (train) p->bnSave.assign(p->ops.size(), nullptr);
  if (!preparedAhead && uses_internal_numbering(p, inOp)) SCN_TRY(start_internal(p, m, inOp, coords, coords_on_device, nrows, ncols, stream, false, &p->ms));
  if (p->ms) {
    M = p->ms;
    p->internal = true;
    if (train) p->lastMd = p->ms;
  }
  if (!p->bnScratch) SCN_CUDA(cudaMalloc((void **)&p->bnScratch, 2 * scn::kBnMaxC * sizeof(float)));
  auto P = [&](long i) -> const float * { return (i < 0 || i >= n_params) ? nullptr : static_cast<const float *>(params[i]); };
  auto T = [&](long i) -> long long { return (i < 0 || i >= n_params || !tags) ? 0 : tags[i]; };
  auto alloc_reg = [&](long r, long rows, int cols, bool shadow, bool halfOnly = false) -> int {
    Reg &R = p->regs[r];
    R.rows = rows;
    R.cols = cols;
    R.pad16 = 0;
    R.p = halfOnly ? nullptr : static_cast<float *>(slot_get(p, (size_t)std::max(1l, rows * cols) * 4));
    if (halfOnly) ++scn::g_counters[scn::kCntHalfOnlyOut];
    if (!R.p && !halfOnly) return -1;
    if (shadow && scn::half_mode(mode) && cols % 32 == 0 && rows > 0) {
      R.p16 = slot_get(p, (size_t)rows * cols * 2);
      if (!R.p16) return -1;
    }
    return 0;
  };
  double macs = 0, mk = 0;
  int rc = 0;
  const size_t statsStride = (size_t)scn::kBnReplicas * 2 * scn::kFusedStatsC;
  if (p->nStats) {
    if (!p->stats) SCN_CUDA(cudaMalloc((void **)&p->stats, p->nStats * statsStride * sizeof(double)));
    SCN_CUDA(cudaMemsetAsync(p->stats, 0, p->nStats * statsStride * sizeof(double), s));
    p->statsDone.assign(p->nStats, 0);
  }
  // what a convolution op asks its launch to fold in: the lateral (a[18..20]), the statistics of the BatchNorm that reads its output
  // (a[21]) and, for a submanifold convolution of the network input, the input layer's zero-padded 16-bit rows
  auto fusion_of = [&](const Op &op) {
    scn::ConvFusion f;
    if (op.a[21] >= 0) f.stats = p->stats + op.a[21] * statsStride;
    if (op.a[18] >= 0) {
      const Reg &Y = p->regs[op.a[18]];
      f.lat = scn::Lateral{Y.p, Y.pad16 ? nullptr : Y.p16, P(op.a[19]), T(op.a[19]), (int)op.a[20], Y.rows};
    }
    const Reg &I = p->regs[op.a[0]];
    if (op.kind == K_SUBM && I.pad16) { f.pad16 = I.p16; f.padC = I.pad16; }
    return f;
  };
  // the convolution did not take the lateral (e.g. it ran on the CUDA-core path): run the 1x1x1 convolution on its own and add it
  auto lateral_fallback = [&](const Op &op, const scn::ConvFused &fused, scn_metadata *md, const long *sz, Reg &out, int Cout) -> int {
    const bool done = fused.lateral;
    if (op.a[18] < 0) return 0;
    const Reg &Y = p->regs[op.a[18]];
    macs += (double)Y.rows * (double)op.a[20] * Cout;
    if (done || out.rows == 0) return 0;
    ++scn::g_counters[scn::kCntLateralFallback];
    if (!out.p) { scn::set_error("program: lateral not folded in although the fp32 output was dropped"); return -2; }
    float *tmp = static_cast<float *>(slot_get(p, (size_t)out.rows * Cout * 4));
    if (!tmp) return -1;
    const long one[3] = {1, 1, 1};
    double mk2 = 0;
    int r = scn::submanifold_forward(md, sz, one, Y.p, tmp, P(op.a[19]), nullptr, (int)op.a[20], Cout, &mk2, Y.pad16 ? nullptr : Y.p16, T(op.a[19]), nullptr, nullptr,
                                     scn::ConvFusion(), nullptr);
    if (r == 0) r = scn_add_features(out.p, tmp, out.p, out.rows * Cout, s, out.p16);
    slot_put(p, tmp);
    return r;
  };
  static const bool firstPlanOn = !(getenv("SCN_FIRST_PLAN_HERE") && atoi(getenv("SCN_FIRST_PLAN_HERE")) == 0);
  const bool firstPlanHere = firstPlanOn && !preparedAhead;
  bool firstPlanDone = false;
  for (int i = 0; i < (int)p->ops.size() && rc == 0; i++) {
    const Op &op = p->ops[i];
    const long *a = op.a;
    switch (op.kind) {
      case K_INPUT: { // out, size[3], mode, batch hint, planes
        long nActive = 0;
        int maxActive = 0;
        if (!scn_input_layer_built(M, &nActive, &maxActive)) { // not prepared ahead (scn_program_prepare)
          rc = scn_program_prepare(p, M, coords, coords_on_device, nrows, ncols);
          if (rc == 0 && !scn_input_layer_built(M, &nActive, &maxActive)) { scn::set_error("program: no input layer"); rc = -2; }
          if (rc) break;
        }
        rc = alloc_reg(a[0], nActive, (int)a[6], false);
        p->regs[a[0]].pad16 = 0;
        const int C0 = (int)a[6], Cp = C0 < 16 ? 16 : 32;
        if (rc == 0 && nActive && scn::half_mode(mode) && a[4] != 0 && C0 % 32 != 0 && C0 < 32 && scn_tensor_core_path_available()) {
          // bf16 mode: the first convolution gathers bf16 rows zero-padded to 16 / 32 channels; written here, by the same pass
          Reg &R0 = p->regs[a[0]];
          R0.p16 = slot_get(p, (size_t)nActive * Cp * 2);
          if (!R0.p16) { rc = -1; break; }
          R0.pad16 = Cp;
          rc = scn_input_layer_forward_padded_bf16(M, feats, R0.p, R0.p16, C0, Cp);
        } else if (rc == 0 && nActive) rc = scn_input_layer_forward(M, feats, p->regs[a[0]].p, (int)a[6]);
        break;
      }
      case K_SUBM: case K_CONV: case K_DECONV: { // in, out, then subm: size[3], filter[3], w, bias, Cin, Cout; (de)conv: inS[3], outS[3], f[3], s[3], w, bias, Cin, Cout
        const bool subm = op.kind == K_SUBM;
        long n = 0;
        if (subm && firstPlanHere && !firstPlanDone) { // the first plan of an unprepared forward: built here, now (see build_subm_on_caller)
          firstPlanDone = true;
          rc = scn::build_subm_on_caller(M, a + 2, a + 5);
          if (rc) break;
        }
        if (op.kind == K_CONV) rc = scn_convolution_prepare(M, a + 2, a + 5, a + 8, a + 11, &n, nullptr);
        else rc = scn_get_nactive(M, subm ? a + 2 : a + 5, &n);
        const int Cout = (int)(subm ? a[11] : a[17]);
        const bool half = !train && a[23] == 1 && scn::half_mode(mode) && n >= kHalfOnlyRows && scn_tensor_core_path_available();
        if (rc == 0) rc = alloc_reg(a[1], n, Cout, half || a[22] >= 0 || a[18] >= 0, half);
        const Reg &I = p->regs[a[0]], &O = p->regs[a[1]];
        const void *in16 = I.pad16 ? nullptr : I.p16;
        const float *add = a[22] >= 0 ? p->regs[a[22]].p : nullptr;
        scn::ConvFused fused;
        if (rc == 0 && subm)
          rc = scn::submanifold_forward(M, a + 2, a + 5, I.p, O.p, P(a[8]), P(a[9]), (int)a[10], Cout, &mk, in16, T(a[8]), add, O.p16, fusion_of(op), &fused);
        else if (rc == 0)
          rc = (op.kind == K_CONV ? scn::convolution_forward : scn::deconvolution_forward)(M, a + 2, a + 5, a + 8, a + 11, I.p, O.p, P(a[14]), P(a[15]), (int)a[16], Cout,
                                                                                            &mk, in16, T(a[14]), add, O.p16, fusion_of(op), &fused);
        if (a[21] >= 0) p->statsDone[a[21]] = fused.stats;
        if (rc == 0) rc = lateral_fallback(op, fused, M, subm ? a + 2 : a + 5, p->regs[a[1]], Cout);
        macs += mk;
        break;
      }
      case K_BN: { // in, out, C, weight, bias, running mean, running var, mode; f: eps, momentum, leakiness
        const Reg &I = p->regs[a[0]];
        const bool fromSums = a[21] >= 0 && p->statsDone[a[21]] && I.rows > 0;
        // (training too: the backward pass reads the leaky-ReLU mask from the bf16 copy, and the consuming convolutions' weight-gradient
        // kernels gather from it)
        static int trainHalf = -1;
        if (trainHalf < 0) trainHalf = getenv("SCN_TRAIN_HALF_BN") ? atoi(getenv("SCN_TRAIN_HALF_BN")) : 1;
        const bool halfOnly = (!train || trainHalf) && fromSums && a[19] == 1 && scn::half_mode(mode) && scn_tensor_core_path_available();
        rc = alloc_reg(a[1], I.rows, (int)a[2], true, halfOnly);
        float *saveM = p->bnScratch, *saveI = p->bnScratch + scn::kBnMaxC;
        if (rc == 0 && train) { // kept for the backward pass
          p->bnSave[i] = static_cast<float *>(slot_get(p, (size_t)2 * a[2] * 4));
          if (!p->bnSave[i]) { rc = -1; break; }
          saveM = p->bnSave[i];
          saveI = saveM + a[2];
        }
        if (rc == 0 && fromSums) {
          ++scn::g_counters[scn::kCntBnFromSums];
          rc = scn::bn_forward_from_sums(I.p, p->regs[a[1]].p, I.rows, (int)a[2], p->stats + a[21] * statsStride, saveM, saveI,
                                         const_cast<float *>(P(a[5])), const_cast<float *>(P(a[6])), P(a[3]), P(a[4]), (float)op.f[0], (float)op.f[1], (int)a[7],
                                         (float)op.f[2], s, p->regs[a[1]].p16);
          break;
        }
        if (rc == 0)
          rc = scn_batchnorm_forward(I.p, p->regs[a[1]].p, I.rows, (int)a[2], saveM, saveI, const_cast<float *>(P(a[5])),
                                     const_cast<float *>(P(a[6])), P(a[3]), P(a[4]), (float)op.f[0], (float)op.f[1], (int)a[7], (float)op.f[2], s, p->regs[a[1]].p16);
        break;
      }
      case K_ADD: { // a, b, out
        const Reg &A = p->regs[a[0]], &B = p->regs[a[1]];
        if (A.rows != B.rows || A.cols != B.cols) { scn::set_error("program: add of differently shaped feature matrices"); rc = -2; break; }
        rc = alloc_reg(a[2], A.rows, A.cols, true);
        if (rc == 0 && A.rows) rc = scn_add_features(A.p, B.p, p->regs[a[2]].p, A.rows * A.cols, s, p->regs[a[2]].p16);
        break;
      }
    }
    if (rc) break;
    scn::timeline_mark("main", op.kind, a[2], p->regs[a[op.kind == K_ADD ? 2 : (op.kind == K_INPUT ? 0 : 1)]].rows);
    for (int r = 0; !train && r < p->nRegs; r++) // free what this op used last (stream-ordered: safe right after the launch)
      if (p->lastUse[r] == i && !p->isOutput[r]) {
        Reg &R = p->regs[r];
        if (R.p) { slot_put(p, R.p); R.p = nullptr; }
        if (R.p16) { slot_put(p, R.p16); R.p16 = nullptr; }
      }
  }
  if (rc) {
    release_regs(p, true);
    if (p->internal) scn_metadata_wait_jobs(m); // the twin reads p->ms, which the next run destroys
    return rc;
  }
  if (macs_out) *macs_out = macs;
  if (p->internal) SCN_TRY(scn_metadata_wait_jobs(m)); // the reference-numbered grids of the outputs
  cudaEvent_t &ev = p->evEnd[p->nRuns & 1];
  if (!ev) SCN_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  SCN_CUDA(cudaEventRecord(ev, s));
  p->nRuns++;
  return 0;
}

// The backward pass of the last TRAINING run (scn_program_set_training), op by op in reverse: the same native backward entries
// the layer-by-layer autograd Functions call (scn_*_convolution_backward, scn_batchnorm_backward, NetworkInNetwork backward for a
// folded lateral), driven from C++ instead of ~100 Python autograd nodes.  d_out[i]: gradient of output register out_regs[i]
// ([rows][cols] float32, device; not modified).  param_grads[j]: device buffer of parameter j's gradient (overwritten) or NULL
// (not wanted).  param_live[j] = 1 when parameter j received a gradient: ops whose output reaches no program output (the dead
// top-down levels of the FPN, SURVEY.md App. D.2) are skipped, as autograd skips them.  d_features: NULL or the gradient of the
// network input [nIn rows][planes].
int scn_program_backward(scn_program *p, int n_out, const int *out_regs, const float *const *d_out, const void *const *params, void *const *param_grads,
                         int n_params, float *d_features, int *param_live, void *const *param_events) {
  SCN_CHECK(p && p->train && p->lastMd && p->nRegs > 0, "scn_program_backward needs a preceding training run of this program");
  scn_metadata *m = p->lastMd;
  cudaStream_t s = p->stream;
  auto P = [&](long i) -> const float * { return (i < 0 || i >= n_params) ? nullptr : static_cast<const float *>(params[i]); };
  auto G = [&](long i) -> float * { return (i < 0 || i >= n_params) ? nullptr : static_cast<float *>(param_grads[i]); };
  std::vector<char> live(std::max(1, n_params), 0);
  int rc = 0;
  auto mark = [&](long i) -> int {
    if (i < 0 || i >= n_params || !param_grads[i]) return 0;
    if (live[i]) { scn::set_error("program backward: a parameter is used by more than one op (not supported by the replayed training step)"); return -2; }
    live[i] = 1;
    return 0;
  };
  // param_events[j] (optional, cudaEvent_t): recorded on the stream right after the kernels that write parameter j's gradient are
  // queued -- a data-parallel caller starts the all-reduce of a gradient bucket behind the event of its last parameter while the
  // backward pass of the earlier layers is still running
  auto done = [&](long i) {
    if (param_events && i >= 0 && i < n_params && param_events[i]) cudaEventRecord(static_cast<cudaEvent_t>(param_events[i]), s);
  };
  std::vector<float *> g(p->nRegs, nullptr);
  auto elems = [&](long r) -> long { return p->regs[r].rows * (long)p->regs[r].cols; };
  // adds `src` to the gradient of register r (first contribution: copy; `owned`: src is a slot buffer that may be adopted)
  auto contribute = [&](long r, float *src, bool owned) -> int {
    const long n = elems(r);
    if (n == 0) { if (owned) slot_put(p, src); return 0; }
    if (!g[r]) {
      if (owned) { g[r] = src; return 0; }
      g[r] = static_cast<float *>(slot_get(p, (size_t)n * 4));
      if (!g[r]) return -1;
      SCN_CUDA(cudaMemcpyAsync(g[r], src, (size_t)n * 4, cudaMemcpyDeviceToDevice, s));
      return 0;
    }
    int r2 = scn_add_features(g[r], src, g[r], n, s, nullptr);
    if (owned) slot_put(p, src);
    return r2;
  };
  for (int i = 0; i < n_out; i++) {
    SCN_CHECK(out_regs[i] >= 0 && out_regs[i] < p->nRegs && p->isOutput[out_regs[i]], "not an output register");
    if (!d_out[i]) continue;
    const long r = out_regs[i];
    if (p->internal && elems(r) > 0) { // the run was numbered internally: bring the gradient rows from the caller's (reference) order into it
      SCN_CHECK(p->ms == m && p->lastRef, "program backward: the internally numbered Metadata of the run is gone");
      float *gi = static_cast<float *>(slot_get(p, (size_t)elems(r) * 4));
      if (!gi) return -1;
      SCN_TRY(scn_rows_from_reference_order(p->lastRef, p->ms, p->outSize[r].data(), d_out[i], gi, p->regs[r].cols));
      SCN_TRY(contribute(r, gi, true));
    } else
      SCN_TRY(contribute(r, const_cast<float *>(d_out[i]), false));
  }
  for (int i = (int)p->ops.size() - 1; i >= 0 && rc == 0; i--) {
    const Op &op = p->ops[i];
    const long *a = op.a;
    const long outReg = op.kind == K_INPUT ? a[0] : (op.kind == K_ADD ? a[2] : a[1]);
    float *dy = g[outReg];
    if (!dy) continue; // nothing downstream of this op reaches an output
    switch (op.kind) {
      case K_INPUT:
        if (d_features) rc = scn_input_layer_backward(m, d_features, dy, (int)a[6]);
        break;
      case K_ADD:
        rc = contribute(a[0], dy, false);
        if (rc == 0) rc = contribute(a[1], dy, false);
        break;
      case K_BN: {
        const Reg &X = p->regs[a[0]], &Y = p->regs[a[1]];
        if (X.rows == 0) break;
        SCN_CHECK(X.p && (Y.p || Y.p16) && p->bnSave[i], "program backward: BatchNorm activations were not kept");
        float *dx = static_cast<float *>(slot_get(p, (size_t)elems(a[0]) * 4));
        if (!dx) { rc = -1; break; }
        if ((rc = mark(a[3])) || (rc = mark(a[4]))) break;
        rc = scn::batchnorm_backward_y16(X.p, dx, Y.p, Y.p ? nullptr : Y.p16, dy, X.rows, (int)a[2], p->bnSave[i], p->bnSave[i] + a[2], P(a[3]), G(a[3]), G(a[4]), (float)op.f[2], s);
        done(a[3]); done(a[4]);
        if (rc == 0) rc = contribute(a[0], dx, true);
        break;
      }
      default: { // the three convolution kinds
        const Reg &I = p->regs[a[0]];
        const int Cin = (int)(op.kind == K_SUBM ? a[10] : a[16]), Cout = (int)(op.kind == K_SUBM ? a[11] : a[17]);
        const long wi = op.kind == K_SUBM ? a[8] : a[14], bi = op.kind == K_SUBM ? a[9] : a[15];
        if (a[22] >= 0 && (rc = contribute(a[22], dy, false))) break;       // addend fused into the epilogue: out = conv + other
        if (a[18] >= 0) {                                                   // folded lateral: out += Y @ W_lat
          const Reg &Y = p->regs[a[18]];
          const int Cl = (int)a[20];
          if (Y.rows > 0) {
            float *dl = static_cast<float *>(slot_get(p, (size_t)Y.rows * Cl * 4));
            if (!dl) { rc = -1; break; }
            if ((rc = mark(a[19]))) break;
            rc = scn_network_in_network_backward_input(dl, dy, P(a[19]), Y.rows, Cl, Cout, s);
            if (rc == 0 && G(a[19])) rc = scn_network_in_network_backward_params(Y.p, dy, G(a[19]), nullptr, Y.rows, Cl, Cout, s);
            done(a[19]);
            if (rc == 0) rc = contribute(a[18], dl, true);
            if (rc) break;
          }
        }
        if (I.rows == 0 || p->regs[outReg].rows == 0) break;
        SCN_CHECK(I.p || (I.p16 && !I.pad16 && Cin % 32 == 0 && scn::half_mode(scn_get_math_mode())), "program backward: convolution input was not kept");
        if ((rc = mark(wi)) || (rc = mark(bi))) break;
        // the gradient of the network input is only computed on request (App. D.13)
        bool inputIsNetworkInput = false;
        for (const Op &o : p->ops) if (o.kind == K_INPUT && o.a[0] == a[0]) inputIsNetworkInput = true;
        const bool wantDIn = !(inputIsNetworkInput && !d_features) || op.kind != K_SUBM;
        float *din = wantDIn ? static_cast<float *>(slot_get(p, (size_t)elems(a[0]) * 4)) : nullptr;
        if (wantDIn && !din) { rc = -1; break; }
        float *dw = G(wi);
        float *dwTmp = nullptr;
        if (!dw) { // gradient not wanted: the entry still needs a buffer
          long K = 1;
          for (int d = 0; d < 3; d++) K *= op.kind == K_SUBM ? a[5 + d] : a[8 + d];
          dwTmp = static_cast<float *>(slot_get(p, (size_t)K * Cin * Cout * 4));
          if (!dwTmp) { rc = -1; break; }
          dw = dwTmp;
        }
        // bf16 mode: the forward pass left a bf16 copy of the input rows (same layout: whole rows, no padding) -- the
        // weight-gradient kernel gathers from it instead of converting the fp32 rows again
        const void *in16 = I.p16 && !I.pad16 && Cin % 32 == 0 && scn::half_mode(scn_get_math_mode()) ? I.p16 : nullptr;
        const float *inRows = I.p;
        float *inTmp = nullptr;
        if (!inRows) { // the forward pass kept only the bf16 copy of these rows (a BatchNorm output read by tensor-core convolutions alone)
          long Kv = 1;
          for (int d = 0; d < 3; d++) Kv *= op.kind == K_SUBM ? a[5 + d] : a[8 + d];
          if (!scn::dw_tc_ok(Cin, Cout, (int)Kv, scn_get_math_mode())) { // the CUDA-core weight-gradient kernel reads fp32 rows: widen the copy (exact)
            inTmp = static_cast<float *>(slot_get(p, (size_t)elems(a[0]) * 4));
            if (!inTmp) { rc = -1; break; }
            if ((rc = scn::from_16(I.p16, inTmp, elems(a[0]), s))) break;
            inRows = inTmp;
          }
        }
        if (op.kind == K_SUBM) rc = scn::submanifold_backward(m, a + 2, a + 5, inRows, din, dy, P(wi), dw, G(bi), Cin, Cout, in16);
        else rc = (op.kind == K_CONV ? scn::convolution_backward : scn::deconvolution_backward)(m, a + 2, a + 5, a + 8, a + 11, inRows, din, dy, P(wi), dw, G(bi), Cin, Cout, in16);
        if (dwTmp) slot_put(p, dwTmp);
        if (inTmp) slot_put(p, inTmp);
        done(wi); done(bi);
        if (rc == 0 && din) rc = contribute(a[0], din, true);
        break;
      }
    }
    if (rc) break;
    slot_put(p, dy); // consumed (stream-ordered: the kernels above were queued before any later user of the slot)
    g[outReg] = nullptr;
  }
  for (float *&q : g) if (q) { slot_put(p, q); q = nullptr; }
  if (rc) return rc;
  if (param_live) for (int j = 0; j < n_params; j++) param_live[j] = live[j];
  ++scn::g_counters[scn::kCntTrainReplay];
  return 0;
}

int scn_copy_device(void *dst, const void *src, long bytes, void *stream) {
  if (bytes > 0) SCN_CUDA(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return 0;
}
// Copies an output register into caller memory (device, on the run's stream) in the row order of `m`: a plain copy, or --
// when the run used the internal numbering -- the rows gathered into the reference numbering.
int scn_program_output_copy(scn_program *p, scn_metadata *m, int reg, const long spatial_size[3], float *dst) {
  SCN_CHECK(p && reg >= 0 && reg < p->nRegs && p->isOutput[reg], "not an output register");
  const Reg &R = p->regs[reg];
  if (R.rows == 0) return 0;
  static const bool skipTwin = getenv("SCN_SKIP_TWIN") && atoi(getenv("SCN_SKIP_TWIN"));
  if (p->internal && !skipTwin) return scn_rows_to_reference_order(m, p->ms, spatial_size, R.p, dst, R.cols);
  return scn_copy_device(dst, R.p, R.rows * R.cols * 4, p->stream);
}
// All output registers at once (regs[i] -> dst[i], grids sizes[3 i .. 3 i + 2]): one gather launch instead of two per map.
int scn_program_outputs_copy(scn_program *p, scn_metadata *m, int n, const int *regs, const long *sizes, float *const *dst) {
  SCN_CHECK(p && n >= 0 && n <= 8, "at most 8 output registers per call");
  static const bool skipTwin = getenv("SCN_SKIP_TWIN") && atoi(getenv("SCN_SKIP_TWIN"));
  static const bool multi = !(getenv("SCN_OUT_MULTI") && atoi(getenv("SCN_OUT_MULTI")) == 0);
  if (!(p->internal && !skipTwin && multi)) {
    for (int i = 0; i < n; i++) SCN_TRY(scn_program_output_copy(p, m, regs[i], sizes + 3 * i, dst[i]));
    return 0;
  }
  const float *src[8];
  int cols[8];
  for (int i = 0; i < n; i++) {
    SCN_CHECK(regs[i] >= 0 && regs[i] < p->nRegs && p->isOutput[regs[i]], "not an output register");
    src[i] = p->regs[regs[i]].p;
    cols[i] = p->regs[regs[i]].cols;
  }
  return scn_rows_to_reference_order_multi(m, p->ms, n, sizes, src, dst, cols);
}
int scn_program_output(scn_program *p, int reg, long *rows, int *cols, const float **ptr) {
  SCN_CHECK(p && reg >= 0 && reg < p->nRegs && p->isOutput[reg], "not an output register");
  *rows = p->regs[reg].rows;
  *cols = p->regs[reg].cols;
  *ptr = p->regs[reg].p;
  return 0;
}
}
