// engine.cu — C-ABI implementation (include/ppsci_b200.h): plan validation, workspace carving
// and the per-chunk launch schedule
//     forward jets (layer by layer)  ->  residual program + MSE  ->  adjoint (dW, dx per layer).
// All device memory except the (tiny) residual program is caller-owned workspace.
#ifdef PPSCI_EMUL
#include "cuda_emul.h"
#endif

#include <stdio.h>
#include <stdlib.h>

#include <string>
#include <vector>

#include "kernels_simt.cuh"
#include "kernels_tc.cuh"
#include "kernels_tc2.cuh"
#include "kernels_fused.cuh"
#include "kernels_thin.cuh"
#include "kernels_gate.cuh"

using namespace ppsci;

static thread_local std::string g_err;

static int fail(const std::string& msg) {
  g_err = msg;
  return 1;
}

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(std::string(#call) + " failed: " + cudaGetErrorString(e_) + " (" __FILE__ ":" + \
                  std::to_string(__LINE__) + ")");                                            \
  } while (0)

struct ppsci_plan {
  ppsci_plan_spec spec;
  std::vector<int32_t> prog, grad_res, grad_in, grad_reg;
  std::vector<double> consts;
  int C = 1;
  int kmax = 1;
  JetLayout J;
  int64_t w_off[PPSCI_MAX_LAYERS + 1];
  int64_t b_off[PPSCI_MAX_LAYERS + 1];
  int ld[PPSCI_MAX_LAYERS + 1];
  int64_t n_params = 0;
  int64_t gate_w_off[2] = {0, 0};  // gated plans: embed_u / embed_v weights and biases behind the layers
  int64_t gate_b_off[2] = {0, 0};
  int64_t alpha_off = 0;  // gated == 2: one residual weight per block behind the embeddings
  // trainable activation parameters (PPSCI_ACT_STAN: one beta per unit; PPSCI_ACT_SWISH_B: one per layer) of hidden
  // layer l, behind everything else; actp_stride 1 / 0, actp_off[l] < 0: layer l's activation has none
  int64_t actp_off[PPSCI_MAX_LAYERS + 1];
  int actp_stride = 0;
  int ld_hidden_max = 4;
  int chunk = 0;
  int num_sms = 148;
  bool use_tc = false;
  // bit0 forward, bit1 dx, bit2 dW on the tensor cores; bit3 / bit4 / bit5: CTA-pair forward / dx / dW kernels;
  // bit6: layer-fused forward (kernels_fused.cuh).  PPSCI_B200_TC_MASK selects subsets (debugging / cross-checks).
  // bit7: layer-fused dx chain.  bit8: tf32 fused forward also for layers wider than 128.  bit9: fp16 fused forward also for narrow layers.
  int tc_mask = 255;
  // device copies of the residual program
  int* d_prog = nullptr;
  double* d_consts = nullptr;
  int* d_grad_res = nullptr;
  int* d_grad_in = nullptr;
  int* d_grad_reg = nullptr;
  double* aux_grad[PPSCI_MAX_IN] = {};  // ppsci_b200_plan_set_aux_grad
  int64_t launches = 0;
  bool attrs_set = false;
  // optional per-kernel-class timing (bench only; adds event records, no syncs)
  bool profile = false;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  std::vector<int> ev_cls;  // class of event pair i (events 2i, 2i+1)
};

enum { CLS_FWD = 0, CLS_HEAD = 1, CLS_DW = 2, CLS_DX = 3, CLS_MISC = 4, CLS_THIN_FWD = 5, CLS_THIN_DX = 6, CLS_THIN_DW = 7, CLS_COUNT = 8 };

struct ProfScope {
  ppsci_plan* P;
  cudaStream_t st;
  bool on;
  ProfScope(ppsci_plan* P_, int cls, cudaStream_t st_) : P(P_), st(st_), on(P_->profile) {
    if (!on) return;
    if (P->ev_used + 2 > P->ev_pool.size()) {
      for (int i = 0; i < 64; ++i) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) { on = false; return; }
        P->ev_pool.push_back(e);
      }
    }
    P->ev_cls.push_back(cls);
    cudaEventRecord(P->ev_pool[P->ev_used], st);
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(P->ev_pool[P->ev_used + 1], st);
    P->ev_used += 2;
  }
};

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline int round4(int x) { return (x + 3) / 4 * 4; }

struct Carve {
  size_t z[PPSCI_MAX_LAYERS + 1];  // z[l] for l = 1..n_layers-1 (hidden pre-activations)
  size_t a[PPSCI_MAX_LAYERS + 1];  // a[l] = act_jets(z[l]) stashed by the tcgen05 forward for the dW kernel
  size_t y, ybar, zbar0, zbar1;
  size_t zb[PPSCI_MAX_LAYERS + 1];  // zb[l] = Zbar_l, one buffer per hidden layer (fused dx chain: every Zbar_l outlives the chain)
  size_t wt[PPSCI_MAX_LAYERS + 1];
  size_t loss_acc;
  size_t tc;  // scratch of the tcgen05 backend
  size_t w16;  // fp16 hi / lo weight images of the fused forward's layers 2.. (+ per-layer |W|max and scale words)
  // gated plans (ModifiedMLP): gated jets G_l per hidden layer, pre-activations of embed_u / embed_v and their adjoints
  size_t gt[PPSCI_MAX_LAYERS + 1];
  size_t zu, zv, zub, zvb;
  size_t xres, wtu, wtv;  // gated == 2: adjoint carried by the blocks' residual path; transposed embedding weights
  size_t total;
};

static size_t tc_scratch_bytes(const ppsci_plan* P, int64_t nc);
static bool tc_astash_needed(const ppsci_plan* P, int l);
static bool fused_fwd_ok(const ppsci_plan* P);
static bool fused_dx_ok(const ppsci_plan* P);
static bool fused_fwd16_ok(const ppsci_plan* P);

// gated plans: 1 when layer 1 is an embedding layer whose stored output feeds the embed_u / embed_v layers and the
// first gated layer (PirateNet always; ModifiedMLP with a Fourier embedding, act_first >= 0), 0 when they read the seeds
static inline int gate_emb(const ppsci_plan_spec& s) { return (s.gated == 2 || (s.gated == 1 && s.act_first >= 0)) ? 1 : 0; }

static void carve(const ppsci_plan* P, int64_t nc, Carve* cv) {
  const size_t es = P->spec.dtype == PPSCI_F64 ? 8 : 4;
  const int L = P->spec.n_layers;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + bytes, 256);
    return o;
  };
  for (int l = 1; l < L; ++l) cv->z[l] = take((size_t)P->C * nc * P->ld[l] * es);
  cv->y = take((size_t)P->C * nc * P->ld[L] * es);
  cv->ybar = take((size_t)P->C * nc * P->ld[L] * es);
  const bool fdx = fused_dx_ok(P);
  cv->zbar0 = take(fdx ? 0 : (size_t)P->C * nc * P->ld_hidden_max * es);
  cv->zbar1 = take(fdx ? 0 : (size_t)P->C * nc * P->ld_hidden_max * es);
  for (int l = 1; l < L; ++l) cv->zb[l] = take(fdx ? (size_t)P->C * nc * P->ld[l] * es : 0);
  for (int l = 2; l <= L; ++l) cv->wt[l] = take((size_t)P->spec.widths[l] * P->spec.widths[l - 1] * es);
  cv->loss_acc = take(PPSCI_MAX_RES * sizeof(double));
  cv->tc = take(tc_scratch_bytes(P, nc));
  cv->w16 = take(fused_fwd16_ok(P) ? (size_t)(L - 3 > 0 ? L - 3 : 0) * P->spec.widths[1] * P->spec.widths[1] * 4 + 16 * PPSCI_MAX_LAYERS : 0);
  for (int l = 1; l < L; ++l) cv->a[l] = take(tc_astash_needed(P, l) ? (size_t)P->C * nc * P->ld[l] * es : 0);
  const bool gated = P->spec.gated != 0;
  for (int l = 1; l < L; ++l) cv->gt[l] = take(gated ? (size_t)P->C * nc * P->ld[l] * es : 0);
  const int emb = gate_emb(P->spec);
  const int lg = (gated && emb + 1 <= L) ? emb + 1 : 1;  // first gated layer
  cv->zu = take(gated ? (size_t)P->C * nc * P->ld[lg] * es : 0);
  cv->zv = take(gated ? (size_t)P->C * nc * P->ld[lg] * es : 0);
  cv->zub = take(gated ? (size_t)P->C * nc * P->ld[lg] * es : 0);
  cv->zvb = take(gated ? (size_t)P->C * nc * P->ld[lg] * es : 0);
  const bool pirate = P->spec.gated == 2;
  cv->xres = take(pirate ? (size_t)P->C * nc * P->ld[1] * es : 0);
  cv->wtu = take(gated && emb ? (size_t)P->spec.widths[1] * P->spec.widths[lg] * es : 0);
  cv->wtv = take(gated && emb ? (size_t)P->spec.widths[1] * P->spec.widths[lg] * es : 0);
  cv->total = off;
}

extern "C" const char* ppsci_b200_last_error(void) { return g_err.c_str(); }
extern "C" const char* ppsci_b200_version(void) {
#ifdef PPSCI_EMUL
  return "ppsci_b200 0.1 (CPU emulation build: TEST ONLY)";
#else
  return "ppsci_b200 0.1 (sm_100a)";
#endif
}

static int op_arity(int op) {
  switch (op) {
    case PPSCI_OP_CONST: return 0;
    case PPSCI_OP_MOV: case PPSCI_OP_NEG: case PPSCI_OP_POWI: case PPSCI_OP_SIN: case PPSCI_OP_COS:
    case PPSCI_OP_TANH: case PPSCI_OP_EXP: case PPSCI_OP_LOG: case PPSCI_OP_SQRT: case PPSCI_OP_ABS:
    case PPSCI_OP_SIGN: case PPSCI_OP_SINH: case PPSCI_OP_COSH: case PPSCI_OP_HEAVISIDE:
      return 1;
    case PPSCI_OP_ADD: case PPSCI_OP_SUB: case PPSCI_OP_MUL: case PPSCI_OP_DIV: case PPSCI_OP_POW:
    case PPSCI_OP_MAX: case PPSCI_OP_MIN: case PPSCI_OP_FMA:
      return 2;
    default: return -1;
  }
}

extern "C" int ppsci_b200_plan_create(const ppsci_plan_spec* s, ppsci_plan** out) {
  if (!s || !out) return fail("plan_create: null argument");
  *out = nullptr;
  if (s->dtype != PPSCI_F32 && s->dtype != PPSCI_F64) return fail("plan_create: dtype must be f32 or f64");
  if (s->n_in < 1 || s->n_in > PPSCI_MAX_IN) return fail("plan_create: n_in out of range");
  if (s->dense_in) {  // dense [n_points][n_feat] first-layer operand (header: dense_in)
    if (s->n_in != 1) return fail("plan_create: dense_in needs n_in == 1 (one row-major matrix)");
    if (s->n_dir != 0) return fail("plan_create: dense_in has no input derivatives (n_dir must be 0)");
    if (s->n_feat < 1 || s->n_feat > 4096) return fail("plan_create: n_feat out of range");
  } else if (s->n_feat < 1 || s->n_feat > PPSCI_MAX_FEAT) {
    return fail("plan_create: n_feat out of range");
  }
  if (s->n_layers < 1 || s->n_layers > PPSCI_MAX_LAYERS) return fail("plan_create: n_layers out of range");
  if (s->widths[0] != s->n_feat) return fail("plan_create: widths[0] must equal n_feat");
  for (int l = 0; l <= s->n_layers; ++l)
    if (s->widths[l] < 1 || s->widths[l] > 4096) return fail("plan_create: layer width out of range");
  if (s->act < 0 || s->act > PPSCI_ACT_LAST) return fail("plan_create: unknown activation");
  if (s->act_first < -1 || s->act_first > PPSCI_ACT_LAST) return fail("plan_create: unknown first-layer activation");
  for (int f = 0; f < (s->dense_in ? 0 : s->n_feat); ++f) {
    if (s->feat_src[f] < 0 || s->feat_src[f] >= s->n_in) return fail("plan_create: feat_src out of range");
    if (s->feat_kind[f] < 0 || s->feat_kind[f] > PPSCI_FEAT_SIN) return fail("plan_create: bad feat_kind");
  }
  if (s->n_dir < 0 || s->n_dir > PPSCI_MAX_DIR) return fail("plan_create: n_dir out of range");
  if (s->act_first == PPSCI_ACT_STAN || s->act_first == PPSCI_ACT_SWISH_B)
    return fail("plan_create: act_first cannot be an activation with a trainable parameter");
  if ((s->act == PPSCI_ACT_STAN || s->act == PPSCI_ACT_SWISH_B) && (s->gated || s->backend == 2))
    return fail("plan_create: activations with a trainable parameter (stan, swish) run on plain MLP plans, CUDA-core kernels");
  if (s->gated) {  // ModifiedMLP: the gate multiplies every hidden layer's output with the (same-width) embeddings
    if (s->n_layers < 2) return fail("plan_create: a gated network needs at least one hidden layer");
    if (s->gated != 1 && s->gated != 2) return fail("plan_create: gated must be 0, 1 (ModifiedMLP) or 2 (PirateNet)");
    if (s->dense_in) return fail("plan_create: gated networks do not take dense_in");
    if (s->gated == 2 && (s->n_layers < 5 || (s->n_layers - 2) % 3 != 0))
      return fail("plan_create: gated kind 2 needs 1 embedding layer + 3 layers per block + the output layer");
    const int emb = gate_emb(*s);
    if (s->n_layers < emb + 2) return fail("plan_create: a gated network needs a hidden layer behind its embedding layer");
    for (int l = emb + 2; l < s->n_layers; ++l)
      if (s->widths[l] != s->widths[emb + 1]) return fail("plan_create: a gated network needs equal hidden widths");
    if (s->gated == 2 && s->widths[1] != s->widths[2])
      return fail("plan_create: gated kind 2 adds a block's input to its output: the embedding layer needs the blocks' width");
    if (s->backend == 2) return fail("plan_create: gated networks run on the CUDA-core kernels (backend 0 or 1)");
  }
  int C = 1, kmax = 1;
  for (int d = 0; d < s->n_dir; ++d) {
    if (s->dir_order[d] < 1 || s->dir_order[d] > PPSCI_MAX_ORDER) return fail("plan_create: dir_order out of range");
    C += s->dir_order[d];
    if (s->dir_order[d] > kmax) kmax = s->dir_order[d];
  }
  if (C > RC) return fail("plan_create: too many jet channels (max 32)");
  const int n_out = s->widths[s->n_layers];
  if (s->n_aux < 0 || s->n_aux > PPSCI_MAX_IN) return fail("plan_create: n_aux out of range");
  const int n_inreg = C * n_out + s->n_in + s->n_aux;
  if (s->n_reg < n_inreg || s->n_reg > PPSCI_MAX_REG) return fail("plan_create: n_reg out of range (max 256)");
  if (s->n_res < 0 || s->n_res > PPSCI_MAX_RES) return fail("plan_create: n_res out of range");
  if (s->n_ops < 0 || (s->n_ops > 0 && !s->prog)) return fail("plan_create: bad program");
  for (int i = 0; i < s->n_ops; ++i) {
    const int op = s->prog[4 * i], dst = s->prog[4 * i + 1], a = s->prog[4 * i + 2], b = s->prog[4 * i + 3];
    const int ar = op_arity(op);
    if (ar < 0) return fail("plan_create: unknown opcode at op " + std::to_string(i));
    if (dst < 0 || dst >= s->n_reg) return fail("plan_create: dst register out of range at op " + std::to_string(i));
    if (op == PPSCI_OP_CONST) {
      if (a < 0 || a >= s->n_consts) return fail("plan_create: const index out of range at op " + std::to_string(i));
    } else {
      if (a < 0 || a >= s->n_reg) return fail("plan_create: src register out of range at op " + std::to_string(i));
      if (ar == 2 && (b < 0 || b >= s->n_reg)) return fail("plan_create: src register out of range at op " + std::to_string(i));
    }
  }
  for (int k = 0; k < s->n_res; ++k) {
    if (s->res_reg[k] < 0 || s->res_reg[k] >= s->n_reg) return fail("plan_create: res_reg out of range");
    if (s->reduction[k] != PPSCI_REDUCE_MEAN && s->reduction[k] != PPSCI_REDUCE_SUM) return fail("plan_create: bad reduction");
  }
  if (s->n_grad < 0) return fail("plan_create: n_grad < 0");
  for (int g = 0; g < s->n_grad; ++g) {
    if (s->grad_res[g] < 0 || s->grad_res[g] >= s->n_res) return fail("plan_create: grad_res out of range");
    if (s->grad_in[g] < 0 || s->grad_in[g] >= C * n_out) return fail("plan_create: grad_in out of range");
    if (s->grad_reg[g] < 0 || s->grad_reg[g] >= s->n_reg) return fail("plan_create: grad_reg out of range");
    if (g > 0 && s->grad_in[g] < s->grad_in[g - 1]) return fail("plan_create: grad list must be sorted by grad_in");
  }
  if (s->n_pgrad < 0 || s->n_pgrad > PPSCI_MAX_PGRAD) return fail("plan_create: n_pgrad out of range");
  for (int g = 0; g < s->n_pgrad; ++g) {
    if (s->pgrad_res[g] < 0 || s->pgrad_res[g] >= s->n_res) return fail("plan_create: pgrad_res out of range");
    if (s->pgrad_aux[g] < 0 || s->pgrad_aux[g] >= s->n_aux || !s->aux_bcast[s->pgrad_aux[g]])
      return fail("plan_create: pgrad_aux must name a learnable (aux_bcast) parameter");
    if (s->pgrad_reg[g] < 0 || s->pgrad_reg[g] >= s->n_reg) return fail("plan_create: pgrad_reg out of range");
  }

  ppsci_plan* P = new ppsci_plan();
  P->spec = *s;
  P->prog.assign(s->prog, s->prog + 4 * (size_t)s->n_ops);
  P->consts.assign(s->consts, s->consts + (size_t)s->n_consts);
  P->grad_res.assign(s->grad_res, s->grad_res + (size_t)s->n_grad);
  P->grad_in.assign(s->grad_in, s->grad_in + (size_t)s->n_grad);
  P->grad_reg.assign(s->grad_reg, s->grad_reg + (size_t)s->n_grad);
  P->spec.prog = nullptr; P->spec.consts = nullptr;
  P->spec.grad_res = P->spec.grad_in = P->spec.grad_reg = nullptr;
  P->C = C;
  P->kmax = kmax;
  P->J.C = C;
  P->J.n_dir = s->n_dir;
  int base = 1;
  for (int d = 0; d < PPSCI_MAX_DIR; ++d) {
    P->J.dir_order[d] = d < s->n_dir ? s->dir_order[d] : 0;
    P->J.dir_base[d] = base;
    if (d < s->n_dir) base += s->dir_order[d];
  }
  int64_t off = 0;
  P->ld[0] = round4(s->widths[0]);
  for (int l = 1; l <= s->n_layers; ++l) {
    P->w_off[l] = off;
    off += (int64_t)s->widths[l - 1] * s->widths[l];
    P->b_off[l] = off;
    off += s->widths[l];
    P->ld[l] = round4(s->widths[l]);
    if (l < s->n_layers && P->ld[l] > P->ld_hidden_max) P->ld_hidden_max = P->ld[l];
  }
  if (s->gated) {
    for (int e = 0; e < 2; ++e) {
      P->gate_w_off[e] = off;
      const int emb = gate_emb(*s);  // 1: the embeddings read layer 1's output
      off += (int64_t)s->widths[emb] * s->widths[emb + 1];
      P->gate_b_off[e] = off;
      off += s->widths[emb + 1];
    }
    if (s->gated == 2) {
      P->alpha_off = off;
      off += (s->n_layers - 2) / 3;
    }
  }
  P->actp_stride = s->act == PPSCI_ACT_STAN ? 1 : 0;
  for (int l = 0; l <= PPSCI_MAX_LAYERS; ++l) P->actp_off[l] = -1;
  for (int l = 1; l < s->n_layers; ++l) {
    const int a_l = (l == 1 && s->act_first >= 0) ? s->act_first : s->act;
    if (a_l != PPSCI_ACT_STAN && a_l != PPSCI_ACT_SWISH_B) continue;
    P->actp_off[l] = off;
    off += a_l == PPSCI_ACT_STAN ? s->widths[l] : 1;
  }
  P->n_params = off;
  // default points per workspace chunk: large chunks amortise kernel prologues / tails and give the dW kernels long
  // reductions per split (measured on cfg3: 65,536 -> 77.7 ms/step, 262,144 -> 73.7 ms/step); capped below by memory
  P->chunk = s->chunk_points > 0 ? s->chunk_points : (s->dtype == PPSCI_F64 ? 32768 : 262144);
  if (s->chunk_points <= 0) {
    if (const char* m = getenv("PPSCI_B200_CHUNK_POINTS")) {  // tuning knob: points per workspace chunk
      const long long v = atoll(m);
      if (v >= 1024 && v <= (1 << 22)) P->chunk = (int)v;
    }
  }
  {  // the tensor-core dW kernels address a chunk's plane set with 32-bit element offsets
    long long ld_max = 4;
    for (int l = 0; l <= s->n_layers; ++l) ld_max = std::max<long long>(ld_max, (s->widths[l] + 3) / 4 * 4);
    while ((long long)C * P->chunk * ld_max >= (1LL << 32) && P->chunk > 1024) P->chunk /= 2;
  }

  int dev = 0;
  cudaDeviceProp prop;
  if (cudaGetDevice(&dev) == cudaSuccess && cudaGetDeviceProperties(&prop, dev) == cudaSuccess) {
    P->num_sms = prop.multiProcessorCount;
#ifndef PPSCI_EMUL
    if (prop.major != 10) {
      delete P;
      return fail("plan_create: this library is built for sm_100a (B200) only; found compute capability " +
                  std::to_string(prop.major) + "." + std::to_string(prop.minor));
    }
#endif
  } else {
    delete P;
    return fail("plan_create: no CUDA device available (the engine has no CPU fallback)");
  }
  P->use_tc = tc_plan_supported(P->spec, P->C, P->kmax) && s->backend != 1 && !s->gated &&
              s->act != PPSCI_ACT_STAN && s->act != PPSCI_ACT_SWISH_B;
  // the tensor-core kernels apply s.act to every hidden layer, layer 1 included (fill_act, the fused forward / dx
  // chains): a different first-layer activation (a Fourier embedding's sin) runs on the CUDA-core kernels
  if (s->act_first >= 0 && s->act_first != s->act) P->use_tc = false;
#ifdef PPSCI_EMUL
  if (s->backend != 2) P->use_tc = false;  // the emulated tensor-core kernels (1,024 OS threads per CTA pair) run on request only
#endif
  if (const char* m = getenv("PPSCI_B200_TC_MASK")) P->tc_mask = atoi(m);
  if (s->backend == 2 && !P->use_tc) {
    delete P;
    return fail("plan_create: backend=2 (tcgen05) requested but the plan is not eligible (needs f32, no gated layers, "
                "one activation across all hidden layers and not stan / swish, and at least one layer after the first "
                "with K a multiple of 32 up to 1024 and N a multiple of 32 up to 256)");
  }

  auto up = [&](const void* src, size_t bytes, void** dst) -> cudaError_t {
    cudaError_t e = cudaMalloc(dst, bytes ? bytes : 16);
    if (e != cudaSuccess) return e;
    if (bytes) return cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice);
    return cudaSuccess;
  };
  cudaError_t e = cudaSuccess;
  if (e == cudaSuccess) e = up(P->prog.data(), P->prog.size() * 4, (void**)&P->d_prog);
  if (e == cudaSuccess) e = up(P->consts.data(), P->consts.size() * 8, (void**)&P->d_consts);
  if (e == cudaSuccess) e = up(P->grad_res.data(), P->grad_res.size() * 4, (void**)&P->d_grad_res);
  if (e == cudaSuccess) e = up(P->grad_in.data(), P->grad_in.size() * 4, (void**)&P->d_grad_in);
  if (e == cudaSuccess) e = up(P->grad_reg.data(), P->grad_reg.size() * 4, (void**)&P->d_grad_reg);
  if (e != cudaSuccess) {
    ppsci_b200_plan_destroy(P);
    return fail(std::string("plan_create: device upload of the residual program failed: ") + cudaGetErrorString(e));
  }
  if (s->chunk_points <= 0 && getenv("PPSCI_B200_CHUNK_POINTS") == nullptr) {
    // default chunk: keep one call's workspace under ~40 GB of the 180 GB of HBM (cfg3 at 262,144 points: 17.6 GB)
    for (;;) {
      Carve cv;
      carve(P, P->chunk, &cv);
      if (cv.total <= (size_t)40 << 30 || P->chunk <= 16384) break;
      P->chunk /= 2;
    }
  }
  *out = P;
  return 0;
}

extern "C" void ppsci_b200_plan_destroy(ppsci_plan* P) {
  if (!P) return;
  cudaFree(P->d_prog);
  cudaFree(P->d_consts);
  cudaFree(P->d_grad_res);
  cudaFree(P->d_grad_in);
  cudaFree(P->d_grad_reg);
  for (cudaEvent_t e : P->ev_pool) cudaEventDestroy(e);
  delete P;
}

extern "C" int64_t ppsci_b200_plan_param_count(const ppsci_plan* P) { return P ? P->n_params : -1; }
extern "C" int32_t ppsci_b200_plan_channels(const ppsci_plan* P) { return P ? P->C : -1; }
extern "C" int64_t ppsci_b200_plan_last_launches(const ppsci_plan* P) { return P ? P->launches : -1; }
extern "C" int ppsci_b200_plan_set_profile(ppsci_plan* P, int32_t on) {
  if (!P) return fail("null plan");
  P->profile = on != 0;
  return 0;
}
// ms[c] / count[c] for c in {fwd GEMM, head, dW GEMM, dx GEMM, misc} of the most recent call.
extern "C" int ppsci_b200_plan_get_profile(ppsci_plan* P, double* ms, int64_t* count) {
  if (!P || !ms || !count) return fail("null argument");
  for (int c = 0; c < CLS_COUNT; ++c) { ms[c] = 0.0; count[c] = 0; }
#ifndef PPSCI_EMUL
  for (size_t i = 0; i < P->ev_cls.size(); ++i) {
    float t = 0.f;
    CK(cudaEventSynchronize(P->ev_pool[2 * i + 1]));
    CK(cudaEventElapsedTime(&t, P->ev_pool[2 * i], P->ev_pool[2 * i + 1]));
    ms[P->ev_cls[i]] += t;
    count[P->ev_cls[i]] += 1;
  }
#endif
  return 0;
}
extern "C" int32_t ppsci_b200_plan_uses_tcgen05(const ppsci_plan* P) { return (P && P->use_tc) ? 1 : 0; }

// Debug / test accessor: byte offset (from the 256-aligned workspace base) of the jet planes of
// `layer` for a call with n_points points: layer in [1, n_layers) -> hidden pre-activations Z_l,
// layer == n_layers -> output jets Y.  Layout [C][min(n_points, chunk)][ld], ld = round4(width).
extern "C" int64_t ppsci_b200_plan_stash_offset(const ppsci_plan* P, int64_t n_points, int32_t layer) {
  if (!P || n_points <= 0) return -1;
  const int64_t nc = n_points < P->chunk ? n_points : P->chunk;
  Carve cv;
  carve(P, nc, &cv);
  if (layer > 100 && layer - 100 < P->spec.n_layers) return (int64_t)cv.zb[layer - 100];   // debug: Zbar_l (fused dx chain)
  if (layer > 200 && layer - 200 < P->spec.n_layers) return (int64_t)cv.a[layer - 200];    // debug: a-stash of layer l
  if (layer == 300) return (int64_t)cv.ybar;  // output adjoints Ybar (values_bwd_kept accepts this address: no seeding copy)
  if (layer < 1 || layer > P->spec.n_layers) return -1;
  return (int64_t)(layer < P->spec.n_layers ? cv.z[layer] : cv.y);
}

extern "C" size_t ppsci_b200_plan_workspace_bytes(const ppsci_plan* P, int64_t n_points) {
  if (!P || n_points <= 0) return 0;
  const int64_t nc = n_points < P->chunk ? n_points : P->chunk;
  Carve cv;
  carve(P, nc, &cv);
  return cv.total;
}

// ---------------------------------------------------------------------------------------------
template <typename T>
struct Dims {
  static constexpr int TN = sizeof(T) == 8 ? 64 : 128;
};

// bring-up instrumentation: PPSCI_B200_DEBUG_TIMELINE=<device pointer> PPSCI_B200_DEBUG_KERNEL=<0 dW | 1 fwd | 2 dx>
static long long* debug_timeline_ptr(int which) {
  const char* dp = getenv("PPSCI_B200_DEBUG_TIMELINE");
  if (!dp) return nullptr;
  const char* dk = getenv("PPSCI_B200_DEBUG_KERNEL");
  if ((dk ? atoi(dk) : 0) != which) return nullptr;
  return reinterpret_cast<long long*>(strtoull(dp, nullptr, 0));
}

template <typename T, int KMAX>
static int set_attrs_once(ppsci_plan* P) {
  constexpr int TN = Dims<T>::TN;
  auto kf = k_gemm_fwd<T, TN, KMAX>;
  auto kx = k_gemm_dx<T, TN, KMAX>;
  auto kw = k_gemm_dw<T, TN, KMAX>;
  const int smem_f = (KC * TMS + KC * TN) * (int)sizeof(T);
  const int smem_x = std::max(smem_f, TM * TN * (int)sizeof(T));
  const int smem_w = (RC * TMS + RC * TN) * (int)sizeof(T);
  CK(cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_f));
  CK(cudaFuncSetAttribute(kx, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_x));
  CK(cudaFuncSetAttribute(kw, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_w));
  (void)P;
  return 0;
}

template <typename T>
static void fill_seed(const ppsci_plan* P, const void* const* x_cols, int64_t x_off, AOperand<T>* A) {
  const ppsci_plan_spec& s = P->spec;
  A->mode = A_SEED;
  A->act = s.act;
  A->Z = nullptr;
  A->ld = 0;
  A->plane = 0;
  A->x_off = x_off;
  SeedSpec& S = A->seed;
  S.n_in = s.n_in;
  S.n_feat = s.n_feat;
  for (int f = 0; f < PPSCI_MAX_FEAT; ++f) {
    S.feat_src[f] = f < s.n_feat ? s.feat_src[f] : 0;
    S.feat_kind[f] = f < s.n_feat ? s.feat_kind[f] : 0;
    S.feat_omega[f] = f < s.n_feat ? s.feat_omega[f] : 0.0;
  }
  for (int d = 0; d < PPSCI_MAX_DIR; ++d)
    for (int i = 0; i < PPSCI_MAX_IN; ++i) S.dir_vec[d][i] = (d < s.n_dir && i < s.n_in) ? s.dir_vec[d][i] : 0.0;
  for (int i = 0; i < PPSCI_MAX_IN; ++i) S.x_cols[i] = i < s.n_in ? x_cols[i] : nullptr;
}

// activation applied to the output of linear layer `lin` (1-based)
static inline int act_of_layer(const ppsci_plan_spec& s, int lin) { return (lin == 1 && s.act_first >= 0) ? s.act_first : s.act; }
static inline bool act_has_param(int act) { return act == PPSCI_ACT_STAN || act == PPSCI_ACT_SWISH_B; }

template <typename T>
static void fill_act(const ppsci_plan* P, const T* Z, int ld, int64_t nc, int mode, AOperand<T>* A, int lin = 0) {
  A->mode = mode;
  A->act = act_of_layer(P->spec, lin);
  A->Z = Z;
  A->ld = ld;
  A->plane = (long long)nc * ld;
  A->x_off = 0;
  memset(&A->seed, 0, sizeof(SeedSpec));
}

// first-layer operand: input seeds, or (dense_in) the caller's row-major [n_points][n_feat] matrix as a plain operand
template <typename T>
static void fill_first(const ppsci_plan* P, const void* const* x_cols, int64_t x_off, int64_t nc, AOperand<T>* A) {
  if (P->spec.dense_in) {
    const int nf = P->spec.n_feat;
    fill_act<T>(P, reinterpret_cast<const T*>(x_cols[0]) + x_off * nf, nf, nc, A_PLAIN, A);
  } else {
    fill_seed<T>(P, x_cols, x_off, A);
  }
}

struct CallArgs {
  const void* const* x_cols;
  const void* const* aux_cols;
  const void* const* label_cols;
  const double* label_const;
  const void* const* weight_cols;
  int64_t n_points;
  int64_t n_norm;
  const void* params;
  void* grads;
  void* loss_out;
  void* const* residual_out;
  void* jets_out;
  void* workspace;
  size_t workspace_bytes;
  void* stream;
  bool want_loss;
  const void* ybar_in = nullptr;  // values_fwd_bwd: caller-supplied dL/dy [n_points][n_out]
  int phase = 0;                  // 0: forward + adjoint; 1: forward only, stash kept for a later adjoint; 2: adjoint from the kept stash
};

template <typename T, int KMAX>
static int run(ppsci_plan* P, const CallArgs& a) {
  constexpr int TN = Dims<T>::TN;
  const ppsci_plan_spec& s = P->spec;
  const int L = s.n_layers;
  const int C = P->C;
  const int n_out = s.widths[L];
  if (!P->attrs_set) {
    if (set_attrs_once<T, KMAX>(P)) return 1;
    P->attrs_set = true;
  }
  const int64_t nc_max = a.n_points < P->chunk ? a.n_points : P->chunk;
  Carve cv;
  carve(P, nc_max, &cv);
  if (cv.total > a.workspace_bytes)
    return fail("workspace too small: need " + std::to_string(cv.total) + " bytes, got " + std::to_string(a.workspace_bytes));
  if ((reinterpret_cast<uintptr_t>(a.workspace) & 255) != 0) return fail("workspace must be 256-byte aligned");
  unsigned char* ws = reinterpret_cast<unsigned char*>(a.workspace);
  cudaStream_t st = (cudaStream_t)a.stream;
  const T* params = reinterpret_cast<const T*>(a.params);
  T* grads = reinterpret_cast<T*>(a.grads);
  double* loss_acc = reinterpret_cast<double*>(ws + cv.loss_acc);
  P->launches = 0;
  P->ev_used = 0;
  P->ev_cls.clear();

  auto kf = k_gemm_fwd<T, TN, KMAX>;
  auto kx = k_gemm_dx<T, TN, KMAX>;
  auto kw = k_gemm_dw<T, TN, KMAX>;
  const int smem_f = (KC * TMS + KC * TN) * (int)sizeof(T);
  const int smem_x = std::max(smem_f, TM * TN * (int)sizeof(T));
  const int smem_w = (RC * TMS + RC * TN) * (int)sizeof(T);
  const int TP = TM / C;
  const int PT = RC / C;
  const bool thin_on = getenv("PPSCI_B200_NO_THIN") == nullptr;
  const bool gated = s.gated != 0;  // ModifiedMLP: generic tile GEMMs + the gate kernels (kernels_gate.cuh)
  const bool thin_first = thin_on && L >= 2 && s.widths[0] <= THIN_MAXF && !s.dense_in && !gated;
  const bool thin_last = thin_on && L >= 2 && n_out <= THIN_MAXM && C * n_out <= THIN_MAXCM && !gated && !act_has_param(s.act);
  // A_ACT operand of layer lin + 1: beta(s) of layer lin's activation
  auto set_actp = [&](AOperand<T>* A, int lin) {
    if (lin >= 1 && lin < L && P->actp_off[lin] >= 0) {
      A->act_param = params + P->actp_off[lin];
      A->act_pstride = P->actp_stride;
    }
  };
  if (gated && a.phase != 0) return fail("two-phase value calls are not offered for gated networks");
  const bool pirate = s.gated == 2;  // PirateNet: layer 1 = embedding, blocks of (gate, gate, adaptive residual)
  auto kgf = k_gate_fwd<T, KMAX>;
  auto kgb = k_gate_bwd<T, KMAX>;
  auto kmf = k_mix_fwd<T, KMAX>;
  auto kmb = k_mix_bwd<T, KMAX>;
  // what follows hidden layer l in a gated plan: 0 gate, 1 adaptive residual (end of a block), 2 plain activation
  const int emb = gated ? gate_emb(s) : 0;  // layer 1 is an embedding layer (its stored output feeds embed_u / embed_v)
  auto post_kind = [&](int l) -> int { return (emb && l == 1) ? 2 : ((pirate && (l - 2) % 3 == 2) ? 1 : 0); };
  auto fill_mix = [&](int l, int64_t nc, MixArgs<T>* ma) {
    memset(ma, 0, sizeof(*ma));
    ma->J = P->J;
    ma->act = act_of_layer(s, l);
    ma->Z = reinterpret_cast<const T*>(ws + cv.z[l]);
    if (post_kind(l) == 1) {
      ma->Xprev = reinterpret_cast<const T*>(ws + cv.gt[l - 3]);
      ma->alpha = params + P->alpha_off + (l - 2) / 3;
    }
    ma->ld = P->ld[l];
    ma->plane = (long long)nc_max * P->ld[l];
    ma->Np = nc;
    ma->H = s.widths[l];
  };
  auto fill_gate = [&](int l, int64_t nc, GateArgs<T>* ga) {  // gate of hidden layer l
    memset(ga, 0, sizeof(*ga));
    ga->J = P->J;
    ga->act = s.act;
    ga->Z = reinterpret_cast<const T*>(ws + cv.z[l]);
    ga->Zu = reinterpret_cast<const T*>(ws + cv.zu);
    ga->Zv = reinterpret_cast<const T*>(ws + cv.zv);
    ga->ld = P->ld[l];
    ga->plane = (long long)nc_max * P->ld[l];
    ga->Np = nc;
    ga->H = s.widths[l];
  };
  // fp32 + one of the compile-time jet layouts: vectorised thin kernels (kernels_thin.cuh)
  const int thin_lay = tc_pick_layout(P->J, PPSCI_ACT_TANH);
  const bool thin_vec = sizeof(T) == 4 && thin_lay != TC_LAY_DYN && getenv("PPSCI_B200_NO_THINV") == nullptr;

  if (a.want_loss) CK(cudaMemsetAsync(loss_acc, 0, PPSCI_MAX_RES * sizeof(double), st));
  // phase 1 runs the forward exactly as a training call would (stash of everything the adjoint reads), phase 2 only the adjoint
  const bool do_bwd = ((a.want_loss || a.ybar_in) && grads != nullptr) || a.phase == 1;
  if (a.phase == 2 && a.n_points > nc_max)
    return fail("values_bwd_kept: the kept stash covers one workspace chunk (" + std::to_string(nc_max) + " points); got " +
                std::to_string(a.n_points));
  if (do_bwd) {
    for (int l = 2; l <= L; ++l) {
      const int K = s.widths[l - 1], N = s.widths[l];
      const long long tot = (long long)K * N;
      auto kt = k_transpose<T>;
      ProfScope ps_(P, CLS_MISC, st);
      PPSCI_LAUNCH(kt, dim3((unsigned)((tot + 255) / 256)), dim3(256), 0, st, params + P->w_off[l],
                   reinterpret_cast<T*>(ws + cv.wt[l]), K, N);
      P->launches++;
    }
    for (int e = 0; e < (emb ? 2 : 0); ++e) {  // the embeddings hand an adjoint back to layer 1's output
      const int K = s.widths[1], N = s.widths[2];
      const long long tot = (long long)K * N;
      auto kt = k_transpose<T>;
      ProfScope ps_(P, CLS_MISC, st);
      PPSCI_LAUNCH(kt, dim3((unsigned)((tot + 255) / 256)), dim3(256), 0, st, params + P->gate_w_off[e],
                   reinterpret_cast<T*>(ws + (e == 0 ? cv.wtu : cv.wtv)), K, N);
      P->launches++;
    }
  }

  if constexpr (sizeof(T) == 4) {
    if (P->use_tc) {
      for (int l = 2; l <= L; ++l) {  // hidden -> hidden layers and a wide output layer
        if (!tc_layer_ok(s, l)) continue;
        const int K = s.widths[l - 1], N = s.widths[l];
        const long long tot = (long long)K * N;
        ProfScope ps_(P, CLS_MISC, st);
        PPSCI_LAUNCH(tc::k_tc_prep_w, dim3((unsigned)((tot + 255) / 256)), dim3(256), 0, st,
                     reinterpret_cast<const float*>(params) + P->w_off[l],
                     reinterpret_cast<float*>(ws + cv.tc + tc_img_offset(s, l)), K, N, 0);
        P->launches++;
      }
      if ((P->tc_mask & 1) && tc_dense_first_ok(s)) {  // dense first layer: K rounded up to the chunk width, zero rows beyond
        const int K = s.widths[0], N = s.widths[1];
        float* img = reinterpret_cast<float*>(ws + cv.tc + tc_dense_img_offset(s));
        ProfScope ps_(P, CLS_MISC, st);
        CK(cudaMemsetAsync(img, 0, (size_t)tc_dense_kpad(s) * N * 8, st));
        PPSCI_LAUNCH(tc::k_tc_prep_w, dim3((unsigned)(((long long)K * N + 255) / 256)), dim3(256), 0, st,
                     reinterpret_cast<const float*>(params) + P->w_off[1], img, K, N, 0);
        P->launches++;
      }
      if (do_bwd && (P->tc_mask & 2)) {
        for (int l = 2; l <= L; ++l) {
          if (!tc_dx_ok(s, l)) continue;
          const int K = s.widths[l], N = s.widths[l - 1];  // gemm K = fan-out, gemm N = fan-in
          const long long tot = (long long)K * N;
          ProfScope ps_(P, CLS_MISC, st);
          PPSCI_LAUNCH(tc::k_tc_prep_w, dim3((unsigned)((tot + 255) / 256)), dim3(256), 0, st,
                       reinterpret_cast<const float*>(params) + P->w_off[l],
                       reinterpret_cast<float*>(ws + cv.tc + tc_imgT_offset(s, l)), K, N, 1);
          P->launches++;
        }
      }
    }
  }
  for (int64_t c0 = 0; c0 < a.n_points; c0 += nc_max) {
    const int64_t nc = (a.n_points - c0) < nc_max ? (a.n_points - c0) : nc_max;
    const unsigned ptiles = (unsigned)((nc + TP - 1) / TP);
    // ---------------- forward ----------------
    for (int l = (a.phase == 2 ? L + 1 : 1); l <= L; ++l) {
      if (l == 1 && thin_first) {
        FirstArgs<T> f;
        memset(&f, 0, sizeof(f));
        fill_seed<T>(P, a.x_cols, c0, &f.A);
        f.J = P->J;
        f.W = params + P->w_off[1];
        f.bias = params + P->b_off[1];
        f.nf = s.widths[0];
        f.N = s.widths[1];
        f.Out = reinterpret_cast<T*>(ws + (L > 1 ? cv.z[1] : cv.y));
        f.ldo = P->ld[1];
        f.oplane = (long long)nc_max * P->ld[1];
        f.Np = nc;
        const long long tot = (long long)nc * f.N;
        if constexpr (sizeof(T) == 4) {
          if (thin_vec && f.N % 4 == 0) {  // compile-time layout, 128-bit stores, seeds staged once per point
            void (*kv)(FirstArgs<float>) = nullptr;
            PPSCI_THIN_PICK_L(k_first_fwd_v, thin_lay, KMAX, kv);
            ProfScope ps_(P, CLS_THIN_FWD, st);
            PPSCI_LAUNCH(kv, dim3((unsigned)((nc + thin::PB - 1) / thin::PB)), dim3(256), 0, st, f);
            P->launches++;
            continue;
          }
        }
        auto k1 = k_first_fwd<T, KMAX>;
        ProfScope ps_(P, CLS_THIN_FWD, st);
        PPSCI_LAUNCH(k1, dim3((unsigned)((tot + 255) / 256)), dim3(256), 0, st, f);
        P->launches++;
        continue;
      }
      if (l == L && thin_last) {
        LastArgs<T> f;
        memset(&f, 0, sizeof(f));
        fill_act<T>(P, reinterpret_cast<const T*>(ws + cv.z[L - 1]), P->ld[L - 1], nc_max, A_ACT, &f.A, L - 1);
        f.J = P->J;
        f.W = params + P->w_off[L];
        f.bias = params + P->b_off[L];
        f.K = s.widths[L - 1];
        f.m = s.widths[L];
        f.Y = reinterpret_cast<T*>(ws + cv.y);
        f.ldy = P->ld[L];
        f.yplane = (long long)nc_max * P->ld[L];
        f.Np = nc;
        if constexpr (sizeof(T) == 4) {
          if (thin_vec && f.K % 4 == 0 && f.m <= 4) {
            void (*kv)(LastArgs<float>) = nullptr;
            PPSCI_THIN_PICK_LM(k_last_fwd_v, thin_lay, f.m, kv);
            ProfScope ps_(P, CLS_THIN_FWD, st);
            PPSCI_LAUNCH(kv, dim3((unsigned)((nc + 7) / 8)), dim3(256), 0, st, f);
            P->launches++;
            continue;
          }
        }
        auto k2 = k_last_fwd<T, KMAX>;
        ProfScope ps_(P, CLS_THIN_FWD, st);
        PPSCI_LAUNCH(k2, dim3((unsigned)((nc + 7) / 8)), dim3(256), 0, st, f);
        P->launches++;
        continue;
      }
      if constexpr (sizeof(T) == 4) {
        if (l == 1 && P->use_tc && (P->tc_mask & 1) && tc_dense_first_ok(s)) {
          // dense first layer (DeepONet branch net: [N][num_loc] sensor matrix) on the tensor cores: the operand is the
          // caller's matrix itself ("activation" = identity, values only), columns beyond K read as zero
          tc::TcFwdArgs t;
          memset(&t, 0, sizeof(t));
          const int nf = s.widths[0];
          fill_act<float>(P, reinterpret_cast<const float*>(a.x_cols[0]) + c0 * nf, nf, nc_max, A_ACT, &t.A);
          t.A.act = PPSCI_ACT_IDENTITY;
          t.J = P->J;
          t.Wimg = reinterpret_cast<const float*>(ws + cv.tc + tc_dense_img_offset(s));
          t.Kdim = tc_dense_kpad(s);
          t.Kvalid = nf;
          t.Nout = s.widths[1];
          t.bias = reinterpret_cast<const float*>(params) + P->b_off[1];
          t.Out = reinterpret_cast<float*>(ws + (L > 1 ? cv.z[1] : cv.y));
          t.ldo = P->ld[1];
          t.oplane = (long long)nc_max * P->ld[1];
          t.Np = nc;
          t.TP = TP;
          t.num_tiles = (int)ptiles;
          const int smem_tc = tc::tc_fwd_smem_bytes(t.Nout);
          const unsigned gridx = ptiles < (unsigned)P->num_sms ? ptiles : (unsigned)P->num_sms;
          void (*kd)(tc::TcFwdArgs) = tc::k_tc_fwd<tc::SLay<0, 0, 0, 0>, -1>;
          {
            cudaError_t e_ = cudaFuncSetAttribute(kd, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_tc);
            if (e_ != cudaSuccess) return fail(std::string("cudaFuncSetAttribute(k_tc_fwd dense): ") + cudaGetErrorString(e_));
          }
          ProfScope ps_(P, CLS_FWD, st);
          PPSCI_KLAUNCH(kd, dim3(gridx), dim3(tc::THREADS), smem_tc, st, 1, t);
          P->launches++;
          continue;
        }
        if (l == 2 && fused_fwd16_ok(P)) {  // fused forward, fp16 hi / lo operands after the first layer (accurate for wide layers)
          const int H = s.widths[1], NLf = L - 2;
          unsigned char* w16 = ws + cv.w16;
          const size_t img_bytes = (size_t)H * H * 4;
          unsigned* absmax = reinterpret_cast<unsigned*>(w16 + (size_t)(NLf - 1) * img_bytes);
          float* wscale = reinterpret_cast<float*>(absmax + PPSCI_MAX_LAYERS);
          if (c0 == 0) {  // weight scales + fp16 images once per call
            ProfScope ps_(P, CLS_MISC, st);
            CK(cudaMemsetAsync(absmax, 0, 2 * sizeof(unsigned) * PPSCI_MAX_LAYERS, st));
            for (int i = 1; i < NLf; ++i) {
              const float* Wl = reinterpret_cast<const float*>(params) + P->w_off[2 + i];
              PPSCI_LAUNCH(tc::k_w16_absmax, dim3(64), dim3(256), 0, st, Wl, (long long)H * H, absmax + i);
              PPSCI_LAUNCH(tc::k_w16_scale, dim3(1), dim3(1), 0, st, absmax + i, wscale + i);
              PPSCI_LAUNCH(tc::k_tc_prep_w16, dim3((unsigned)(((long long)H * H + 255) / 256)), dim3(256), 0, st, Wl,
                           reinterpret_cast<unsigned short*>(w16 + (size_t)(i - 1) * img_bytes), H, H, wscale + i);
              P->launches += 3;
            }
          }
          tc::FusedFwd16Args ta;
          memset(&ta, 0, sizeof(ta));
          tc::FusedFwdArgs& t = ta.f;
          t.J = P->J;
          t.act = s.act;
          t.H = H;
          t.n_fused = NLf;
          t.Zin = reinterpret_cast<const float*>(ws + cv.z[1]);
          t.ld = P->ld[1];
          t.plane = (long long)nc_max * P->ld[1];
          for (int i = 0; i < NLf; ++i) {
            t.Wimg[i] = i == 0 ? reinterpret_cast<const float*>(ws + cv.tc + tc_img_offset(s, 2))
                               : reinterpret_cast<const float*>(w16 + (size_t)(i - 1) * img_bytes);
            t.bias[i] = reinterpret_cast<const float*>(params) + P->b_off[2 + i];
            t.Zout[i] = reinterpret_cast<float*>(ws + cv.z[2 + i]);
            t.Astash[i] = (do_bwd && tc_astash_needed(P, 1 + i)) ? reinterpret_cast<float*>(ws + cv.a[1 + i]) : nullptr;
          }
          t.Np = nc;
          t.num_tiles = (int)ptiles;
          t.dbg = debug_timeline_ptr(3);
          ta.wscale = wscale;
          const int smemf = tc::fused_fwd16_smem_bytes(H);
          const unsigned tile_pairs = (ptiles + 1) / 2, sm_pairs = (unsigned)P->num_sms / 2;
          const unsigned gridf = 2 * (tile_pairs < sm_pairs ? tile_pairs : sm_pairs);
          ProfScope ps_(P, CLS_FWD, st);
          PPSCI_FUSED_LAUNCH(k_fused_fwd16, tc_pick_layout(P->J, s.act), dim3(gridf), smemf, st, ta,
                             return fail(std::string("cudaFuncSetAttribute(k_fused_fwd16): ") + cudaGetErrorString(e_)));
          P->launches++;
          l = L - 1;
          continue;
        }
        if (l == 2 && fused_fwd_ok(P)) {  // every hidden -> hidden layer in ONE launch, jets stay on chip between layers
          tc::FusedFwdArgs t;
          memset(&t, 0, sizeof(t));
          t.J = P->J;
          t.act = s.act;
          t.H = s.widths[1];
          t.n_fused = L - 2;
          t.Zin = reinterpret_cast<const float*>(ws + cv.z[1]);
          t.ld = P->ld[1];
          t.plane = (long long)nc_max * P->ld[1];
          for (int i = 0; i < L - 2; ++i) {
            t.Wimg[i] = reinterpret_cast<const float*>(ws + cv.tc + tc_img_offset(s, 2 + i));
            t.bias[i] = reinterpret_cast<const float*>(params) + P->b_off[2 + i];
            t.Zout[i] = reinterpret_cast<float*>(ws + cv.z[2 + i]);
            t.Astash[i] = (do_bwd && tc_astash_needed(P, 1 + i)) ? reinterpret_cast<float*>(ws + cv.a[1 + i]) : nullptr;
          }
          t.Np = nc;
          t.num_tiles = (int)ptiles;
          t.dbg = debug_timeline_ptr(3);
          const int smemf = tc::fused_fwd_smem_bytes(t.H);
          const unsigned tile_pairs = (ptiles + 1) / 2, sm_pairs = (unsigned)P->num_sms / 2;
          const unsigned gridf = 2 * (tile_pairs < sm_pairs ? tile_pairs : sm_pairs);
          ProfScope ps_(P, CLS_FWD, st);
          PPSCI_FUSED_LAUNCH(k_fused_fwd, tc_pick_layout(P->J, s.act), dim3(gridf), smemf, st, t,
                             return fail(std::string("cudaFuncSetAttribute(k_fused_fwd): ") + cudaGetErrorString(e_)));
          P->launches++;
          l = L - 1;  // the loop's ++l continues with the output layer
          continue;
        }
      }
      if constexpr (sizeof(T) == 4) {
        if (P->use_tc && (P->tc_mask & 1) && tc_layer_ok(s, l)) {
          tc::TcFwdArgs t;
          memset(&t, 0, sizeof(t));
          fill_act<float>(P, reinterpret_cast<const float*>(ws + cv.z[l - 1]), P->ld[l - 1], nc_max, A_ACT, &t.A);
          t.J = P->J;
          t.Wimg = reinterpret_cast<const float*>(ws + cv.tc + tc_img_offset(s, l));
          t.Kdim = s.widths[l - 1];
          t.Nout = s.widths[l];
          t.bias = reinterpret_cast<const float*>(params) + P->b_off[l];
          t.Out = reinterpret_cast<float*>(ws + (l == L ? cv.y : cv.z[l]));  // a wide output layer writes Y
          t.ldo = P->ld[l];
          t.oplane = (long long)nc_max * P->ld[l];
          t.Np = nc;
          t.TP = TP;
          t.num_tiles = (int)ptiles;
          t.dbg = debug_timeline_ptr(1);
          if (do_bwd && tc_astash_needed(P, l - 1)) {
            t.Astash = reinterpret_cast<float*>(ws + cv.a[l - 1]);
            t.lda = P->ld[l - 1];
            t.aplane = (long long)nc_max * P->ld[l - 1];
          }
          const int lay_f = tc_pick_layout(P->J, s.act);
          if ((P->tc_mask & 8) && lay_f != TC_LAY_DYN && P->num_sms >= 2) {  // CTA pairs (cta_group::2)
            const int smem2 = tc::tc2_smem_bytes(t.Nout);
            const unsigned tile_pairs = (ptiles + 1) / 2, sm_pairs = (unsigned)P->num_sms / 2;
            const unsigned gridx2 = 2 * (tile_pairs < sm_pairs ? tile_pairs : sm_pairs);
            ProfScope ps_(P, CLS_FWD, st);
            PPSCI_TC2_LAUNCH(k_tc2_fwd, lay_f, dim3(gridx2), smem2, st, t,
                             return fail(std::string("cudaFuncSetAttribute(k_tc2_fwd): ") + cudaGetErrorString(e_)));
            P->launches++;
            continue;
          }
          const int smem_tc = tc::tc_fwd_smem_bytes(t.Nout);
          const unsigned gridx = ptiles < (unsigned)P->num_sms ? ptiles : (unsigned)P->num_sms;
          ProfScope ps_(P, CLS_FWD, st);
          PPSCI_TC_LAUNCH(k_tc_fwd, tc_pick_layout(P->J, s.act), KMAX, dim3(gridx), smem_tc, st, t,
                          return fail(std::string("cudaFuncSetAttribute(k_tc_fwd): ") + cudaGetErrorString(e_)));
          P->launches++;
          continue;
        }
      }
      GemmArgs<T> g;
      memset(&g, 0, sizeof(g));
      if (l == 1) fill_first<T>(P, a.x_cols, c0, nc_max, &g.A);
      else if (gated)  // the gate / residual / activation that follows layer l-1 was stored when that layer finished
        fill_act<T>(P, reinterpret_cast<const T*>(ws + cv.gt[l - 1]), P->ld[l - 1], nc_max, A_PLAIN, &g.A);
      else {
        fill_act<T>(P, reinterpret_cast<const T*>(ws + cv.z[l - 1]), P->ld[l - 1], nc_max, A_ACT, &g.A, l - 1);
        set_actp(&g.A, l - 1);
      }
      g.J = P->J;
      g.B = params + P->w_off[l];
      g.Kdim = s.widths[l - 1];
      g.Nout = s.widths[l];
      g.ldb = s.widths[l];
      g.bias = params + P->b_off[l];
      g.Out = reinterpret_cast<T*>(ws + (l < L ? cv.z[l] : cv.y));
      g.ldo = P->ld[l];
      g.oplane = (long long)nc_max * P->ld[l];
      g.Np = nc;
      g.TP = TP;
      dim3 grid(ptiles, (unsigned)((g.Nout + TN - 1) / TN));
      {
        ProfScope ps_(P, CLS_FWD, st);
        PPSCI_LAUNCH(kf, grid, dim3(NTHREADS), smem_f, st, g);
        P->launches++;
      }
      auto post_fwd = [&](int lay) {  // operand of layer lay + 1
        const long long tot = (long long)nc * s.widths[lay];
        ProfScope ps_(P, CLS_MISC, st);
        if (post_kind(lay) == 0) {  // G = V + act(Z) (U - V)
          GateArgs<T> ga;
          fill_gate(lay, nc, &ga);
          ga.G = reinterpret_cast<T*>(ws + cv.gt[lay]);
          PPSCI_LAUNCH(kgf, dim3((unsigned)((tot + 127) / 128)), dim3(128), 0, st, ga);
        } else {  // X = alpha act(Z) + (1 - alpha) X_block_in, or X = act(Z)
          MixArgs<T> ma;
          fill_mix(lay, nc, &ma);
          ma.X = reinterpret_cast<T*>(ws + cv.gt[lay]);
          PPSCI_LAUNCH(kmf, dim3((unsigned)((tot + 127) / 128)), dim3(128), 0, st, ma);
        }
        P->launches++;
      };
      if (emb && l == 1) post_fwd(1);
      if (gated && l == 1) {  // embed_u / embed_v: two more layers from the seeds, or from the embedding layer's output
        dim3 grid_e = grid;
        if (emb) {
          fill_act<T>(P, reinterpret_cast<const T*>(ws + cv.gt[1]), P->ld[1], nc_max, A_PLAIN, &g.A);
          g.Kdim = s.widths[1];
          g.Nout = s.widths[2];
          g.ldb = s.widths[2];
          g.ldo = P->ld[2];
          g.oplane = (long long)nc_max * P->ld[2];
          grid_e = dim3(ptiles, (unsigned)((g.Nout + TN - 1) / TN));
        }
        for (int e = 0; e < 2; ++e) {
          g.B = params + P->gate_w_off[e];
          g.bias = params + P->gate_b_off[e];
          g.Out = reinterpret_cast<T*>(ws + (e == 0 ? cv.zu : cv.zv));
          ProfScope ps_(P, CLS_FWD, st);
          PPSCI_LAUNCH(kf, grid_e, dim3(NTHREADS), smem_f, st, g);
          P->launches++;
        }
      }
      if (gated && l < L && !(emb && l == 1)) post_fwd(l);
    }
    // ---------------- residual program + loss + output adjoints ----------------
    if (a.jets_out) {
      const long long tot = (long long)C * nc * n_out;
      auto kc = k_copy_jets<T>;
      ProfScope ps_(P, CLS_MISC, st);
      PPSCI_LAUNCH(kc, dim3((unsigned)((tot + 255) / 256)), dim3(256), 0, st,
                   reinterpret_cast<const T*>(ws + cv.y), P->ld[L], (long long)nc_max * P->ld[L],
                   reinterpret_cast<T*>(a.jets_out), (long long)a.n_points, (long long)c0, (long long)nc, C, n_out);
      P->launches++;
    }
    if (s.n_res > 0 && (a.want_loss || a.residual_out) && !a.ybar_in) {
      HeadArgs<T> h;
      memset(&h, 0, sizeof(h));
      h.P.prog = P->d_prog;
      h.P.consts = P->d_consts;
      h.P.n_ops = s.n_ops;
      h.P.n_reg = s.n_reg;
      h.P.n_res = s.n_res;
      for (int k = 0; k < PPSCI_MAX_RES; ++k) h.P.res_reg[k] = k < s.n_res ? s.res_reg[k] : 0;
      h.P.n_grad = s.n_grad;
      h.P.grad_res = P->d_grad_res;
      h.P.grad_in = P->d_grad_in;
      h.P.grad_reg = P->d_grad_reg;
      h.P.n_pgrad = s.n_pgrad;
      for (int g = 0; g < PPSCI_MAX_PGRAD; ++g) {
        h.P.pgrad_res[g] = g < s.n_pgrad ? s.pgrad_res[g] : 0;
        h.P.pgrad_aux[g] = g < s.n_pgrad ? s.pgrad_aux[g] : -1;
        h.P.pgrad_reg[g] = g < s.n_pgrad ? s.pgrad_reg[g] : 0;
      }
      for (int i = 0; i < PPSCI_MAX_IN; ++i) {
        h.aux_bcast[i] = i < s.n_aux ? s.aux_bcast[i] : 0;
        h.aux_grad[i] = (i < s.n_aux && s.aux_bcast[i] && do_bwd) ? P->aux_grad[i] : nullptr;
      }
      h.C = C;
      h.n_out = n_out;
      h.n_in = s.n_in;
      h.n_aux = s.n_aux;
      h.Y = reinterpret_cast<const T*>(ws + cv.y);
      h.ldy = P->ld[L];
      h.yplane = (long long)nc_max * P->ld[L];
      h.Ybar = do_bwd ? reinterpret_cast<T*>(ws + cv.ybar) : nullptr;
      for (int i = 0; i < s.n_in; ++i) h.x_cols[i] = a.x_cols[i];
      for (int i = 0; i < s.n_aux; ++i) h.aux_cols[i] = a.aux_cols ? a.aux_cols[i] : nullptr;
      h.x_off = c0;
      h.Np = nc;
      for (int k = 0; k < s.n_res; ++k) {
        h.label_cols[k] = a.label_cols ? a.label_cols[k] : nullptr;
        h.label_const[k] = a.label_const ? a.label_const[k] : 0.0;
        h.weight_cols[k] = a.weight_cols ? a.weight_cols[k] : nullptr;
        h.coef[k] = s.loss_weight[k] * (s.reduction[k] == PPSCI_REDUCE_MEAN ? 1.0 / (double)a.n_norm : 1.0);
        h.residual_out[k] = a.residual_out ? a.residual_out[k] : nullptr;
      }
      h.loss_acc = a.want_loss ? loss_acc : nullptr;
      auto kh = k_head<T>;
      ProfScope ps_(P, CLS_HEAD, st);
      PPSCI_LAUNCH(kh, dim3((unsigned)((nc + HEAD_THREADS - 1) / HEAD_THREADS)), dim3(HEAD_THREADS), 0, st, h);
      P->launches++;
    }
    if (!do_bwd || a.phase == 1) continue;
    if (a.ybar_in && a.ybar_in != static_cast<const void*>(ws + cv.ybar)) {  // output adjoints from the caller (not already in place)
      const long long tot = (long long)nc * P->ld[L];
      auto ks = k_seed_ybar<T>;
      ProfScope ps_(P, CLS_MISC, st);
      PPSCI_LAUNCH(ks, dim3((unsigned)((tot + 255) / 256)), dim3(256), 0, st, reinterpret_cast<const T*>(a.ybar_in),
                   (long long)c0, (long long)nc, n_out, C, reinterpret_cast<T*>(ws + cv.ybar), P->ld[L],
                   (long long)nc_max * P->ld[L]);
      P->launches++;
    }
    // ---------------- adjoint ----------------
    const T* zbar_cur = reinterpret_cast<const T*>(ws + cv.ybar);
    int zbar_ld = P->ld[L];
    int flip = 0;
    const bool fdx = fused_dx_ok(P);
    bool fdx_done = false;
    // destination of Zbar_{lower}: its own buffer under the fused dx chain, the two ping-pong buffers otherwise
    auto zbar_dst = [&](int lower) -> T* {
      return reinterpret_cast<T*>(ws + (fdx ? cv.zb[lower] : (flip ? cv.zbar1 : cv.zbar0)));
    };
    for (int l = L; l >= 1; --l) {
      if constexpr (sizeof(T) == 4) {
        if (fdx && l == L - 1 && !fdx_done) {  // Zbar_{L-1} is in place: Zbar_{L-2} .. Zbar_1 in ONE launch
          tc::FusedDxArgs t;
          memset(&t, 0, sizeof(t));
          t.J = P->J;
          t.act = s.act;
          t.H = s.widths[1];
          t.n_fused = L - 2;
          t.ZbarIn = reinterpret_cast<const float*>(ws + cv.zb[L - 1]);
          t.ld = P->ld[1];
          t.plane = (long long)nc_max * P->ld[1];
          for (int i = 0; i < L - 2; ++i) {
            const int ll = L - 1 - i;
            t.WimgT[i] = reinterpret_cast<const float*>(ws + cv.tc + tc_imgT_offset(s, ll));
            t.Zprev[i] = reinterpret_cast<const float*>(ws + cv.z[ll - 1]);
            t.ZbarOut[i] = reinterpret_cast<float*>(ws + cv.zb[ll - 1]);
          }
          t.Np = nc;
          t.num_tiles = (int)ptiles;
          t.dbg = debug_timeline_ptr(4);
          const int smemf = tc::fused_fwd_smem_bytes(t.H);
          const unsigned tile_pairs = (ptiles + 1) / 2, sm_pairs = (unsigned)P->num_sms / 2;
          const unsigned gridf = 2 * (tile_pairs < sm_pairs ? tile_pairs : sm_pairs);
          ProfScope ps_(P, CLS_DX, st);
          PPSCI_FUSED_LAUNCH(k_fused_dx, tc_pick_layout(P->J, s.act), dim3(gridf), smemf, st, t,
                             return fail(std::string("cudaFuncSetAttribute(k_fused_dx): ") + cudaGetErrorString(e_)));
          P->launches++;
          fdx_done = true;
        }
      }
      if (l == L && thin_last) {  // dW_L, db_L and Zbar_{L-1} in one streaming pass
        LastArgs<T> f;
        memset(&f, 0, sizeof(f));
        fill_act<T>(P, reinterpret_cast<const T*>(ws + cv.z[L - 1]), P->ld[L - 1], nc_max, A_ACT, &f.A, L - 1);
        f.J = P->J;
        f.W = params + P->w_off[L];
        f.K = s.widths[L - 1];
        f.m = s.widths[L];
        f.Ybar = zbar_cur;
        f.ldy = P->ld[L];
        f.yplane = (long long)nc_max * P->ld[L];
        T* outp = zbar_dst(L - 1);
        f.ZbarOut = outp;
        f.ldo = P->ld[L - 1];
        f.oplane = (long long)nc_max * P->ld[L - 1];
        f.dW = grads + P->w_off[L];
        f.db = grads + P->b_off[L];
        f.Np = nc;
        f.pts_per_block = 64;
        bool last_done = false;
        if constexpr (sizeof(T) == 4) {
          if (thin_vec && f.K % 4 == 0 && f.m <= 4) {
            f.pts_per_block = 128;
            void (*kv)(LastArgs<float>) = nullptr;
            PPSCI_THIN_PICK_LM(k_last_bwd_v, thin_lay, f.m, kv);
            ProfScope ps_(P, CLS_THIN_DX, st);
            PPSCI_LAUNCH(kv, dim3((unsigned)((f.K + 255) / 256), (unsigned)((nc + 127) / 128)), dim3(256), 0, st, f);
            P->launches++;
            last_done = true;
          }
        }
        if (!last_done) {
          auto k3 = k_last_bwd<T, KMAX>;
          ProfScope ps_(P, CLS_THIN_DX, st);
          PPSCI_LAUNCH(k3, dim3((unsigned)((f.K + 255) / 256), (unsigned)((nc + 63) / 64)), dim3(256), 0, st, f);
          P->launches++;
        }
        zbar_cur = outp;
        zbar_ld = P->ld[L - 1];
        flip ^= 1;
        continue;
      }
      if (l == 1 && thin_first) {
        FirstArgs<T> f;
        memset(&f, 0, sizeof(f));
        fill_seed<T>(P, a.x_cols, c0, &f.A);
        f.J = P->J;
        f.nf = s.widths[0];
        f.N = s.widths[1];
        f.Zbar = zbar_cur;
        f.ldzb = zbar_ld;
        f.zbplane = (long long)nc_max * zbar_ld;
        f.dW = grads + P->w_off[1];
        f.db = grads + P->b_off[1];
        f.Np = nc;
        f.pts_per_block = 32;
        if constexpr (sizeof(T) == 4) {
          if (thin_vec && f.N % 4 == 0) {
            f.pts_per_block = 256;
            void (*kv)(FirstArgs<float>) = nullptr;
            PPSCI_THIN_PICK_L(k_first_dw_v, thin_lay, KMAX, kv);
            ProfScope ps_(P, CLS_THIN_DW, st);
            PPSCI_LAUNCH(kv, dim3((unsigned)((f.N + 255) / 256), (unsigned)((nc + 255) / 256)), dim3(256), 0, st, f);
            P->launches++;
            break;
          }
        }
        auto k4 = k_first_dw<T, KMAX>;
        ProfScope ps_(P, CLS_THIN_DW, st);
        PPSCI_LAUNCH(k4, dim3((unsigned)((f.N + 255) / 256), (unsigned)((nc + 31) / 32)), dim3(256), 0, st, f);
        P->launches++;
        break;
      }
      bool dw_done = false;
      if constexpr (sizeof(T) == 4) {
        const bool dense_tc = l == 1 && P->use_tc && (P->tc_mask & 1) && (P->tc_mask & 4) && tc_dense_first_ok(s);
        if (dense_tc || (l >= 2 && tc_astash_needed(P, l - 1))) {
          tc::TcDwArgs t;
          memset(&t, 0, sizeof(t));
          if (dense_tc) {  // the operand of dW_1 is the caller's sensor matrix itself (fan-in rows beyond K are masked)
            t.Aact = reinterpret_cast<const float*>(a.x_cols[0]) + c0 * s.widths[0];
            t.lda = s.widths[0];
            t.aplane = 0;
          } else {
            t.Aact = reinterpret_cast<const float*>(ws + cv.a[l - 1]);
            t.lda = P->ld[l - 1];
            t.aplane = (long long)nc_max * P->ld[l - 1];
          }
          t.J = P->J;
          t.Zbar = reinterpret_cast<const float*>(zbar_cur);
          t.ldzb = zbar_ld;
          t.zbplane = (long long)nc_max * zbar_ld;
          t.Kdim = s.widths[l - 1];
          t.Nout = s.widths[l];
          t.dW = reinterpret_cast<float*>(grads) + P->w_off[l];
          t.Np = nc;
          const int PTt = tc::KCH / C;
          t.PT = PTt;
          const int NC = tc_dw_cols_per_cta(s.widths[l]);
          t.Nout = NC;
          t.n0_stride = NC;
          t.ldw = s.widths[l];
          const long long total_chunks = (nc + PTt - 1) / PTt;
          bool db_fused = false;
          if ((P->tc_mask & 32) && t.Kdim % 256 == 0 && s.widths[l] % 256 == 0 && P->num_sms >= 2) {
            // CTA pairs (cta_group::2): one pair per 256 x 256 block of dW and reduction split
            const unsigned kt2 = (unsigned)(t.Kdim / 256), nb2 = (unsigned)(s.widths[l] / 256);
            long long want2 = (P->num_sms / 2) / (kt2 * nb2);
            if (want2 < 1) want2 = 1;
            if (want2 > total_chunks) want2 = total_chunks;
            const long long cps2 = (total_chunks + want2 - 1) / want2;
            const unsigned splits2 = (unsigned)((total_chunks + cps2 - 1) / cps2);
            t.chunks_per_split = (int)cps2;
            t.dbg = debug_timeline_ptr(0);
            t.db = reinterpret_cast<float*>(grads) + P->b_off[l];  // bias gradient fused into the Zbar producer
            db_fused = true;
            const int smem2 = tc::tc2_smem_bytes(256);
            ProfScope ps_(P, CLS_DW, st);
            PPSCI_TC2_LAUNCH_L(k_tc2_dw, tc_pick_layout(P->J, PPSCI_ACT_TANH), dim3(2 * kt2, splits2, nb2), smem2, st, t,
                               return fail(std::string("cudaFuncSetAttribute(k_tc2_dw): ") + cudaGetErrorString(e_)));
            P->launches++;
          } else {
          const unsigned kt = (unsigned)((t.Kdim + 127) / 128), nb = (unsigned)(s.widths[l] / NC);
          long long want = P->num_sms / (kt * nb);
          if (want < 1) want = 1;
          if (want > total_chunks) want = total_chunks;
          const long long cps = (total_chunks + want - 1) / want;
          const unsigned splits = (unsigned)((total_chunks + cps - 1) / cps);
          t.chunks_per_split = (int)cps;
          t.dbg = debug_timeline_ptr(0);
          const int smem_tc = tc::tc_dw_smem_bytes(NC);
          {
            ProfScope ps_(P, CLS_DW, st);
            PPSCI_TC_LAUNCH_L(k_tc_dw, tc_pick_layout(P->J, PPSCI_ACT_TANH), KMAX, dim3(kt, splits, nb), smem_tc, st, t,
                            return fail(std::string("cudaFuncSetAttribute(k_tc_dw): ") + cudaGetErrorString(e_)));
            P->launches++;
          }
          }
          if (!db_fused) {
            ProfScope ps_(P, CLS_THIN_DW, st);
            const int ppb = 512;
            PPSCI_LAUNCH(tc::k_bias_grad, dim3((unsigned)((s.widths[l] + 127) / 128), (unsigned)((nc + ppb - 1) / ppb)), dim3(128), 0, st,
                         reinterpret_cast<const float*>(zbar_cur), zbar_ld, (long long)nc, s.widths[l],
                         reinterpret_cast<float*>(grads) + P->b_off[l], ppb);
            P->launches++;
          }
          dw_done = true;
        }
      }
      if (!dw_done)
      {  // dW_l, db_l
        DwArgs<T> g;
        memset(&g, 0, sizeof(g));
        if (l == 1) fill_first<T>(P, a.x_cols, c0, nc_max, &g.A);
        else if (gated) fill_act<T>(P, reinterpret_cast<const T*>(ws + cv.gt[l - 1]), P->ld[l - 1], nc_max, A_PLAIN, &g.A);
        else {
          fill_act<T>(P, reinterpret_cast<const T*>(ws + cv.z[l - 1]), P->ld[l - 1], nc_max, A_ACT, &g.A, l - 1);
          set_actp(&g.A, l - 1);
        }
        g.J = P->J;
        g.Zbar = zbar_cur;
        g.ldzb = zbar_ld;
        g.zbplane = (long long)nc_max * zbar_ld;
        g.Kdim = s.widths[l - 1];
        g.Nout = s.widths[l];
        g.dW = grads + P->w_off[l];
        g.db = grads + P->b_off[l];
        g.Np = nc;
        g.PT = PT;
        const unsigned kt = (unsigned)((g.Kdim + TM - 1) / TM), nt = (unsigned)((g.Nout + TN - 1) / TN);
        const long long total_chunks = (nc + PT - 1) / PT;
        long long want = (4LL * P->num_sms + kt * nt - 1) / (kt * nt);
        if (want < 1) want = 1;
        if (want > total_chunks) want = total_chunks;
        const long long cps = (total_chunks + want - 1) / want;
        const unsigned splits = (unsigned)((total_chunks + cps - 1) / cps);
        g.chunks_per_split = (int)cps;
        {
          ProfScope ps_(P, CLS_DW, st);
          PPSCI_LAUNCH(kw, dim3(kt, nt, splits), dim3(NTHREADS), smem_w, st, g);
          P->launches++;
        }
        if (gated && l == 1) {  // dWu, dbu, dWv, dbv from the adjoints the gates accumulated
          unsigned kt_e = kt, nt_e = nt;
          if (emb) {
            fill_act<T>(P, reinterpret_cast<const T*>(ws + cv.gt[1]), P->ld[1], nc_max, A_PLAIN, &g.A);
            g.Kdim = s.widths[1];
            g.Nout = s.widths[2];
            kt_e = (unsigned)((g.Kdim + TM - 1) / TM);
            nt_e = (unsigned)((g.Nout + TN - 1) / TN);
          }
          for (int e = 0; e < 2; ++e) {
            g.Zbar = reinterpret_cast<const T*>(ws + (e == 0 ? cv.zub : cv.zvb));
            g.ldzb = P->ld[emb + 1];
            g.zbplane = (long long)nc_max * P->ld[emb + 1];
            g.dW = grads + P->gate_w_off[e];
            g.db = grads + P->gate_b_off[e];
            ProfScope ps_(P, CLS_DW, st);
            PPSCI_LAUNCH(kw, dim3(kt_e, nt_e, splits), dim3(NTHREADS), smem_w, st, g);
            P->launches++;
          }
        }
      }
      if (l == 1) break;
      if (fdx && l <= L - 1) {  // Zbar_{l-1} was produced by the fused chain
        zbar_cur = reinterpret_cast<const T*>(ws + cv.zb[l - 1]);
        zbar_ld = P->ld[l - 1];
        continue;
      }
      if constexpr (sizeof(T) == 4) {
        if (P->use_tc && (P->tc_mask & 2) && tc_dx_ok(s, l)) {
          tc::TcDxArgs t;
          memset(&t, 0, sizeof(t));
          fill_act<float>(P, reinterpret_cast<const float*>(zbar_cur), zbar_ld, nc_max, A_PLAIN, &t.A);
          t.J = P->J;
          t.Wimg = reinterpret_cast<const float*>(ws + cv.tc + tc_imgT_offset(s, l));
          t.Kdim = s.widths[l];
          t.Nout = s.widths[l - 1];
          t.Zprev = reinterpret_cast<const float*>(ws + cv.z[l - 1]);
          t.ldz = P->ld[l - 1];
          t.zplane = (long long)nc_max * P->ld[l - 1];
          t.act = s.act;
          float* outp = reinterpret_cast<float*>(zbar_dst(l - 1));
          t.Out = outp;
          t.ldo = P->ld[l - 1];
          t.oplane = (long long)nc_max * P->ld[l - 1];
          t.Np = nc;
          t.TP = TP;
          t.num_tiles = (int)ptiles;
          t.dbg = debug_timeline_ptr(2);
          const int lay_x = tc_pick_layout(P->J, s.act);
          if ((P->tc_mask & 16) && lay_x != TC_LAY_DYN && P->num_sms >= 2) {  // CTA pairs (cta_group::2)
            const int smem2 = tc::tc2_smem_bytes(t.Nout);
            const unsigned tile_pairs = (ptiles + 1) / 2, sm_pairs = (unsigned)P->num_sms / 2;
            const unsigned gridx2 = 2 * (tile_pairs < sm_pairs ? tile_pairs : sm_pairs);
            ProfScope ps_(P, CLS_DX, st);
            PPSCI_TC2_LAUNCH(k_tc2_dx, lay_x, dim3(gridx2), smem2, st, t,
                             return fail(std::string("cudaFuncSetAttribute(k_tc2_dx): ") + cudaGetErrorString(e_)));
            P->launches++;
          } else {
          const int smem_tc = tc::tc_fwd_smem_bytes(t.Nout);
          const unsigned gridx = ptiles < (unsigned)P->num_sms ? ptiles : (unsigned)P->num_sms;
          {
            ProfScope ps_(P, CLS_DX, st);
            PPSCI_TC_LAUNCH(k_tc_dx, tc_pick_layout(P->J, s.act), KMAX, dim3(gridx), smem_tc, st, t,
                            return fail(std::string("cudaFuncSetAttribute(k_tc_dx): ") + cudaGetErrorString(e_)));
            P->launches++;
          }
          }
          zbar_cur = reinterpret_cast<const T*>(outp);
          zbar_ld = P->ld[l - 1];
          flip ^= 1;
          continue;
        }
      }
      {  // Zbar_{l-1}
        GemmArgs<T> g;
        memset(&g, 0, sizeof(g));
        fill_act<T>(P, zbar_cur, zbar_ld, nc_max, A_PLAIN, &g.A);
        g.J = P->J;
        g.B = reinterpret_cast<const T*>(ws + cv.wt[l]);  // [N_l][K_l]
        g.Kdim = s.widths[l];
        g.Nout = s.widths[l - 1];
        g.ldb = s.widths[l - 1];
        g.bias = nullptr;
        T* outp = zbar_dst(l - 1);
        g.Out = outp;
        g.ldo = P->ld[l - 1];
        g.oplane = (long long)nc_max * P->ld[l - 1];
        g.Np = nc;
        g.TP = TP;
        g.Zprev = reinterpret_cast<const T*>(ws + cv.z[l - 1]);
        g.ldz = P->ld[l - 1];
        g.zplane = (long long)nc_max * P->ld[l - 1];
        g.act = gated ? (int)PPSCI_ACT_IDENTITY : act_of_layer(s, l - 1);  // gated: Gbar_{l-1}, the gate's adjoint follows
        if (!gated && P->actp_off[l - 1] >= 0) {  // trainable activation parameter: dLoss/dbeta comes out of this epilogue
          g.act_param = params + P->actp_off[l - 1];
          g.act_param_grad = grads + P->actp_off[l - 1];
          g.act_pstride = P->actp_stride;
        }
        dim3 grid(ptiles, (unsigned)((g.Nout + TN - 1) / TN));
        {
          ProfScope ps_(P, CLS_DX, st);
          PPSCI_LAUNCH(kx, grid, dim3(NTHREADS), smem_x, st, g);
          P->launches++;
        }
        if (gated && emb && l == 2) {  // layer 1's output also feeds the embeddings: += Zubar Wu^T + Zvbar Wv^T
          for (int e = 0; e < 2; ++e) {
            fill_act<T>(P, reinterpret_cast<const T*>(ws + (e == 0 ? cv.zub : cv.zvb)), P->ld[2], nc_max, A_PLAIN, &g.A);
            g.B = reinterpret_cast<const T*>(ws + (e == 0 ? cv.wtu : cv.wtv));
            g.accum = 1;
            ProfScope ps_(P, CLS_DX, st);
            PPSCI_LAUNCH(kx, grid, dim3(NTHREADS), smem_x, st, g);
            P->launches++;
          }
        }
        if (gated) {  // adjoint of what follows layer l-1, in place: operand adjoint -> Zbar_{l-1}
          const long long tot = (long long)nc * s.widths[l - 1];
          ProfScope ps_(P, CLS_MISC, st);
          if (post_kind(l - 1) == 0) {  // gate; the adjoints of the embeddings' pre-activations accumulate
            GateArgs<T> ga;
            fill_gate(l - 1, nc, &ga);
            ga.G = outp;
            ga.Zub = reinterpret_cast<T*>(ws + cv.zub);
            ga.Zvb = reinterpret_cast<T*>(ws + cv.zvb);
            ga.first = (l - 1 == (pirate ? L - 2 : L - 1)) ? 1 : 0;
            PPSCI_LAUNCH(kgb, dim3((unsigned)((tot + 127) / 128)), dim3(128), 0, st, ga);
          } else {  // adaptive residual of a block (dLoss/dalpha reduced here), or the embedding layer's activation
            MixArgs<T> ma;
            fill_mix(l - 1, nc, &ma);
            ma.X = outp;
            ma.Xres = reinterpret_cast<T*>(ws + cv.xres);
            if (post_kind(l - 1) == 1) {
              ma.alpha_grad = grads + P->alpha_off + (l - 3) / 3;
              ma.use_res = (l - 1 != L - 1) ? 1 : 0;  // the last block's output feeds the output layer only
              ma.write_res = 1;
            } else {
              ma.use_res = pirate ? 1 : 0;  // block 0's residual path
            }
            const long long want = (tot + 127) / 128, cap = 8LL * P->num_sms;
            PPSCI_LAUNCH(kmb, dim3((unsigned)(want < cap ? want : cap)), dim3(128), 0, st, ma);
          }
          P->launches++;
        }
        zbar_cur = outp;
        zbar_ld = P->ld[l - 1];
        flip ^= 1;
      }
    }
  }
  if (a.want_loss && a.loss_out && s.n_res > 0) {
    auto kfin = k_finalize_loss<T>;
    ProfScope ps_(P, CLS_MISC, st);
    PPSCI_LAUNCH(kfin, dim3(1), dim3(32), 0, st, loss_acc, reinterpret_cast<T*>(a.loss_out), s.n_res);
    P->launches++;
  }
  CK(cudaGetLastError());
  return 0;
}

template <typename T>
static int dispatch_k(ppsci_plan* P, const CallArgs& a) {
  if (P->kmax <= 1) return run<T, 1>(P, a);
  if (P->kmax == 2) return run<T, 2>(P, a);
  return run<T, 4>(P, a);
}

static int dispatch(ppsci_plan* P, const CallArgs& a) {
  if (!P) return fail("null plan");
  if (a.n_points <= 0) return fail("n_points must be positive");
  if (!a.x_cols || !a.params || !a.workspace) return fail("null x_cols / params / workspace");
  for (int i = 0; i < P->spec.n_in; ++i)
    if (!a.x_cols[i]) return fail("null input column " + std::to_string(i));
  if (P->spec.n_aux > 0) {
    if (!a.aux_cols) return fail("plan needs aux columns but aux_cols is null");
    for (int i = 0; i < P->spec.n_aux; ++i)
      if (!a.aux_cols[i]) return fail("null aux column " + std::to_string(i));
  }
  if (P->spec.dtype == PPSCI_F64) return dispatch_k<double>(P, a);
  return dispatch_k<float>(P, a);
}

extern "C" int ppsci_b200_plan_set_aux_grad(ppsci_plan* plan, int32_t aux_index, double* grad_dev) {
  if (!plan) return fail("null plan");
  if (aux_index < 0 || aux_index >= plan->spec.n_aux || !plan->spec.aux_bcast[aux_index])
    return fail("plan_set_aux_grad: aux_index is not a learnable (broadcast) parameter of this plan");
  plan->aux_grad[aux_index] = grad_dev;
  return 0;
}

extern "C" int ppsci_b200_values_fwd_bwd(ppsci_plan* plan, const void* const* x_cols, const void* const* aux_cols,
                                         int64_t n_points, const void* params, void* grads, const void* ybar,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  if (!ybar || !grads) return fail("values_fwd_bwd: null ybar / grads");
  CallArgs a;
  memset(&a, 0, sizeof(a));
  a.x_cols = x_cols;
  a.aux_cols = aux_cols;
  a.n_points = n_points;
  a.n_norm = n_points;
  a.params = params;
  a.grads = grads;
  a.workspace = workspace;
  a.workspace_bytes = workspace_bytes;
  a.stream = stream;
  a.want_loss = false;
  a.ybar_in = ybar;
  return dispatch(plan, a);
}

extern "C" int ppsci_b200_residual_loss_fwd_bwd(ppsci_plan* plan, const void* const* x_cols,
                                                const void* const* aux_cols, const void* const* label_cols,
                                                const double* label_const, const void* const* weight_cols,
                                                int64_t n_points, int64_t n_norm, const void* params, void* grads,
                                                void* loss_out, void* const* residual_out, void* workspace,
                                                size_t workspace_bytes, void* stream) {
  if (plan && plan->spec.n_res < 1) return fail("residual_loss_fwd_bwd: plan has no residuals");
  if (!loss_out) return fail("residual_loss_fwd_bwd: loss_out is null");
  if (n_norm <= 0) return fail("residual_loss_fwd_bwd: n_norm must be positive");
  CallArgs a{x_cols, aux_cols, label_cols, label_const, weight_cols, n_points, n_norm, params, grads, loss_out,
             residual_out, nullptr, workspace, workspace_bytes, stream, true};
  return dispatch(plan, a);
}

extern "C" int ppsci_b200_residual_fwd(ppsci_plan* plan, const void* const* x_cols, const void* const* aux_cols,
                                       int64_t n_points, const void* params, void* jets_out,
                                       void* const* residual_out, void* workspace, size_t workspace_bytes,
                                       void* stream) {
  CallArgs a{x_cols, aux_cols, nullptr, nullptr, nullptr, n_points, 1, params, nullptr, nullptr,
             residual_out, jets_out, workspace, workspace_bytes, stream, false};
  return dispatch(plan, a);
}

extern "C" int32_t ppsci_b200_plan_chunk_points(const ppsci_plan* P) { return P ? P->chunk : -1; }

extern "C" int ppsci_b200_values_fwd_keep(ppsci_plan* plan, const void* const* x_cols, const void* const* aux_cols, int64_t n_points,
                                          const void* params, void* y_out, void* workspace, size_t workspace_bytes, void* stream) {
  // y_out may be NULL: the caller then reads the outputs in place, [n_points][ld] at plan_stash_offset(n_layers) of the
  // workspace (no copy; ld = n_out rounded up to a multiple of 4)
  if (plan && n_points > plan->chunk) return fail("values_fwd_keep: at most plan_chunk_points points per call");
  CallArgs a;
  memset(&a, 0, sizeof(a));
  a.x_cols = x_cols;
  a.aux_cols = aux_cols;
  a.n_points = n_points;
  a.n_norm = n_points;
  a.params = params;
  a.jets_out = y_out;  // C = 1: [n_points][n_out]
  a.workspace = workspace;
  a.workspace_bytes = workspace_bytes;
  a.stream = stream;
  a.phase = 1;
  if (plan && plan->C != 1) return fail("values_fwd_keep: the plan must have no input derivatives (C == 1)");
  return dispatch(plan, a);
}

extern "C" int ppsci_b200_values_bwd_kept(ppsci_plan* plan, const void* const* x_cols, const void* const* aux_cols, int64_t n_points,
                                          const void* params, void* grads, const void* ybar, void* workspace,
                                          size_t workspace_bytes, void* stream) {
  if (!ybar || !grads) return fail("values_bwd_kept: null ybar / grads");
  CallArgs a;
  memset(&a, 0, sizeof(a));
  a.x_cols = x_cols;
  a.aux_cols = aux_cols;
  a.n_points = n_points;
  a.n_norm = n_points;
  a.params = params;
  a.grads = grads;
  a.workspace = workspace;
  a.workspace_bytes = workspace_bytes;
  a.stream = stream;
  a.ybar_in = ybar;
  a.phase = 2;
  return dispatch(plan, a);
}

extern "C" int ppsci_b200_deeponet_head(int32_t dtype, int32_t act, const void* b, const void* t, const void* bias,
                                        const void* label, const void* weight, int64_t n, int32_t n_features, double coef,
                                        void* g_out, double* loss_acc, void* bbar, void* tbar, void* dbias, void* stream) {
  if (!b || !t || n <= 0 || n_features <= 0) return fail("deeponet_head: bad arguments");
  if ((bbar == nullptr) != (tbar == nullptr)) return fail("deeponet_head: bbar and tbar must both be given or both be null");
  if (act < 0 || act > PPSCI_ACT_LAST) return fail("deeponet_head: unknown activation");
  if (act_has_param(act)) return fail("deeponet_head: activations with a trainable parameter are not offered here");
  const long long warps = n < 148LL * 64 ? n : 148LL * 64;  // 8 warps per block
  const unsigned blocks = (unsigned)((warps + 7) / 8);
  if (dtype == PPSCI_F64) {
    auto k = k_deeponet_head<double>;
    PPSCI_LAUNCH(k, dim3(blocks), dim3(256), 0, stream, (const double*)b, (const double*)t, (const double*)bias, act,
                 (const double*)label, (const double*)weight, (long long)n, n_features, coef, (double*)g_out, loss_acc,
                 (double*)bbar, (double*)tbar, (double*)dbias);
  } else if (dtype == PPSCI_F32) {
    auto k = k_deeponet_head<float>;
    PPSCI_LAUNCH(k, dim3(blocks), dim3(256), 0, stream, (const float*)b, (const float*)t, (const float*)bias, act,
                 (const float*)label, (const float*)weight, (long long)n, n_features, coef, (float*)g_out, loss_acc,
                 (float*)bbar, (float*)tbar, (float*)dbias);
  } else {
    return fail("deeponet_head: bad dtype");
  }
  CK(cudaGetLastError());
  return 0;
}

extern "C" int ppsci_b200_sample_uniform(int32_t dtype, uint64_t seed, uint64_t offset, int64_t n, int32_t ndim, const double* lo,
                                         const double* hi, void* const* out_cols, void* stream) {
  if (n <= 0 || ndim < 1 || ndim > PPSCI_MAX_IN || !lo || !hi || !out_cols) return fail("sample_uniform: bad arguments");
  SampleArgs a;
  memset(&a, 0, sizeof(a));
  for (int d = 0; d < ndim; ++d) {
    if (!out_cols[d]) return fail("sample_uniform: null output column");
    a.cols[d] = out_cols[d];
    a.lo[d] = lo[d];
    a.hi[d] = hi[d];
  }
  a.ndim = ndim;
  a.n = n;
  a.seed = seed;
  a.offset = offset;
  const unsigned blocks = (unsigned)((n + 255) / 256);
  if (dtype == PPSCI_F64) {
    auto k = k_sample_uniform<double>;
    PPSCI_LAUNCH(k, dim3(blocks), dim3(256), 0, stream, a);
  } else if (dtype == PPSCI_F32) {
    auto k = k_sample_uniform<float>;
    PPSCI_LAUNCH(k, dim3(blocks), dim3(256), 0, stream, a);
  } else {
    return fail("sample_uniform: bad dtype");
  }
  CK(cudaGetLastError());
  return 0;
}

extern "C" int ppsci_b200_adam_step(int32_t dtype, void* params, const void* grads, void* exp_avg, void* exp_avg_sq,
                                    int64_t n, double lr, double beta1, double beta2, double eps, double weight_decay,
                                    int64_t step, double grad_scale, void* stream) {
  if (!params || !grads || !exp_avg || !exp_avg_sq || n <= 0 || step < 1) return fail("adam_step: bad arguments");
  const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
  const unsigned blocks = (unsigned)((n + 255) / 256);
  if (dtype == PPSCI_F64) {
    auto k = k_adam<double>;
    PPSCI_LAUNCH(k, dim3(blocks), dim3(256), 0, stream, (double*)params, (const double*)grads, (double*)exp_avg,
                 (double*)exp_avg_sq, (long long)n, lr, beta1, beta2, eps, weight_decay, bc1, bc2, grad_scale);
  } else if (dtype == PPSCI_F32) {
    auto k = k_adam<float>;
    PPSCI_LAUNCH(k, dim3(blocks), dim3(256), 0, stream, (float*)params, (const float*)grads, (float*)exp_avg,
                 (float*)exp_avg_sq, (long long)n, lr, beta1, beta2, eps, weight_decay, bc1, bc2, grad_scale);
  } else {
    return fail("adam_step: bad dtype");
  }
  CK(cudaGetLastError());
  return 0;
}

extern "C" int ppsci_b200_adam_step_dev(int32_t dtype, void* params, void* grads, void* exp_avg, void* exp_avg_sq,
                                        int64_t n, const double* hyper_dev, double beta1, double beta2, double eps,
                                        double weight_decay, int32_t zero_grads, void* stream) {
  if (!params || !grads || !exp_avg || !exp_avg_sq || !hyper_dev || n <= 0) return fail("adam_step_dev: bad arguments");
  const unsigned blocks = (unsigned)((n + 255) / 256);
  if (dtype == PPSCI_F64) {
    auto k = k_adam_dev<double>;
    PPSCI_LAUNCH(k, dim3(blocks), dim3(256), 0, stream, (double*)params, (double*)grads, (double*)exp_avg,
                 (double*)exp_avg_sq, (long long)n, hyper_dev, beta1, beta2, eps, weight_decay, (int)zero_grads);
  } else if (dtype == PPSCI_F32) {
    auto k = k_adam_dev<float>;
    PPSCI_LAUNCH(k, dim3(blocks), dim3(256), 0, stream, (float*)params, (float*)grads, (float*)exp_avg,
                 (float*)exp_avg_sq, (long long)n, hyper_dev, beta1, beta2, eps, weight_decay, (int)zero_grads);
  } else {
    return fail("adam_step_dev: bad dtype");
  }
  CK(cudaGetLastError());
  return 0;
}

// a_l is stashed by the tensor-core forward of layer l+1 and consumed by the tensor-core dW of layer l+1
static bool tc_astash_needed(const ppsci_plan* P, int l) {
  const int lay = l + 1;
  return P->use_tc && (P->tc_mask & 1) && (P->tc_mask & 4) && lay <= P->spec.n_layers && tc_layer_ok(P->spec, lay) &&
         tc_dw_ok(P->spec, lay);
}
static size_t tc_scratch_bytes(const ppsci_plan* P, int64_t nc) {
  return P->use_tc ? tc_scratch_bytes_impl(P->spec, P->C, nc) : 0;
}

// layer-fused forward: fp32 tanh, one of the static jet layouts, at least one hidden -> hidden layer, all hidden
// widths equal (K = N = H, a multiple of 32 up to 256)
static bool fused_fwd_ok(const ppsci_plan* P) {
  const ppsci_plan_spec& s = P->spec;
  const int L = s.n_layers;
  if (!P->use_tc || !(P->tc_mask & 1) || !(P->tc_mask & 8) || !(P->tc_mask & 64) || P->num_sms < 2) return false;
  if (L < 3 || L - 2 > tc::FUSE_MAXL) return false;
  if (tc_pick_layout(P->J, s.act) == TC_LAY_DYN) return false;
  for (int l = 2; l < L; ++l)
    if (!tc_layer_ok(s, l) || s.widths[l] != s.widths[1]) return false;
  // Accuracy gate.  The fused forward double-buffers ONE accumulator per layer (2 x 256 TMEM columns), i.e. all 12
  // round-toward-zero accumulations of a 32-wide chunk land in the big accumulator: measured on cfg3 (6 x 256) the
  // residual error is 1.3e-5 against 4.4e-6 for the layer-at-a-time kernels, whose exact-product | cross-term split
  // needs all 512 columns.  Up to 128-wide layers the contraction is short enough (cfg2: 1.8e-6) and the fused kernel is
  // the default; wider layers take it only on request (PPSCI_B200_TC_MASK bit 8).  The dx chain has no such gate: its
  // rounding only enters the weight gradient (cfg3: 1.1e-5 against a 5e-5 tolerance).
  if (s.widths[1] > 128 && !(P->tc_mask & 256)) return false;
  return s.widths[1] <= 256;
}

// layer-fused dx chain: same shape constraints as the fused forward, dx of every hidden -> hidden layer tensor-core eligible
static bool fused_dx_ok(const ppsci_plan* P) {
  const ppsci_plan_spec& s = P->spec;
  const int L = s.n_layers;
  if (!P->use_tc || !(P->tc_mask & 2) || !(P->tc_mask & 16) || !(P->tc_mask & 128) || P->num_sms < 2) return false;
  if (L < 3 || L - 2 > tc::FUSE_MAXL) return false;
  if (tc_pick_layout(P->J, s.act) == TC_LAY_DYN) return false;
  for (int l = 2; l < L; ++l)
    if (!tc_dx_ok(s, l) || s.widths[l] != s.widths[1]) return false;
  return s.widths[1] <= 256;
}

// fp16-operand fused forward (k_fused_fwd16): the shape constraints of the fused forward, width a multiple of 64, at
// least two fused layers; the default for layers wider than 128 (where the single tf32 accumulator is not accurate
// enough), on request (PPSCI_B200_TC_MASK bit 9) for narrower ones
static bool fused_fwd16_ok(const ppsci_plan* P) {
  const ppsci_plan_spec& s = P->spec;
  const int L = s.n_layers;
  if (!P->use_tc || !(P->tc_mask & 1) || !(P->tc_mask & 8) || !(P->tc_mask & 64) || P->num_sms < 2) return false;
  if (L < 4 || L - 2 > tc::FUSE_MAXL) return false;
  if (tc_pick_layout(P->J, s.act) == TC_LAY_DYN || s.act != PPSCI_ACT_TANH) return false;
  for (int l = 2; l < L; ++l)
    if (!tc_layer_ok(s, l) || s.widths[l] != s.widths[1]) return false;
  if (s.widths[1] % 64 != 0 || s.widths[1] > 256) return false;
  if (P->tc_mask & 256) return false;  // bit 8: force the tf32 fused forward (cross-check)
  return s.widths[1] > 128 || (P->tc_mask & 512);
}
