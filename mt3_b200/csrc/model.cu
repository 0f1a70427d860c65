// Host orchestration of the MT3 encoder / decoder on sm_100a behind the C ABI.
//
// Reference semantics: network.py:44-85 (EncoderLayer), :88-155 (DecoderLayer), :158-193
// (Encoder), :196-262 (Decoder), :275-361 (Transformer.encode/decode); layers.py for the ops.
// Data layout in HBM (all fp32, row-major):
//   hidden h        [B*T, D]
//   qkv             [B*T, 3Q]   columns [q | k | v], each (head, 64)
//   cross K/V       [Ld][B][K|V][H][T][64]  head-major, fp32 or fp16 (hoisted: computed once per batch)
//   self K/V cache  [Ld][B][K|V][H][L][64]  head-major, fp32 or fp16 (append = 12 rows of 64 per sequence per layer)
// The reference's [B,H,D,L] cache layout (layers.py:249-260) is a TPU scatter trick; the
// ABI exposes tokens and logits, not the cache, so the layout is ours.
#include <string.h>
#include <math.h>
#include <string>
#include <vector>
#include <map>
#include <tuple>

#include "common.cuh"
#include "gemm_simt.cuh"
#include "gemm_tc.cuh"
#include "attention_tc.cuh"
#include "decode.cuh"
#include "layers.cuh"

namespace mt3 {

struct ParamEntry { std::string name; int64_t rows, cols, offset; };

static std::vector<ParamEntry> param_table(const mt3_model_config& c) {
  std::vector<ParamEntry> t;
  int64_t off = 0;
  auto add = [&](const std::string& n, int64_t r, int64_t co) {
    t.push_back({n, r, co, off});
    off += r * co;
  };
  const int64_t D = c.emb_dim, Q = (int64_t)c.num_heads * c.head_dim, F = c.mlp_dim, V = c.vocab_size;
  add("encoder/continuous_inputs_projection/kernel", c.input_depth, D);
  for (int i = 0; i < c.num_encoder_layers; ++i) {
    const std::string p = "encoder/layers_" + std::to_string(i) + "/";
    add(p + "pre_attention_layer_norm/scale", 1, D);
    add(p + "attention/query/kernel", D, Q);
    add(p + "attention/key/kernel", D, Q);
    add(p + "attention/value/kernel", D, Q);
    add(p + "attention/out/kernel", Q, D);
    add(p + "pre_mlp_layer_norm/scale", 1, D);
    add(p + "mlp/wi_0/kernel", D, F);
    add(p + "mlp/wi_1/kernel", D, F);
    add(p + "mlp/wo/kernel", F, D);
  }
  add("encoder/encoder_norm/scale", 1, D);
  add("decoder/token_embedder/embedding", V, D);
  for (int i = 0; i < c.num_decoder_layers; ++i) {
    const std::string p = "decoder/layers_" + std::to_string(i) + "/";
    add(p + "pre_self_attention_layer_norm/scale", 1, D);
    add(p + "self_attention/query/kernel", D, Q);
    add(p + "self_attention/key/kernel", D, Q);
    add(p + "self_attention/value/kernel", D, Q);
    add(p + "self_attention/out/kernel", Q, D);
    add(p + "pre_cross_attention_layer_norm/scale", 1, D);
    add(p + "encoder_decoder_attention/query/kernel", D, Q);
    add(p + "encoder_decoder_attention/key/kernel", D, Q);
    add(p + "encoder_decoder_attention/value/kernel", D, Q);
    add(p + "encoder_decoder_attention/out/kernel", Q, D);
    add(p + "pre_mlp_layer_norm/scale", 1, D);
    add(p + "mlp/wi_0/kernel", D, F);
    add(p + "mlp/wi_1/kernel", D, F);
    add(p + "mlp/wo/kernel", F, D);
  }
  add("decoder/decoder_norm/scale", 1, D);
  add("decoder/logits_dense/kernel", D, V);
  return t;
}

// K-major ("transposed", [N,K]) copy of a prepared weight for the tcgen05 path, optionally tf32 hi/lo split.
struct TcW { float* hi = nullptr; float* lo = nullptr; TcOperand op; int K = 0, N = 0; };
// An activation buffer [rows, ld]; lo != null when it is carried as a tf32 hi/lo pair.
struct Act { float* hi = nullptr; float* lo = nullptr; TcOperand op; };

struct EncLayer { float *wqkv, *wo, *wi, *wo2; TcW t_wqkv, t_wo, t_wi, t_wo2; };
struct DecLayer { float *wqkv, *wo, *wq_c, *wkv_c, *wo_c, *wi, *wo2; float* wc1 = nullptr; TcW t_wkv_c; };   // wc1: [Q+D, Q] = [Wo.Wq ; Wq]

struct Model {
  mt3_model_config cfg;
  int D, H, Q, F, V, Le, Ld, L;
  float* slab = nullptr;          // all prepared weights
  float* slab_tc = nullptr;       // K-major (and hi/lo) copies for the tcgen05 path
  bool fuse_q = true;             // MT3_DEC_FUSE=0: keep the self-attention out-projection and the cross-attention query
                                  // projection as two launches (default: one launch with a precomposed weight block)
  float *dy2 = nullptr, *dssq = nullptr;   // second residual-stream buffer (ping-pong) and [B][D/32] sum-of-squares partials
  bool tc = false, split3 = false;
  TcW t_w_in;
  Act a_x, a_h, a_ao, a_g, a_enc, a_qkv, a_vt; // tcgen05-path activation buffers (workspace); a_vt = per-head V^T
  bool pdl = false;               // MT3_PDL=1: programmatic dependent launch between all decode-step kernels
  bool pdl_attn = true;           // MT3_PDL=2 (default): only the attention launches (K/V prefetch under the preceding GEMM)
  bool pdl_gemm = false;          // MT3_PDL=4: only the GEMM launches; bits combine (6 = attention + GEMM); 0 = off
  bool dec_cluster = true;        // MT3_DEC_CLUSTER=0: split-K reduction through global scratch instead of DSMEM
  int pf_attn = 16;               // MT3_PF_ATTN=n: the decode-step attention kernels prefetch the n K/V tiles that follow their
                                  // shared-memory ring into L2 while they wait under the preceding GEMM (decode.cuh; value-neutral;
                                  // 0 = off: 449.6 -> 442.3 ms per batch at 16, profiles/r02_call63_ab_l2_prefetch.txt)
  int dec_pipe = 3;               // MT3_DEC_PIPE bits of the cluster decode GEMM (decode.cuh dec_cluster_body): 1 = staged
                                  // operand loads, 2 = exchange by bulk DSMEM copies, 0 = neither; bit-identical results
                                  // (0 -> 3: 453.6 -> 428.8 ms per batch on a B200, profiles/r03_call3_bench_*)
  int kv_fmt = 0;                 // cfg.kv_cache_format: storage format of the self and cross K/V rows (kv_dest())
  int kv_row = 256;               // bytes per K/V row of 64 elements
  // debug timeline (mt3_debug_trace_step): while `tracing` is set every decode GEMM / attention launch gets a slot
  unsigned long long* trace = nullptr;
  bool tracing = false;
  std::vector<std::string> trace_names;
  bool tc_attn_ok = true;         // MT3_TC_ATTENTION=0 in the environment forces the exact-fp32 attention kernel
  float* w_in = nullptr;
  std::vector<EncLayer> enc;
  float* enc_norm_g = nullptr;
  float* emb = nullptr;
  std::vector<DecLayer> dec;
  float* w_logits = nullptr;
  float* pe = nullptr;            // [2048, D] sinusoid table (FixedEmbed.max_length, layers.py:565)
  int pe_rows = 2048;

  // workspace (caller-owned)
  char* ws = nullptr;
  int64_t ws_bytes = 0;
  int B = 0, T = 0;
  float *h = nullptr, *rstd = nullptr, *qkv = nullptr, *ao = nullptr, *g = nullptr, *encoded = nullptr;
  char *ckv = nullptr, *skv = nullptr;   // head-major K/V rows (kv_row bytes each)
  float *dy = nullptr, *drstd = nullptr, *dq = nullptr, *dao = nullptr, *dg = nullptr, *dlogits = nullptr;
  int *tok_cur = nullptr, *finished = nullptr, *tokens = nullptr, *state = nullptr;
  float* att_scratch = nullptr;   // key-split encoder attention (T > 256): unnormalised O parts + (max, sum) pairs
  float* beam_f = nullptr; int* beam_i = nullptr;   // beam-size-1 search state (MT3_GEN_BEAM1)
  float* dpartial = nullptr;      // split-K scratch of the non-cluster decode GEMM
  int dcounters_n = 0;
  int* dcounters = nullptr;
  int sm_count = 148;
  bool have_cross = false;
  int host_pos = 0;               // host mirror of the device position (cache overflow guard)

  // CUDA graph of one greedy step
  cudaStream_t cap_stream = nullptr;
  cudaGraph_t graph = nullptr;              // the graph of the CURRENT (workspace, B, T) binding ...
  cudaGraphExec_t graph_exec = nullptr;
  uint64_t graph_kernels = 0;
  int graph_mode = 1;
  struct StepGraph { cudaGraph_t g; cudaGraphExec_t e; uint64_t kernels; };
  std::map<std::tuple<const void*, int, int, int>, StepGraph> graphs;   // ... kept per binding, so that a short tail batch does not
                                                                   // throw away the full batch's graph (and vice versa)
  int* h_flag = nullptr;          // pinned
};

// byte address of layer l's K/V block: [B][K|V][H][cap] rows of kv_row bytes
static char* kv_layer(const Model* m, char* base, int l, int cap) {
  return base + (int64_t)l * m->B * cap * 2 * m->H * m->kv_row;
}

static int64_t prepared_floats(const mt3_model_config& c) {
  const int64_t D = c.emb_dim, Q = (int64_t)c.num_heads * c.head_dim, F = c.mlp_dim, V = c.vocab_size;
  int64_t n = (int64_t)c.input_depth * D;
  n += (int64_t)c.num_encoder_layers * (D * 3 * Q + Q * D + D * 2 * F + F * D);
  n += D;          // encoder_norm
  n += V * D;      // embedding
  n += (int64_t)c.num_decoder_layers * (D * 3 * Q + Q * D + D * Q + D * 2 * Q + Q * D + D * 2 * F + F * D);
  n += D * V;      // logits
  n += (int64_t)c.num_decoder_layers * (Q + D) * Q;   // precomposed [Wo.Wq ; Wq] blocks
  n += 2048 * D;   // PE
  return n;
}

// out [Q + D, Q]: rows [0, Q) = Wo [Q, D] . Wq [D, Q] accumulated in fp64 and rounded once; rows [Q, Q + D) = Wq.
// (q = rstd . (y + o.Wo) . Wq  =  rstd . ([o | y] . out): the out-projection folded into the query projection.)
__global__ void compose_out_q_kernel(const float* __restrict__ wo, const float* __restrict__ wq, int Q, int D, float* __restrict__ out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
  if (j >= Q) return;
  if (i < Q) {
    double acc = 0.0;
    for (int k = 0; k < D; ++k) acc += (double)wo[(long long)i * D + k] * (double)wq[(long long)k * Q + j];
    out[(long long)i * Q + j] = (float)acc;
  } else {
    out[(long long)i * Q + j] = wq[(long long)(i - Q) * Q + j];
  }
}

static int prep_copy(cudaStream_t s, const float* src, int K, int N, const float* g, float* dst, int ldd, int col_off,
                     int col_stride) {
  const long long n = (long long)K * N;
  scale_copy_cols_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, K, N, g, dst, ldd, col_off, col_stride);
  MT3_LAUNCH_CHECK();
  return MT3_OK;
}
#define MT3_TRY(expr)            \
  do {                           \
    int _r = (expr);             \
    if (_r != MT3_OK) return _r; \
  } while (0)

static int gemm(Model* m, const GemmArgs& a, cudaStream_t s) {
  (void)m;
  return launch_sgemm(a, s);
}

static GemmArgs gemm_args(const float* A, int lda, const float* B, int ldb, int M, int N, int K, float* C, int ldc) {
  GemmArgs a;
  memset(&a, 0, sizeof(a));
  a.A = A; a.lda = lda; a.B = B; a.ldb = ldb; a.M = M; a.N = N; a.K = K;
  a.C = C; a.ldc = ldc; a.n_split = N; a.epi = EPI_STORE;
  return a;
}

static int launch_rstd(const float* x, int ld, int M, int D, float* rstd, cudaStream_t s) {
  row_rstd_kernel<<<cdiv(M, 8), 256, 0, s>>>(x, nullptr, ld, M, D, 1e-6f, rstd);
  MT3_LAUNCH_CHECK();
  return MT3_OK;
}

static int set_attr_once() {
  static bool done = false;
  if (done) return MT3_OK;
  MT3_CUDA_CHECK(cudaFuncSetAttribute(enc_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  done = true;
  return MT3_OK;
}

static int prep_tc_weight(Model* m, cudaStream_t s, const float* w, int K, int N, float*& cursor, TcW* out) {
  out->K = K; out->N = N;
  out->hi = cursor; cursor += (int64_t)K * N;
  if (m->split3) { out->lo = cursor; cursor += (int64_t)K * N; }
  transpose_split_kernel<<<dim3(cdiv(N, 32), cdiv(K, 32)), dim3(32, 8), 0, s>>>(w, K, N, out->hi, out->lo);
  MT3_LAUNCH_CHECK();
  return make_operand(&out->op, out->hi, out->lo, N, K, K);
}

static int64_t tc_weight_floats(const mt3_model_config& c) {
  const int64_t D = c.emb_dim, Q = (int64_t)c.num_heads * c.head_dim, F = c.mlp_dim;
  int64_t n = (int64_t)c.input_depth * D;
  n += (int64_t)c.num_encoder_layers * (D * 3 * Q + Q * D + D * 2 * F + F * D);
  n += (int64_t)c.num_decoder_layers * (D * 2 * Q);
  return n * (c.gemm_mode == MT3_GEMM_TF32X3 ? 2 : 1);
}

static TcGemmArgs tc_args(int M, int N, int K, float* C_hi, float* C_lo, int ldc) {
  TcGemmArgs a;
  memset(&a, 0, sizeof(a));
  a.M = M; a.N = N; a.K = K; a.C_hi = C_hi; a.C_lo = C_lo; a.ldc = ldc; a.n_split = N; a.epi = EPI_STORE;
  return a;
}

// Encoder on the tcgen05 path.  Activations that feed a GEMM are kept as tf32 hi/lo pairs in TF32X3 mode.
static int encode_tc_impl(Model* m, const float* x, float* encoded, cudaStream_t s) {
  const int M = m->B * m->T, D = m->D, Q = m->Q, F = m->F, depth = m->cfg.input_depth;
  MT3_TRY(set_attr_once());
  TcOperand opx;
  if (m->split3) {
    const long long n4 = (long long)M * depth / 4;
    split_pair_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, s>>>(x, m->a_x.hi, m->a_x.lo, n4);
    MT3_LAUNCH_CHECK();
    opx = m->a_x.op;
  } else {
    MT3_TRY(make_operand(&opx, x, nullptr, M, depth, depth));
  }
  {
    TcGemmArgs a = tc_args(M, D, depth, m->a_h.hi, m->a_h.lo, D);
    a.epi = EPI_ADD_PE; a.pe = m->pe; a.pe_T = m->T; a.pe_ld = D;
    MT3_TRY(launch_tc_gemm(opx, m->t_w_in.op, a, m->split3, s));
  }
  const size_t attn_smem = (size_t)(32 * kHD + 32 * (m->T + 4) + 64 * 68) * sizeof(float);
  MT3_REQUIRE(attn_smem <= 200 * 1024, MT3_ERR_UNSUPPORTED, "encode: input_length %d too long for the attention kernel", m->T);
  const bool tc_attn = m->tc_attn_ok && enc_attention_tc_supported(m->T);
  for (int l = 0; l < m->Le; ++l) {
    const EncLayer& w = m->enc[l];
    row_rstd_kernel<<<cdiv(M, 8), 256, 0, s>>>(m->a_h.hi, m->a_h.lo, D, M, D, 1e-6f, m->rstd);
    MT3_LAUNCH_CHECK();
    {
      // qkv goes out as a tf32 hi/lo pair when the tcgen05 attention kernel consumes it
      TcGemmArgs a = tc_args(M, 3 * Q, D, m->qkv, tc_attn ? m->a_qkv.lo : nullptr, 3 * Q);
      a.row_scale = m->rstd;
      if (tc_attn) {   // the V third goes out transposed per head: the K-major operand of P.V
        a.VT_hi = m->a_vt.hi; a.VT_lo = m->a_vt.lo; a.vt_col0 = 2 * Q; a.vt_T = m->T; a.vt_H = m->H;
      }
      MT3_TRY(launch_tc_gemm(m->a_h.op, w.t_wqkv.op, a, m->split3, s));
    }
    if (tc_attn) {
      MT3_TRY(launch_enc_attention_tc(m->a_qkv.op, m->a_vt.op, m->B, m->T, m->H, m->a_ao.hi, m->a_ao.lo, m->split3, s, nullptr, 0, nullptr,
                                      m->att_scratch));
    } else {
      enc_attention_kernel<<<dim3(cdiv(m->T, 32), m->H, m->B), 256, attn_smem, s>>>(m->qkv, 3 * Q, m->T, m->H, m->a_ao.hi,
                                                                                     m->a_ao.lo, Q);
      MT3_LAUNCH_CHECK();
    }
    {
      TcGemmArgs a = tc_args(M, D, Q, m->a_h.hi, m->a_h.lo, D);
      a.epi = EPI_RESIDUAL; a.R_hi = m->a_h.hi; a.R_lo = m->a_h.lo; a.ldr = D;
      MT3_TRY(launch_tc_gemm(m->a_ao.op, w.t_wo.op, a, m->split3, s));
    }
    row_rstd_kernel<<<cdiv(M, 8), 256, 0, s>>>(m->a_h.hi, m->a_h.lo, D, M, D, 1e-6f, m->rstd);
    MT3_LAUNCH_CHECK();
    {
      TcGemmArgs a = tc_args(M, 2 * F, D, m->a_g.hi, m->a_g.lo, F);
      a.row_scale = m->rstd; a.epi = EPI_GATED_GELU;
      MT3_TRY(launch_tc_gemm(m->a_h.op, w.t_wi.op, a, m->split3, s));
    }
    {
      TcGemmArgs a = tc_args(M, D, F, m->a_h.hi, m->a_h.lo, D);
      a.epi = EPI_RESIDUAL; a.R_hi = m->a_h.hi; a.R_lo = m->a_h.lo; a.ldr = D;
      MT3_TRY(launch_tc_gemm(m->a_g.op, w.t_wo2.op, a, m->split3, s));
    }
  }
  rmsnorm_kernel<<<cdiv(M, 8), 256, 0, s>>>(m->a_h.hi, m->a_h.lo, D, M, D, 1e-6f, m->enc_norm_g, encoded, D);
  MT3_LAUNCH_CHECK();
  return MT3_OK;
}

static int cross_kv_tc_impl(Model* m, const float* encoded, cudaStream_t s) {
  const int M = m->B * m->T, D = m->D, Q = m->Q;
  TcOperand ope;
  if (m->split3) {
    const long long n4 = (long long)M * D / 4;
    split_pair_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, s>>>(encoded, m->a_enc.hi, m->a_enc.lo, n4);
    MT3_LAUNCH_CHECK();
    ope = m->a_enc.op;
  } else {
    MT3_TRY(make_operand(&ope, encoded, nullptr, M, D, D));
  }
  for (int l = 0; l < m->Ld; ++l) {
    TcGemmArgs a = tc_args(M, 2 * Q, D, nullptr, nullptr, 2 * Q);
    a.n_split = 0; a.C1 = kv_layer(m, m->ckv, l, m->T); a.kv_fmt = m->kv_fmt; a.hm_rows_per_b = m->T; a.hm_cap = m->T; a.hm_H = m->H;
    MT3_TRY(launch_tc_gemm(ope, m->dec[l].t_wkv_c.op, a, m->split3, s));
  }
  return MT3_OK;
}

static int encode_impl(Model* m, const float* x, float* encoded, cudaStream_t s) {
  if (m->tc) return encode_tc_impl(m, x, encoded, s);
  const int M = m->B * m->T, D = m->D, Q = m->Q, F = m->F;
  MT3_TRY(set_attr_once());
  {
    GemmArgs a = gemm_args(x, m->cfg.input_depth, m->w_in, D, M, D, m->cfg.input_depth, m->h, D);
    a.epi = EPI_ADD_PE; a.pe = m->pe; a.pe_T = m->T; a.pe_ld = D;
    MT3_TRY(gemm(m, a, s));
  }
  const size_t attn_smem = (size_t)(32 * kHD + 32 * (m->T + 4) + 64 * 68) * sizeof(float);
  MT3_REQUIRE(attn_smem <= 200 * 1024, MT3_ERR_UNSUPPORTED, "encode: input_length %d too long for the attention kernel", m->T);
  for (int l = 0; l < m->Le; ++l) {
    const EncLayer& w = m->enc[l];
    MT3_TRY(launch_rstd(m->h, D, M, D, m->rstd, s));
    {
      GemmArgs a = gemm_args(m->h, D, w.wqkv, 3 * Q, M, 3 * Q, D, m->qkv, 3 * Q);
      a.row_scale = m->rstd;
      MT3_TRY(gemm(m, a, s));
    }
    {
      dim3 grid(cdiv(m->T, 32), m->H, m->B);
      enc_attention_kernel<<<grid, 256, attn_smem, s>>>(m->qkv, 3 * Q, m->T, m->H, m->ao, nullptr, Q);
      MT3_LAUNCH_CHECK();
    }
    {
      GemmArgs a = gemm_args(m->ao, Q, w.wo, D, M, D, Q, m->h, D);
      a.epi = EPI_RESIDUAL; a.R = m->h; a.ldr = D;
      MT3_TRY(gemm(m, a, s));
    }
    MT3_TRY(launch_rstd(m->h, D, M, D, m->rstd, s));
    {
      GemmArgs a = gemm_args(m->h, D, w.wi, 2 * F, M, 2 * F, D, m->g, F);
      a.row_scale = m->rstd; a.epi = EPI_GATED_GELU;
      MT3_TRY(gemm(m, a, s));
    }
    {
      GemmArgs a = gemm_args(m->g, F, w.wo2, D, M, D, F, m->h, D);
      a.epi = EPI_RESIDUAL; a.R = m->h; a.ldr = D;
      MT3_TRY(gemm(m, a, s));
    }
  }
  rmsnorm_kernel<<<cdiv(M, 8), 256, 0, s>>>(m->h, nullptr, D, M, D, 1e-6f, m->enc_norm_g, encoded, D);
  MT3_LAUNCH_CHECK();
  return MT3_OK;
}

static int cross_kv_impl(Model* m, const float* encoded, cudaStream_t s) {
  const int M = m->B * m->T, D = m->D, Q = m->Q;
  if (m->tc) {
    MT3_TRY(cross_kv_tc_impl(m, encoded, s));
  } else {
    for (int l = 0; l < m->Ld; ++l) {
      GemmArgs a = gemm_args(encoded, D, m->dec[l].wkv_c, 2 * Q, M, 2 * Q, D, nullptr, 2 * Q);
      a.n_split = 0; a.C1 = kv_layer(m, m->ckv, l, m->T); a.kv_fmt = m->kv_fmt; a.hm_rows_per_b = m->T; a.hm_cap = m->T; a.hm_H = m->H;
      MT3_TRY(gemm(m, a, s));
    }
  }
  MT3_CUDA_CHECK(cudaMemsetAsync(m->state, 0, 4 * sizeof(int), s));
  MT3_CUDA_CHECK(cudaMemsetAsync(m->dcounters, 0, (size_t)m->dcounters_n * sizeof(int), s));
  MT3_CUDA_CHECK(cudaMemsetAsync(m->finished, 0, (size_t)m->B * sizeof(int), s));
  MT3_CUDA_CHECK(cudaMemsetAsync(m->tok_cur, 0, (size_t)m->B * sizeof(int), s));
  m->have_cross = true;
  m->host_pos = 0;
  return MT3_OK;
}

// A contiguous block of sequences decoded in one launch (batches above 64 rows run in 64-row blocks).
struct Rows { int begin, count; };

constexpr int kTraceSlots = 256, kTraceWords = 16;   // words 8..15: %smid of the 8 CTAs of tile 0's cluster
static unsigned long long* trace_slot(Model* m, const char* name) {
  if (!m->tracing || (int)m->trace_names.size() >= kTraceSlots) return nullptr;
  m->trace_names.push_back(name);
  return m->trace + (size_t)(m->trace_names.size() - 1) * kTraceWords;
}

// Decode-step GEMM on M = B rows: split-K exact-fp32 cluster kernel with the RMSNorm statistic fused (decode.cuh), in every
// gemm_mode (the tcgen05 variants of both rounds are correct but slower: csrc/experiments/).
static int dec_gemm(Model* m, const float* A, int lda, const float* W, int N, int K, int norm, int epi, float* C, int ldc,
                    int n_split, char* kv, const int* pos, const Rows& rows, cudaStream_t s) {
  for (int r0 = rows.begin; r0 < rows.begin + rows.count; r0 += kDecBM) {
    DecGemmArgs a;
    memset(&a, 0, sizeof(a));
    a.A = A + (int64_t)r0 * lda; a.lda = lda; a.W = W; a.ldw = N; a.M = std::min(kDecBM, rows.begin + rows.count - r0);
    a.N = N; a.K = K;
    a.norm = norm; a.eps = 1e-6f; a.epi = epi;
    a.R = C + (int64_t)r0 * ldc; a.ldr = ldc;                  // residual is always added in place
    a.C = C + (int64_t)r0 * ldc; a.ldc = ldc; a.n_split = n_split;
    if (kv) {  // rows_per_b = 1: skip r0 sequences, each 2*H*cap rows
      a.C1 = kv + (int64_t)r0 * 2 * m->H * m->L * m->kv_row; a.kv_fmt = m->kv_fmt;
      a.hm_rows_per_b = 1; a.hm_cap = m->L; a.hm_H = m->H; a.hm_pos = pos;
    }
    a.partial = m->dpartial;
    a.counters = m->dcounters;
    a.trace = trace_slot(m, K == m->F ? "gemm_mlp_out" : (N == 2 * m->F ? "gemm_mlp_in" : (kv ? "gemm_qkv_append" : (N == m->V ? "gemm_logits" : (K == m->Q ? "gemm_attn_out" : "gemm_cross_q")))));
    int rc = MT3_ERR_UNSUPPORTED;
    if (m->dec_cluster) rc = launch_dec_gemm_cluster(a, s, m->pdl_gemm, m->dec_pipe);
    if (rc == MT3_ERR_UNSUPPORTED) rc = launch_dec_gemm(a, s, m->pdl_gemm);   // shapes the cluster kernel does not tile
    MT3_TRY(rc);
  }
  return MT3_OK;
}

// prefetch: the launch is part of a decode step (the kernel starts under the preceding GEMM): L2 prefetch of m->pf_attn tiles
template <int FMT>
static int launch_dec_attention_t(Model* m, const float* q, const char* kv, int cap, const int* len_ptr, int len_add,
                                  float* out, const Rows& rows, cudaStream_t s, const float* q_ssq, size_t smem, int max_len,
                                  bool prefetch) {
  static bool attr_done = false;
  if (!attr_done) {
    MT3_CUDA_CHECK(cudaFuncSetAttribute(dec_attention_bulk_kernel<FMT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    MT3_CUDA_CHECK(cudaFuncSetAttribute(dec_attention_bulk_kernel<FMT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    attr_done = true;
  }
  MT3_CUDA_CHECK(launch_kernel(m->tracing ? dec_attention_bulk_kernel<FMT, true> : dec_attention_bulk_kernel<FMT, false>,
                               dim3(m->H, rows.count), dim3(kAttThreads), smem, s, m->pdl_attn,
                               q + (int64_t)rows.begin * m->Q, m->Q, 0,
                               (const void*)(kv + (int64_t)rows.begin * 2 * m->H * cap * m->kv_row), m->H, cap,
                               len_ptr, len_add, max_len, out + (int64_t)rows.begin * m->Q, m->Q,
                               q_ssq ? q_ssq + (int64_t)rows.begin * (m->D / 32) : (const float*)nullptr, m->D / 32, m->D / 32,
                               (float)m->D, 1e-6f, trace_slot(m, len_ptr ? "attn_self" : "attn_cross"), prefetch ? m->pf_attn : 0));
  MT3_LAUNCH_CHECK();
  return MT3_OK;
}

static int launch_dec_attention(Model* m, const float* q, const char* kv, int cap, const int* len_ptr, int len_add,
                                float* out, const Rows& rows, cudaStream_t s, const float* q_ssq = nullptr, bool prefetch = false) {
  const int max_len = std::max(m->L, m->T);
  const size_t smem = dec_attention_smem(max_len);
  MT3_REQUIRE(smem <= 100 * 1024, MT3_ERR_UNSUPPORTED, "decode attention: length %d too long", max_len);
  switch (m->kv_fmt) {
    case MT3_KV_F16: return launch_dec_attention_t<1>(m, q, kv, cap, len_ptr, len_add, out, rows, s, q_ssq, smem, max_len, prefetch);
    case MT3_KV_P24: return launch_dec_attention_t<2>(m, q, kv, cap, len_ptr, len_add, out, rows, s, q_ssq, smem, max_len, prefetch);
    default: return launch_dec_attention_t<0>(m, q, kv, cap, len_ptr, len_add, out, rows, s, q_ssq, smem, max_len, prefetch);
  }
}

// y_out = y_in + o.Wo  and  q_raw = [o | y_in].[Wo.Wq ; Wq]  in ONE launch; the RMSNorm factor of y_out is applied to
// q inside the cross-attention kernel from the per-tile sums of squares this launch leaves in m->dssq.
static int dec_gemm_out_q(Model* m, const DecLayer& w, const float* y_in, float* y_out, const Rows& rows, cudaStream_t s) {
  const int D = m->D, Q = m->Q;
  if (rows.count > kDecBM || Q != 384 || D != 512) return MT3_ERR_UNSUPPORTED;
  const int64_t r0 = rows.begin;
  DecGemmArgs a0, a1;
  memset(&a0, 0, sizeof(a0));
  a0.A = m->dao + r0 * Q; a0.lda = Q; a0.W = w.wo; a0.ldw = D; a0.M = rows.count; a0.N = D; a0.K = Q;
  a0.eps = 1e-6f; a0.epi = EPI_RESIDUAL; a0.R = y_in + r0 * D; a0.ldr = D; a0.C = y_out + r0 * D; a0.ldc = D; a0.n_split = D;
  a0.ssq_out = m->dssq + r0 * (D / 32); a0.ssq_ld = D / 32;
  a0.trace = trace_slot(m, "gemm_out+cross_q");
  memset(&a1, 0, sizeof(a1));
  a1.A = m->dao + r0 * Q; a1.lda = Q; a1.A2 = y_in + r0 * D; a1.lda2 = D; a1.K0 = Q;
  a1.W = w.wc1; a1.ldw = Q; a1.M = rows.count; a1.N = Q; a1.K = Q + D;
  a1.eps = 1e-6f; a1.epi = EPI_STORE; a1.C = m->dq + r0 * Q; a1.ldc = Q; a1.n_split = Q;
  a1.R = a1.C; a1.ldr = Q;
  a1.trace = a0.trace;
  return launch_dec_gemm_out_q(a0, a1, s, m->pdl_gemm, m->dec_pipe);
}

// The residual stream of one step (ping-pongs between m->dy and m->dy2 across fused launches).
struct DecBranch { Rows rows; cudaStream_t s; float* y; int fused; };

static int dec_embed(Model* m, DecBranch& b, const int* tok_in) {
  MT3_CUDA_CHECK(launch_kernel(embed_kernel, dim3(b.rows.count), dim3(128), 0, b.s, m->pdl, tok_in, (const float*)m->emb, m->D, m->V,
                               (const float*)m->pe, (const int*)m->state, m->dy, b.rows.begin));
  MT3_LAUNCH_CHECK();
  b.y = m->dy;
  return MT3_OK;
}
// fused RMSNorm + QKV projection + K/V cache append (layers.py:238-240, :272-289)
static int dec_layer_qkv(Model* m, DecBranch& b, int l) {
  return dec_gemm(m, b.y, m->D, m->dec[l].wqkv, 3 * m->Q, m->D, 1, EPI_STORE, m->dq, m->Q, m->Q, kv_layer(m, m->skv, l, m->L), m->state,
                  b.rows, b.s);
}
static int dec_layer_self(Model* m, DecBranch& b, int l) {
  return launch_dec_attention(m, m->dq, kv_layer(m, m->skv, l, m->L), m->L, m->state, 1, m->dao, b.rows, b.s, nullptr, true);
}
// self-attention out-projection + residual, cross-attention query projection (one launch when fused)
static int dec_layer_outq(Model* m, DecBranch& b, int l) {
  const DecLayer& w = m->dec[l];
  const int D = m->D, Q = m->Q;
  b.fused = MT3_ERR_UNSUPPORTED;
  if (m->fuse_q && m->dec_cluster) {
    float* y_next = (b.y == m->dy) ? m->dy2 : m->dy;    // the fused launch reads y while other CTAs write y': ping-pong
    b.fused = dec_gemm_out_q(m, w, b.y, y_next, b.rows, b.s);
    if (b.fused == MT3_OK) b.y = y_next;
    else if (b.fused != MT3_ERR_UNSUPPORTED) return b.fused;
  }
  if (b.fused != MT3_OK) {
    MT3_TRY(dec_gemm(m, m->dao, Q, w.wo, D, Q, 0, EPI_RESIDUAL, b.y, D, D, nullptr, nullptr, b.rows, b.s));
    MT3_TRY(dec_gemm(m, b.y, D, w.wq_c, Q, D, 1, EPI_STORE, m->dq, Q, Q, nullptr, nullptr, b.rows, b.s));
  }
  return MT3_OK;
}
static int dec_layer_cross(Model* m, DecBranch& b, int l) {
  return launch_dec_attention(m, m->dq, kv_layer(m, m->ckv, l, m->T), m->T, nullptr, m->T, m->dao, b.rows, b.s,
                              b.fused == MT3_OK ? m->dssq : nullptr, true);
}
static int dec_layer_mlp(Model* m, DecBranch& b, int l) {
  const DecLayer& w = m->dec[l];
  const int D = m->D, Q = m->Q, F = m->F;
  MT3_TRY(dec_gemm(m, m->dao, Q, w.wo_c, D, Q, 0, EPI_RESIDUAL, b.y, D, D, nullptr, nullptr, b.rows, b.s));
  MT3_TRY(dec_gemm(m, b.y, D, w.wi, 2 * F, D, 1, EPI_GATED_GELU, m->dg, F, 2 * F, nullptr, nullptr, b.rows, b.s));
  MT3_TRY(dec_gemm(m, m->dg, F, w.wo2, D, F, 0, EPI_RESIDUAL, b.y, D, D, nullptr, nullptr, b.rows, b.s));
  return MT3_OK;
}

// One decode step (network.py:303-361 -> :196-262 -> :88-155) for the whole batch.  tok_in DEV [B]; logits
// DEV [B,V]; greedy != 0 runs the argmax/bookkeeping kernel (tok_user optional), else only the position advances.
// 7 launches per layer: [norm+QKV+KV-append] [self-attn] [out+residual | norm+q] [cross-attn] [out+residual]
// [norm+gated-GELU MLP in] [MLP out+residual].
// loop_step: a step of mt3_generate's loop -- the decoder input m->dy was already written (by dec_embed before the first
// step, by the previous step's argmax kernel afterwards), and this step's argmax kernel writes the next one.
static int decode_step_impl(Model* m, const int* tok_in, float* logits, int greedy, int* tok_user, int use_finished,
                            int* tokens_ws, cudaStream_t s, bool loop_step = false) {
  DecBranch b{Rows{0, m->B}, s, nullptr, MT3_ERR_UNSUPPORTED};
  if (loop_step) b.y = m->dy;
  else MT3_TRY(dec_embed(m, b, tok_in));
  for (int l = 0; l < m->Ld; ++l) {
    MT3_TRY(dec_layer_qkv(m, b, l));
    MT3_TRY(dec_layer_self(m, b, l));
    MT3_TRY(dec_layer_outq(m, b, l));
    MT3_TRY(dec_layer_cross(m, b, l));
    MT3_TRY(dec_layer_mlp(m, b, l));
  }
  MT3_TRY(dec_gemm(m, b.y, m->D, m->w_logits, m->V, m->D, 1, EPI_STORE, logits, m->V, m->V, nullptr, nullptr, b.rows, s));
  if (greedy == 2) {        // T5X beam_search bookkeeping at num_decodes = 1 (generate loop only)
    MT3_CUDA_CHECK(launch_kernel(beam1_step_kernel, dim3(m->B), dim3(256), 0, s, m->pdl, (const float*)logits, m->V, m->B, m->tok_cur,
                                 m->finished, tokens_ws, m->L, m->state, m->beam_f, m->beam_i, 0.6f, m->L, (const float*)m->emb,
                                 (const float*)m->pe, m->D, loop_step ? m->dy : (float*)nullptr));
    MT3_LAUNCH_CHECK();
  } else if (greedy) {
    MT3_CUDA_CHECK(launch_kernel(argmax_step_kernel, dim3(m->B), dim3(256), 0, s, m->pdl, (const float*)logits, m->V, m->B,
                                 use_finished ? m->tok_cur : (int*)nullptr, use_finished ? m->finished : (int*)nullptr,
                                 tokens_ws, m->L, tok_user, m->state, 1, 0, (const float*)m->emb, (const float*)m->pe, m->D,
                                 loop_step ? m->dy : (float*)nullptr));
    MT3_LAUNCH_CHECK();
  } else {
    MT3_CUDA_CHECK(launch_kernel(advance_pos_kernel, dim3(1), dim3(1), 0, s, m->pdl, m->state));
    MT3_LAUNCH_CHECK();
  }
  return MT3_OK;
}

static void drop_graphs(Model* m) {
  for (auto& kv : m->graphs) {
    if (kv.second.e) cudaGraphExecDestroy(kv.second.e);
    if (kv.second.g) cudaGraphDestroy(kv.second.g);
  }
  m->graphs.clear();
  m->graph_exec = nullptr;
  m->graph = nullptr;
}

// make the graph of the current (workspace, B, T, decode mode) binding current, if one has been captured
static void select_graph(Model* m, int mode = 1) {
  m->graph_mode = mode;
  const auto it = m->graphs.find(std::make_tuple((const void*)m->ws, m->B, m->T, mode));
  if (it == m->graphs.end()) {
    m->graph = nullptr; m->graph_exec = nullptr; m->graph_kernels = 0;
  } else {
    m->graph = it->second.g; m->graph_exec = it->second.e; m->graph_kernels = it->second.kernels;
  }
}

// mode: 1 greedy, 2 beam-size-1 search; nsteps consecutive decode steps per graph (the position lives on the device, so a
// graph of 16 steps is the single-step graph 16 times over: one graph launch and its ~3 us of inter-launch latency per 16 steps)
static int ensure_graph(Model* m, int mode, int nsteps = 1) {
  const int key = mode | (nsteps << 8);
  if (m->graph_mode != key) select_graph(m, key);
  if (m->graph_exec) return MT3_OK;
  if (!m->cap_stream) MT3_CUDA_CHECK(cudaStreamCreateWithFlags(&m->cap_stream, cudaStreamNonBlocking));
  const uint64_t before = g_launch_count.load();
  MT3_CUDA_CHECK(cudaStreamBeginCapture(m->cap_stream, cudaStreamCaptureModeThreadLocal));
  int r = MT3_OK;
  for (int i = 0; i < nsteps && r == MT3_OK; ++i)
    r = decode_step_impl(m, m->tok_cur, m->dlogits, mode, nullptr, 1, m->tokens, m->cap_stream, true);
  cudaGraph_t g = nullptr;
  cudaError_t e = cudaStreamEndCapture(m->cap_stream, &g);
  if (r != MT3_OK) {
    if (g) cudaGraphDestroy(g);
    return r;
  }
  if (e != cudaSuccess) return fail(MT3_ERR_CUDA, "cudaStreamEndCapture -> %s", cudaGetErrorString(e));
  m->graph = g;
  m->graph_kernels = g_launch_count.load() - before;
  g_launch_count.fetch_sub(m->graph_kernels);   // capture does not execute
  MT3_CUDA_CHECK(cudaGraphInstantiate(&m->graph_exec, m->graph, 0));
  if (m->graphs.size() >= 12) {                 // bound the cache: forget everything but the new graph
    const Model::StepGraph keep{m->graph, m->graph_exec, m->graph_kernels};
    m->graph = nullptr; m->graph_exec = nullptr;
    drop_graphs(m);
    m->graph = keep.g; m->graph_exec = keep.e; m->graph_kernels = keep.kernels;
  }
  m->graphs[std::make_tuple((const void*)m->ws, m->B, m->T, key)] = Model::StepGraph{m->graph, m->graph_exec, m->graph_kernels};
  return MT3_OK;
}

}  // namespace mt3

using namespace mt3;

extern "C" int64_t mt3_model_num_params(const mt3_model_config* cfg) {
  if (!cfg) return -1;
  auto t = param_table(*cfg);
  return t.back().offset + t.back().rows * t.back().cols;
}

extern "C" int64_t mt3_model_param_offset(const mt3_model_config* cfg, const char* name, int64_t* numel) {
  if (!cfg || !name) return -1;
  for (const auto& e : param_table(*cfg))
    if (e.name == name) {
      if (numel) *numel = e.rows * e.cols;
      return e.offset;
    }
  return -1;
}

extern "C" int mt3_model_create(const mt3_model_config* cfg, const float* weights, mt3_model** out, void* stream) {
  MT3_REQUIRE(cfg && weights && out, MT3_ERR_BAD_ARG, "mt3_model_create: null argument");
  MT3_REQUIRE(cfg->head_dim == kHD, MT3_ERR_UNSUPPORTED, "mt3_model_create: head_dim %d (kernels are built for 64)", cfg->head_dim);
  MT3_REQUIRE(cfg->emb_dim % 64 == 0 && cfg->mlp_dim % 64 == 0 && cfg->input_depth % 16 == 0 && cfg->vocab_size % 4 == 0,
              MT3_ERR_UNSUPPORTED, "mt3_model_create: emb/mlp dims must be multiples of 64, input depth of 16, vocab of 4");
  MT3_REQUIRE(cfg->num_heads > 0 && cfg->num_encoder_layers >= 0 && cfg->num_decoder_layers > 0 && cfg->max_batch > 0 &&
                  cfg->max_input_length > 0 && cfg->max_decode_length > 0,
              MT3_ERR_BAD_ARG, "mt3_model_create: non-positive size");
  MT3_REQUIRE(cfg->max_decode_length <= 2048 && cfg->max_input_length <= 2048, MT3_ERR_UNSUPPORTED,
              "mt3_model_create: lengths above FixedEmbed.max_length=2048 (layers.py:565)");
  MT3_REQUIRE(cfg->gemm_mode == MT3_GEMM_FP32_SIMT || cfg->gemm_mode == MT3_GEMM_TF32X3 || cfg->gemm_mode == MT3_GEMM_TF32,
              MT3_ERR_BAD_ARG, "mt3_model_create: unknown gemm_mode %d", cfg->gemm_mode);
  MT3_REQUIRE(cfg->kv_cache_format == MT3_KV_F32 || cfg->kv_cache_format == MT3_KV_F16 || cfg->kv_cache_format == MT3_KV_P24, MT3_ERR_BAD_ARG,
              "mt3_model_create: unknown kv_cache_format %d", cfg->kv_cache_format);
  if (cfg->gemm_mode != MT3_GEMM_FP32_SIMT)
    MT3_REQUIRE(cfg->emb_dim % 32 == 0 && cfg->mlp_dim % 32 == 0 && cfg->input_depth % 32 == 0, MT3_ERR_UNSUPPORTED,
                "mt3_model_create: the tcgen05 path needs emb/mlp/input dims that are multiples of 32");
  cudaStream_t s = (cudaStream_t)stream;
  Model* m = new Model();
  m->cfg = *cfg;
  m->D = cfg->emb_dim; m->H = cfg->num_heads; m->Q = cfg->num_heads * cfg->head_dim; m->F = cfg->mlp_dim;
  m->V = cfg->vocab_size; m->Le = cfg->num_encoder_layers; m->Ld = cfg->num_decoder_layers; m->L = cfg->max_decode_length;
  const int D = m->D, Q = m->Q, F = m->F, V = m->V;
  cudaError_t e = cudaMalloc((void**)&m->slab, (size_t)prepared_floats(*cfg) * sizeof(float));
  if (e != cudaSuccess) {
    delete m;
    return fail(MT3_ERR_CUDA, "mt3_model_create: cudaMalloc -> %s", cudaGetErrorString(e));
  }
  float* p = m->slab;
  auto take = [&](int64_t n) { float* r = p; p += n; return r; };
  auto t = param_table(*cfg);
  auto W = [&](const std::string& n) -> const float* {
    for (const auto& en : t) if (en.name == n) return weights + en.offset;
    return nullptr;
  };
  int rc = MT3_OK;
#define PREP(...) do { if (rc == MT3_OK) rc = prep_copy(s, __VA_ARGS__); } while (0)
  m->w_in = take((int64_t)cfg->input_depth * D);
  PREP(W("encoder/continuous_inputs_projection/kernel"), cfg->input_depth, D, nullptr, m->w_in, D, 0, 1);
  m->enc.resize(m->Le);
  for (int i = 0; i < m->Le; ++i) {
    const std::string pre = "encoder/layers_" + std::to_string(i) + "/";
    EncLayer& L = m->enc[i];
    const float* g1 = W(pre + "pre_attention_layer_norm/scale");
    const float* g2 = W(pre + "pre_mlp_layer_norm/scale");
    L.wqkv = take((int64_t)D * 3 * Q);
    PREP(W(pre + "attention/query/kernel"), D, Q, g1, L.wqkv, 3 * Q, 0, 1);
    PREP(W(pre + "attention/key/kernel"), D, Q, g1, L.wqkv, 3 * Q, Q, 1);
    PREP(W(pre + "attention/value/kernel"), D, Q, g1, L.wqkv, 3 * Q, 2 * Q, 1);
    L.wo = take((int64_t)Q * D);
    PREP(W(pre + "attention/out/kernel"), Q, D, nullptr, L.wo, D, 0, 1);
    L.wi = take((int64_t)D * 2 * F);
    PREP(W(pre + "mlp/wi_0/kernel"), D, F, g2, L.wi, 2 * F, 0, 2);
    PREP(W(pre + "mlp/wi_1/kernel"), D, F, g2, L.wi, 2 * F, 1, 2);
    L.wo2 = take((int64_t)F * D);
    PREP(W(pre + "mlp/wo/kernel"), F, D, nullptr, L.wo2, D, 0, 1);
  }
  m->enc_norm_g = take(D);
  PREP(W("encoder/encoder_norm/scale"), 1, D, nullptr, m->enc_norm_g, D, 0, 1);
  m->emb = take((int64_t)V * D);
  PREP(W("decoder/token_embedder/embedding"), V, D, nullptr, m->emb, D, 0, 1);
  m->dec.resize(m->Ld);
  for (int i = 0; i < m->Ld; ++i) {
    const std::string pre = "decoder/layers_" + std::to_string(i) + "/";
    DecLayer& L = m->dec[i];
    const float* g1 = W(pre + "pre_self_attention_layer_norm/scale");
    const float* g2 = W(pre + "pre_cross_attention_layer_norm/scale");
    const float* g3 = W(pre + "pre_mlp_layer_norm/scale");
    L.wqkv = take((int64_t)D * 3 * Q);
    PREP(W(pre + "self_attention/query/kernel"), D, Q, g1, L.wqkv, 3 * Q, 0, 1);
    PREP(W(pre + "self_attention/key/kernel"), D, Q, g1, L.wqkv, 3 * Q, Q, 1);
    PREP(W(pre + "self_attention/value/kernel"), D, Q, g1, L.wqkv, 3 * Q, 2 * Q, 1);
    L.wo = take((int64_t)Q * D);
    PREP(W(pre + "self_attention/out/kernel"), Q, D, nullptr, L.wo, D, 0, 1);
    L.wq_c = take((int64_t)D * Q);
    PREP(W(pre + "encoder_decoder_attention/query/kernel"), D, Q, g2, L.wq_c, Q, 0, 1);
    L.wc1 = take((int64_t)(Q + D) * Q);
    if (rc == MT3_OK) {
      compose_out_q_kernel<<<dim3(cdiv(Q, 128), Q + D), 128, 0, s>>>(L.wo, L.wq_c, Q, D, L.wc1);
      if (cudaGetLastError() != cudaSuccess) rc = fail(MT3_ERR_CUDA, "mt3_model_create: compose_out_q launch failed");
    }
    L.wkv_c = take((int64_t)D * 2 * Q);   // applied to `encoded`, which is already normed: no fold
    PREP(W(pre + "encoder_decoder_attention/key/kernel"), D, Q, nullptr, L.wkv_c, 2 * Q, 0, 1);
    PREP(W(pre + "encoder_decoder_attention/value/kernel"), D, Q, nullptr, L.wkv_c, 2 * Q, Q, 1);
    L.wo_c = take((int64_t)Q * D);
    PREP(W(pre + "encoder_decoder_attention/out/kernel"), Q, D, nullptr, L.wo_c, D, 0, 1);
    L.wi = take((int64_t)D * 2 * F);
    PREP(W(pre + "mlp/wi_0/kernel"), D, F, g3, L.wi, 2 * F, 0, 2);
    PREP(W(pre + "mlp/wi_1/kernel"), D, F, g3, L.wi, 2 * F, 1, 2);
    L.wo2 = take((int64_t)F * D);
    PREP(W(pre + "mlp/wo/kernel"), F, D, nullptr, L.wo2, D, 0, 1);
  }
  m->w_logits = take((int64_t)D * V);
  PREP(W("decoder/logits_dense/kernel"), D, V, W("decoder/decoder_norm/scale"), m->w_logits, V, 0, 1);
#undef PREP
  m->pe = take((int64_t)2048 * D);
  if (rc == MT3_OK) {
    // layers.py:51-82 (float64 on the host, rounded to float32 like the reference's numpy code)
    std::vector<float> pe((size_t)2048 * D, 0.f);
    const int half = D / 2;
    const double scale_factor = -log(10000.0 / 1.0) / (double)(half - 1);
    for (int pos = 0; pos < 2048; ++pos)
      for (int i = 0; i < half; ++i) {
        const double div = 1.0 * exp((double)i * scale_factor);
        pe[(size_t)pos * D + i] = (float)sin((double)pos * div);
        pe[(size_t)pos * D + half + i] = (float)cos((double)pos * div);
      }
    e = cudaMemcpyAsync(m->pe, pe.data(), pe.size() * sizeof(float), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) rc = fail(MT3_ERR_CUDA, "mt3_model_create: PE upload -> %s", cudaGetErrorString(e));
  }
  {
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0)
      m->sm_count = sms;
  }
  {
    const char* e_pdl = getenv("MT3_PDL");
    // default: attention launches only (their K/V prefetch and launch latency hide under the preceding GEMM: 437.8 ->
    // 415.4 ms per batch); PDL on the GEMM launches measured slower (451.8), profiles/r02_call1_bench_pdl*.json
    const int pdl_bits = e_pdl ? atoi(e_pdl) : 2;
    m->pdl = (pdl_bits & 1) != 0;
    m->pdl_attn = (pdl_bits & 3) != 0;
    m->pdl_gemm = (pdl_bits & 5) != 0;
    const char* e_fuse = getenv("MT3_DEC_FUSE");
    m->fuse_q = !(e_fuse && e_fuse[0] == '0');
    const char* e_clu = getenv("MT3_DEC_CLUSTER");
    m->dec_cluster = !(e_clu && e_clu[0] == '0');
    const char* e_attn = getenv("MT3_TC_ATTENTION");
    m->tc_attn_ok = !(e_attn && e_attn[0] == '0');
    const char* e_pfa = getenv("MT3_PF_ATTN");
    if (e_pfa) m->pf_attn = std::max(0, atoi(e_pfa));
    const char* e_pipe = getenv("MT3_DEC_PIPE");
    if (e_pipe) m->dec_pipe = atoi(e_pipe) & 3;
  }
  m->kv_fmt = cfg->kv_cache_format;
  m->kv_row = kv_row_bytes(m->kv_fmt);
  m->tc = cfg->gemm_mode != MT3_GEMM_FP32_SIMT;
  m->split3 = cfg->gemm_mode == MT3_GEMM_TF32X3;
  if (rc == MT3_OK && m->tc) {
    e = cudaMalloc((void**)&m->slab_tc, (size_t)tc_weight_floats(*cfg) * sizeof(float));
    if (e != cudaSuccess) rc = fail(MT3_ERR_CUDA, "mt3_model_create: cudaMalloc(tc weights) -> %s", cudaGetErrorString(e));
    float* cur = m->slab_tc;
#define TCPREP(src, K, N, dst) do { if (rc == MT3_OK) rc = prep_tc_weight(m, s, src, K, N, cur, dst); } while (0)
    TCPREP(m->w_in, cfg->input_depth, D, &m->t_w_in);
    for (int i = 0; i < m->Le; ++i) {
      EncLayer& L = m->enc[i];
      TCPREP(L.wqkv, D, 3 * Q, &L.t_wqkv);
      TCPREP(L.wo, Q, D, &L.t_wo);
      TCPREP(L.wi, D, 2 * F, &L.t_wi);
      TCPREP(L.wo2, F, D, &L.t_wo2);
    }
    for (int i = 0; i < m->Ld; ++i) TCPREP(m->dec[i].wkv_c, D, 2 * Q, &m->dec[i].t_wkv_c);
#undef TCPREP
    if (rc == MT3_OK) {
      e = cudaStreamSynchronize(s);
      if (e != cudaSuccess) rc = fail(MT3_ERR_CUDA, "mt3_model_create: tc weight prep -> %s", cudaGetErrorString(e));
    }
  }
  if (rc == MT3_OK) {
    e = cudaMallocHost((void**)&m->h_flag, 4 * sizeof(int));
    if (e != cudaSuccess) rc = fail(MT3_ERR_CUDA, "mt3_model_create: cudaMallocHost -> %s", cudaGetErrorString(e));
  }
  if (rc != MT3_OK) {
    cudaFree(m->slab);
    cudaFree(m->slab_tc);
    delete m;
    return rc;
  }
  *out = reinterpret_cast<mt3_model*>(m);
  return MT3_OK;
}

extern "C" int mt3_model_destroy(mt3_model* h) {
  if (!h) return MT3_OK;
  Model* m = reinterpret_cast<Model*>(h);
  drop_graphs(m);
  if (m->cap_stream) cudaStreamDestroy(m->cap_stream);
  if (m->h_flag) cudaFreeHost(m->h_flag);
  cudaFree(m->slab);
  cudaFree(m->slab_tc);
  delete m;
  return MT3_OK;
}

namespace {
struct WsLayout {
  int64_t x_hi, x_lo, h_lo, ao_lo, g_lo, enc_hi, enc_lo, qkv_lo, vt_hi, vt_lo;
  int64_t dy2, dssq;
  int64_t h, rstd, qkv, ao, g, encoded, ckv, skv, dy, drstd, dq, dao, dg, dlogits, tok_cur, finished, tokens, state, dpartial, dcounters, beam_f, beam_i, att_scratch, total;
};
WsLayout ws_layout(const Model* m, int B, int T) {
  WsLayout w;
  int64_t off = 0;
  auto take = [&](int64_t bytes) { int64_t r = off; off += align_up(bytes, 256); return r; };
  const int64_t M = (int64_t)B * T, D = m->D, Q = m->Q, F = m->F, V = m->V, L = m->L;
  const bool s3 = m->split3;
  w.x_hi = take(s3 ? M * m->cfg.input_depth * 4 : 0);
  w.x_lo = take(s3 ? M * m->cfg.input_depth * 4 : 0);
  w.h_lo = take(s3 ? M * D * 4 : 0);
  w.ao_lo = take(s3 ? M * Q * 4 : 0);
  w.g_lo = take(s3 ? M * F * 4 : 0);
  w.enc_hi = take(s3 ? M * D * 4 : 0);
  w.enc_lo = take(s3 ? M * D * 4 : 0);
  w.qkv_lo = take(s3 ? M * 3 * Q * 4 : 0);
  w.vt_hi = take(m->tc ? M * Q * 4 : 0);
  w.vt_lo = take(s3 ? M * Q * 4 : 0);
  w.h = take(M * D * 4);
  w.rstd = take(M * 4);
  w.qkv = take(M * 3 * Q * 4);
  w.ao = take(M * Q * 4);
  w.g = take(M * F * 4);
  w.encoded = take(M * D * 4);
  w.ckv = take((int64_t)m->Ld * M * 2 * m->H * m->kv_row);
  w.skv = take((int64_t)m->Ld * B * L * 2 * m->H * m->kv_row);
  w.dy = take((int64_t)B * D * 4);
  w.drstd = take((int64_t)B * 4);
  w.dy2 = take((int64_t)B * D * 4);
  w.dssq = take((int64_t)B * (D / 32) * 4);
  w.dq = take((int64_t)B * Q * 4);
  w.dao = take((int64_t)B * Q * 4);
  w.dg = take((int64_t)B * F * 4);
  w.dlogits = take((int64_t)B * V * 4);
  w.tok_cur = take((int64_t)B * 4);
  w.finished = take((int64_t)B * 4);
  w.tokens = take((int64_t)B * L * 4);
  w.state = take(64);
  w.dpartial = take((int64_t)16 * cdiv(std::max(std::max(3 * (int)Q, 2 * (int)F), (int)V), kDecBN) * kDecTileFloats * 4);   // up to 16 K chunks
  w.dcounters = take((int64_t)cdiv(std::max(std::max(3 * (int)Q, 2 * (int)F), (int)V), kDecBN) * 4);
  w.att_scratch = take(m->tc ? enc_attention_tc_scratch_floats(B, T, m->H) * 4 : 0);
  w.beam_f = take((int64_t)B * 2 * 4);
  w.beam_i = take((int64_t)B * 4);
  w.total = off;
  return w;
}
}  // namespace

extern "C" int64_t mt3_workspace_bytes(const mt3_model* h, int32_t batch, int32_t input_length) {
  if (!h || batch <= 0 || input_length <= 0) return -1;
  return ws_layout(reinterpret_cast<const Model*>(h), batch, input_length).total;
}

extern "C" int mt3_model_set_workspace(mt3_model* h, void* workspace, int64_t bytes, int32_t batch, int32_t input_length) {
  MT3_REQUIRE(h && workspace, MT3_ERR_BAD_ARG, "mt3_model_set_workspace: null argument");
  Model* m = reinterpret_cast<Model*>(h);
  MT3_REQUIRE(batch > 0 && batch <= m->cfg.max_batch, MT3_ERR_SHAPE, "batch %d outside (0, max_batch=%d]", batch, m->cfg.max_batch);
  MT3_REQUIRE(input_length > 0 && input_length <= m->cfg.max_input_length, MT3_ERR_SHAPE,
              "input_length %d outside (0, max_input_length=%d]", input_length, m->cfg.max_input_length);
  MT3_REQUIRE(((uintptr_t)workspace & 255) == 0, MT3_ERR_WORKSPACE, "workspace must be 256-byte aligned");
  const WsLayout w = ws_layout(m, batch, input_length);
  MT3_REQUIRE(bytes >= w.total, MT3_ERR_WORKSPACE, "workspace has %lld bytes, %lld needed", (long long)bytes, (long long)w.total);
  char* b = (char*)workspace;
  m->ws = b; m->ws_bytes = bytes; m->B = batch; m->T = input_length;
  select_graph(m);
  m->h = (float*)(b + w.h); m->rstd = (float*)(b + w.rstd); m->qkv = (float*)(b + w.qkv); m->ao = (float*)(b + w.ao);
  m->g = (float*)(b + w.g); m->encoded = (float*)(b + w.encoded); m->ckv = b + w.ckv; m->skv = b + w.skv;
  m->dy2 = (float*)(b + w.dy2); m->dssq = (float*)(b + w.dssq);
  m->dy = (float*)(b + w.dy); m->drstd = (float*)(b + w.drstd); m->dq = (float*)(b + w.dq); m->dao = (float*)(b + w.dao);
  m->dg = (float*)(b + w.dg); m->dlogits = (float*)(b + w.dlogits); m->tok_cur = (int*)(b + w.tok_cur);
  m->finished = (int*)(b + w.finished); m->tokens = (int*)(b + w.tokens); m->state = (int*)(b + w.state);
  m->dpartial = (float*)(b + w.dpartial); m->dcounters = (int*)(b + w.dcounters);
  m->beam_f = (float*)(b + w.beam_f); m->beam_i = (int*)(b + w.beam_i);
  m->att_scratch = (m->tc && enc_attention_tc_scratch_floats(batch, input_length, m->H) > 0) ? (float*)(b + w.att_scratch) : nullptr;
  m->dcounters_n = cdiv(std::max(std::max(3 * m->Q, 2 * m->F), m->V), kDecBN);
  m->have_cross = false;
  if (m->tc) {
    const int64_t M = (int64_t)batch * input_length;
    const bool s3 = m->split3;
    m->a_x.hi = s3 ? (float*)(b + w.x_hi) : nullptr; m->a_x.lo = s3 ? (float*)(b + w.x_lo) : nullptr;
    m->a_h.hi = m->h; m->a_h.lo = s3 ? (float*)(b + w.h_lo) : nullptr;
    m->a_ao.hi = m->ao; m->a_ao.lo = s3 ? (float*)(b + w.ao_lo) : nullptr;
    m->a_g.hi = m->g; m->a_g.lo = s3 ? (float*)(b + w.g_lo) : nullptr;
    m->a_enc.hi = s3 ? (float*)(b + w.enc_hi) : nullptr; m->a_enc.lo = s3 ? (float*)(b + w.enc_lo) : nullptr;
    if (s3) {
      MT3_TRY(make_operand(&m->a_x.op, m->a_x.hi, m->a_x.lo, M, m->cfg.input_depth, m->cfg.input_depth));
      MT3_TRY(make_operand(&m->a_enc.op, m->a_enc.hi, m->a_enc.lo, M, m->D, m->D));
    }
    MT3_TRY(make_operand(&m->a_h.op, m->a_h.hi, m->a_h.lo, M, m->D, m->D));
    MT3_TRY(make_operand(&m->a_ao.op, m->a_ao.hi, m->a_ao.lo, M, m->Q, m->Q));
    MT3_TRY(make_operand(&m->a_g.op, m->a_g.hi, m->a_g.lo, M, m->F, m->F));
    m->a_qkv.hi = m->qkv; m->a_qkv.lo = s3 ? (float*)(b + w.qkv_lo) : nullptr;
    MT3_TRY(make_operand(&m->a_qkv.op, m->a_qkv.hi, m->a_qkv.lo, M, 3 * m->Q, 3 * m->Q));
    m->a_vt.hi = (float*)(b + w.vt_hi); m->a_vt.lo = s3 ? (float*)(b + w.vt_lo) : nullptr;
    if (input_length % 4 == 0)   // TMA row pitch must be a multiple of 16 bytes; otherwise the SIMT attention kernel runs
      MT3_TRY(make_operand(&m->a_vt.op, m->a_vt.hi, m->a_vt.lo, (uint64_t)batch * m->H * 64, input_length, input_length, 64));
  }
  return MT3_OK;
}

#define MT3_NEED_WS(m) MT3_REQUIRE((m)->ws, MT3_ERR_STATE, "no workspace set (call mt3_model_set_workspace first)")

extern "C" int mt3_encode(mt3_model* h, const float* x, float* encoded, void* stream) {
  MT3_REQUIRE(h && x && encoded, MT3_ERR_BAD_ARG, "mt3_encode: null argument");
  Model* m = reinterpret_cast<Model*>(h);
  MT3_NEED_WS(m);
  return encode_impl(m, x, encoded, (cudaStream_t)stream);
}

extern "C" int mt3_cross_kv(mt3_model* h, const float* encoded, void* stream) {
  MT3_REQUIRE(h && encoded, MT3_ERR_BAD_ARG, "mt3_cross_kv: null argument");
  Model* m = reinterpret_cast<Model*>(h);
  MT3_NEED_WS(m);
  return cross_kv_impl(m, encoded, (cudaStream_t)stream);
}

extern "C" int mt3_decode_step(mt3_model* h, const int32_t* tok_in, float* logits, int32_t* tok_out, void* stream) {
  MT3_REQUIRE(h && tok_in, MT3_ERR_BAD_ARG, "mt3_decode_step: null argument");
  Model* m = reinterpret_cast<Model*>(h);
  MT3_NEED_WS(m);
  MT3_REQUIRE(m->have_cross, MT3_ERR_STATE, "mt3_decode_step before mt3_cross_kv");
  MT3_REQUIRE(m->host_pos < m->L, MT3_ERR_STATE, "mt3_decode_step: cache full (%d steps = max_decode_length)", m->L);
  m->host_pos += 1;
  return decode_step_impl(m, tok_in, logits ? logits : m->dlogits, tok_out != nullptr, tok_out, 0, nullptr,
                          (cudaStream_t)stream);
}

extern "C" int mt3_generate(mt3_model* h, const float* x, int32_t num_steps, int32_t flags, int32_t* tokens_out,
                            int32_t* steps_run, void* stream) {
  MT3_REQUIRE(h && x && tokens_out, MT3_ERR_BAD_ARG, "mt3_generate: null argument");
  Model* m = reinterpret_cast<Model*>(h);
  MT3_NEED_WS(m);
  MT3_REQUIRE(num_steps >= 0 && num_steps <= m->L, MT3_ERR_SHAPE, "num_steps %d outside [0, max_decode_length=%d]", num_steps, m->L);
  MT3_REQUIRE((flags & ~(MT3_GEN_STOP_AT_EOS | MT3_GEN_USE_GRAPH | MT3_GEN_BEAM1)) == 0, MT3_ERR_BAD_ARG, "mt3_generate: unknown flag bits 0x%x", flags);
  cudaStream_t s = (cudaStream_t)stream;
  MT3_TRY(encode_impl(m, x, m->encoded, s));
  MT3_TRY(cross_kv_impl(m, m->encoded, s));
  MT3_CUDA_CHECK(cudaMemsetAsync(m->tokens, 0, (size_t)m->B * m->L * sizeof(int), s));
  const bool use_graph = (flags & MT3_GEN_USE_GRAPH) != 0;
  const bool stop = (flags & MT3_GEN_STOP_AT_EOS) != 0;
  const int mode = (flags & MT3_GEN_BEAM1) ? 2 : 1;
  if (mode == 2) {      // live log-probability 0, finished score NEG_INF (t5x decoding.NEG_INF = -1e7), no finished hypothesis
    std::vector<float> init((size_t)2 * m->B);
    for (int i = 0; i < m->B; ++i) { init[2 * i] = 0.f; init[2 * i + 1] = -1.0e7f; }
    MT3_CUDA_CHECK(cudaMemcpyAsync(m->beam_f, init.data(), init.size() * sizeof(float), cudaMemcpyHostToDevice, s));
    MT3_CUDA_CHECK(cudaStreamSynchronize(s));        // `init` is stack-owned pageable memory
    MT3_CUDA_CHECK(cudaMemsetAsync(m->beam_i, 0, (size_t)m->B * sizeof(int), s));
  }
  constexpr int kBlock = 16;                    // steps per graph launch (and between two polls of the all-finished flag)
  cudaGraphExec_t g1 = nullptr, gN = nullptr;
  uint64_t k1 = 0, kN = 0;
  if (use_graph) {
    if (num_steps >= kBlock) {
      MT3_TRY(ensure_graph(m, mode, kBlock));
      gN = m->graph_exec; kN = m->graph_kernels;
    }
    if (num_steps % kBlock != 0) {
      MT3_TRY(ensure_graph(m, mode, 1));
      g1 = m->graph_exec; k1 = m->graph_kernels;
    }
  }
  if (num_steps > 0) {     // decoder input of step 0: BOS (tok_cur was zeroed by cross_kv) at position 0; later ones come from the argmax kernel
    DecBranch b0{Rows{0, m->B}, s, nullptr, MT3_ERR_UNSUPPORTED};
    MT3_TRY(dec_embed(m, b0, m->tok_cur));
  }
  int ran = 0;
  for (int step = 0; step < num_steps;) {
    int n = 1;
    if (use_graph && gN && num_steps - step >= kBlock) {
      MT3_CUDA_CHECK(cudaGraphLaunch(gN, s));
      count_launch(kN);
      n = kBlock;
    } else if (use_graph) {
      MT3_CUDA_CHECK(cudaGraphLaunch(g1, s));
      count_launch(k1);
    } else {
      MT3_TRY(decode_step_impl(m, m->tok_cur, m->dlogits, mode, nullptr, 1, m->tokens, s, true));
    }
    step += n;
    ran += n;
    m->host_pos += n;
    if (stop && ((step & 15) == 0 || step == num_steps)) {
      MT3_CUDA_CHECK(cudaMemcpyAsync(m->h_flag, m->state + 2, sizeof(int), cudaMemcpyDeviceToHost, s));
      MT3_CUDA_CHECK(cudaStreamSynchronize(s));
      if (m->h_flag[0]) break;
    }
  }
  if (mode == 2) {
    beam1_finalize_kernel<<<m->B, 128, 0, s>>>(m->tokens, m->B, m->L, ran, m->beam_i);
    MT3_LAUNCH_CHECK();
  }
  MT3_CUDA_CHECK(cudaMemcpyAsync(tokens_out, m->tokens, (size_t)m->B * m->L * sizeof(int), cudaMemcpyDeviceToDevice, s));
  if (steps_run) *steps_run = ran;
  return MT3_OK;
}

extern "C" int mt3_vocab_decode(const int32_t* ids, int32_t batch, int32_t length, int32_t num_regular_tokens, int32_t* out,
                                void* stream) {
  MT3_REQUIRE(ids && out, MT3_ERR_BAD_ARG, "mt3_vocab_decode: null argument");
  MT3_REQUIRE(batch >= 0 && length >= 0 && num_regular_tokens >= 0, MT3_ERR_BAD_ARG, "mt3_vocab_decode: negative size");
  if (batch == 0 || length == 0) return MT3_OK;
  vocab_decode_kernel<<<cdiv(batch, 64), 64, 0, (cudaStream_t)stream>>>(ids, batch, length, num_regular_tokens, out);
  MT3_LAUNCH_CHECK();
  return MT3_OK;
}

extern "C" int mt3_dot_product_attention_f32(const float* q, const float* k, const float* v, const float* bias, int32_t batch,
                                             int32_t q_len, int32_t kv_len, int32_t num_heads, int32_t head_dim, float* out,
                                             void* stream) {
  MT3_REQUIRE(q && k && v && out, MT3_ERR_BAD_ARG, "mt3_dot_product_attention_f32: null argument");
  MT3_REQUIRE(batch >= 0 && q_len >= 0 && kv_len > 0 && num_heads > 0 && head_dim > 0, MT3_ERR_BAD_ARG,
              "mt3_dot_product_attention_f32: non-positive size");
  MT3_REQUIRE(kv_len <= 8192, MT3_ERR_UNSUPPORTED, "mt3_dot_product_attention_f32: kv_len %d above 8192", kv_len);
  const long long items = (long long)batch * num_heads * q_len;
  if (items == 0) return MT3_OK;
  const size_t smem = (size_t)4 * kv_len * sizeof(float);
  static size_t attr_smem = 48 * 1024;
  if (smem > attr_smem) {
    MT3_CUDA_CHECK(cudaFuncSetAttribute(dot_product_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_smem = smem;
  }
  dot_product_attention_kernel<<<(unsigned)((items + 3) / 4), 128, smem, (cudaStream_t)stream>>>(q, k, v, bias, batch, q_len, kv_len,
                                                                                                 num_heads, head_dim, out);
  MT3_LAUNCH_CHECK();
  return MT3_OK;
}

__global__ void trace_reset_kernel(unsigned long long* t, int n_slots) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_slots * mt3::kTraceWords) t[i] = (i % mt3::kTraceWords == 0) ? ~0ull : 0ull;
}

extern "C" int mt3_debug_trace_step(mt3_model* h, int32_t pos, uint64_t* out, int32_t max_slots, char* names,
                                    int32_t names_bytes, int32_t* n_slots, void* stream) {
  MT3_REQUIRE(h && out && names && n_slots, MT3_ERR_BAD_ARG, "mt3_debug_trace_step: null argument");
  Model* m = reinterpret_cast<Model*>(h);
  MT3_NEED_WS(m);
  MT3_REQUIRE(pos >= 2 && pos < m->L, MT3_ERR_BAD_ARG, "mt3_debug_trace_step: pos must be in [2, %d)", m->L);
  cudaStream_t s = (cudaStream_t)stream;
  if (!m->trace) MT3_CUDA_CHECK(cudaMalloc(&m->trace, sizeof(unsigned long long) * kTraceSlots * kTraceWords));
  if (!m->cap_stream) MT3_CUDA_CHECK(cudaStreamCreateWithFlags(&m->cap_stream, cudaStreamNonBlocking));
  // capture one greedy step with a trace slot baked into every GEMM / attention node
  m->trace_names.clear();
  m->tracing = true;
  const uint64_t before = g_launch_count.load();
  MT3_CUDA_CHECK(cudaStreamBeginCapture(m->cap_stream, cudaStreamCaptureModeThreadLocal));
  const int r = decode_step_impl(m, m->tok_cur, m->dlogits, 1, nullptr, 1, m->tokens, m->cap_stream, true);
  cudaGraph_t g = nullptr;
  const cudaError_t e = cudaStreamEndCapture(m->cap_stream, &g);
  m->tracing = false;
  g_launch_count.store(before);
  if (r != MT3_OK || e != cudaSuccess) {
    if (g) cudaGraphDestroy(g);
    return r != MT3_OK ? r : fail(MT3_ERR_CUDA, "mt3_debug_trace_step: capture -> %s", cudaGetErrorString(e));
  }
  cudaGraphExec_t ge = nullptr;
  MT3_CUDA_CHECK(cudaGraphInstantiate(&ge, g, 0));
  const int n = (int)m->trace_names.size();
  const int start_pos = pos - 2;                      // two warm replays, the third one (at `pos`) is read back
  MT3_CUDA_CHECK(cudaMemcpyAsync(m->state, &start_pos, sizeof(int), cudaMemcpyHostToDevice, s));
  MT3_CUDA_CHECK(cudaMemsetAsync(m->finished, 0, sizeof(int) * m->B, s));
  for (int it = 0; it < 3; ++it) {
    trace_reset_kernel<<<cdiv(kTraceSlots * kTraceWords, 256), 256, 0, s>>>(m->trace, kTraceSlots);
    MT3_CUDA_CHECK(cudaGraphLaunch(ge, s));
  }
  MT3_CUDA_CHECK(cudaStreamSynchronize(s));
  const int n_out = std::min(n, (int)max_slots);
  MT3_CUDA_CHECK(cudaMemcpy(out, m->trace, sizeof(unsigned long long) * n_out * kTraceWords, cudaMemcpyDeviceToHost));
  std::string all;
  for (int i = 0; i < n_out; ++i) { all += m->trace_names[i]; all += '\n'; }
  snprintf(names, names_bytes, "%s", all.c_str());
  *n_slots = n_out;
  cudaGraphExecDestroy(ge);
  cudaGraphDestroy(g);
  return MT3_OK;
}

extern "C" int mt3_debug_launch(mt3_model* h, int32_t kind, int32_t pos, int32_t iters, void* stream) {
  MT3_REQUIRE(h, MT3_ERR_BAD_ARG, "mt3_debug_launch: null model");
  Model* m = reinterpret_cast<Model*>(h);
  MT3_NEED_WS(m);
  MT3_REQUIRE(pos >= 0 && pos < m->L && iters > 0, MT3_ERR_BAD_ARG, "mt3_debug_launch: bad pos/iters");
  cudaStream_t s = (cudaStream_t)stream;
  const int B = m->B, D = m->D, Q = m->Q, L = m->L, T = m->T, M = B * T;
  for (int it = 0; it < iters; ++it) {
    const int l = it % m->Ld;
    switch (kind) {
      case MT3_K_DEC_SELF_ATTN: {
        MT3_TRY(launch_dec_attention(m, m->dq, kv_layer(m, m->skv, l, L), L, nullptr, pos + 1, m->dao, Rows{0, B}, s));
        break;
      }
      case MT3_K_DEC_CROSS_ATTN: {
        MT3_TRY(launch_dec_attention(m, m->dq, kv_layer(m, m->ckv, l, T), T, nullptr, T, m->dao, Rows{0, B}, s));
        break;
      }
      case MT3_K_DEC_QKV_GEMM: {
        // scratch output: the encoder qkv buffer (B*T rows >= B)
        MT3_TRY(dec_gemm(m, m->dy, D, m->dec[l].wqkv, 3 * Q, D, 1, EPI_STORE, m->qkv, 3 * Q, 3 * Q, nullptr, nullptr, Rows{0, B}, s));
        break;
      }
      case MT3_K_ENC_QKV_GEMM: {
        if (m->tc) {
          TcGemmArgs t = tc_args(M, 3 * Q, D, m->qkv, nullptr, 3 * Q);
          t.row_scale = m->rstd;
          MT3_TRY(launch_tc_gemm(m->a_h.op, m->enc[it % std::max(1, m->Le)].t_wqkv.op, t, m->split3, s));
          break;
        }
        GemmArgs a = gemm_args(m->h, D, m->enc[it % std::max(1, m->Le)].wqkv, 3 * Q, M, 3 * Q, D, m->qkv, 3 * Q);
        a.row_scale = m->rstd;
        MT3_TRY(gemm(m, a, s));
        break;
      }
      case MT3_K_ENC_ATTN: {
        if (m->tc && m->tc_attn_ok && enc_attention_tc_supported(T)) {
          MT3_TRY(launch_enc_attention_tc(m->a_qkv.op, m->a_vt.op, B, T, m->H, m->a_ao.hi, m->a_ao.lo, m->split3, s, nullptr, 0, nullptr,
                                          m->att_scratch));
          break;
        }
        MT3_TRY(set_attr_once());
        const size_t attn_smem = (size_t)(32 * kHD + 32 * (T + 4) + 64 * 68) * sizeof(float);
        enc_attention_kernel<<<dim3(cdiv(T, 32), m->H, B), 256, attn_smem, s>>>(m->qkv, 3 * Q, T, m->H, m->ao, nullptr, Q);
        MT3_LAUNCH_CHECK();
        break;
      }
      default:
        return fail(MT3_ERR_BAD_ARG, "mt3_debug_launch: unknown kind %d", kind);
    }
  }
  return MT3_OK;
}
