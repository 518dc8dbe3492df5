// Tokenise + embed + interleave in one pass, and the matching embedding backward.
//
// Replaces the per-sample python loop of GatoPolicy.tokenize_input_dicts (gato_policy.py:195-432):
// mu-law / uniform discretisation (input_tokenizers.py:5-30), the embed_token gathers, the
// inner-timestep position add (:381-385), the separator broadcast (:343), the
// observation|separator|action interleave (:350-400) and the left / right padding (:408-431).
//
// HBM-bound: one warp owns one output position; it derives (timestep, slot) arithmetically from the
// sample descriptor, computes the id (lane-uniform), then streams the d-float row with 128-bit
// loads/stores.  Algorithmic bytes per token: d*4 (table row) + d*4 (output row) + 16 (id + masks).
#include "common.cuh"
#include "ordered.cuh"

namespace neko {

enum Slot { SLOT_PAD = 0, SLOT_PATCH, SLOT_TEXT, SLOT_COBS, SLOT_DOBS, SLOT_SEP, SLOT_CACT, SLOT_DACT };

struct SlotInfo {
  int kind;
  int t;       // timestep
  int j;       // slot inside the timestep (position-embedding row for observation slots)
  int k;       // index inside the modality block
};

__device__ __forceinline__ SlotInfo locate(const neko_sample_desc& sd, int s, int seq_len) {
  SlotInfo r;
  r.kind = SLOT_PAD; r.t = 0; r.j = 0; r.k = 0;
  if (s < sd.seq_off || s >= seq_len) return r;  // left pad, or right pad of --pad_seq
  const int n_obs = sd.n_patches + sd.n_text + sd.n_cobs + sd.n_dobs;
  const int tpt = n_obs + 1 + sd.n_cact + sd.n_dact;
  const int p = s - sd.seq_off;
  r.t = p / tpt;
  int j = p - r.t * tpt;
  r.j = j;
  if (j < sd.n_patches) { r.kind = SLOT_PATCH; r.k = j; return r; }
  j -= sd.n_patches;
  if (j < sd.n_text) { r.kind = SLOT_TEXT; r.k = j; return r; }
  j -= sd.n_text;
  if (j < sd.n_cobs) { r.kind = SLOT_COBS; r.k = j; return r; }
  j -= sd.n_cobs;
  if (j < sd.n_dobs) { r.kind = SLOT_DOBS; r.k = j; return r; }
  j -= sd.n_dobs;
  if (j == 0) { r.kind = SLOT_SEP; return r; }
  j -= 1;
  if (j < sd.n_cact) { r.kind = SLOT_CACT; r.k = j; return r; }
  j -= sd.n_cact;
  r.kind = SLOT_DACT; r.k = j;
  return r;
}

// ContinuousTokenizer.encode (input_tokenizers.py:17-30) with torch-CPU rounding: every op is a
// separately rounded fp32 op (no FMA contraction), the division is IEEE, and the logarithm is
// correctly rounded (fp64 log rounded once), see DESIGN.md "bit-exact bins".
__device__ __forceinline__ int discretize(float x, bool mu_law, float mu, float denom, float half_bins) {
  float y = x;
  if (mu_law) {
    const float a = fabsf(x);
    float t = __fmul_rn(mu, a);
    t = __fadd_rn(1.0f, t);
    const float lg = (float)log((double)t);
    const float sgn = (x > 0.0f) ? 1.0f : ((x < 0.0f) ? -1.0f : 0.0f);
    const float num = __fmul_rn(sgn, lg);
    y = __fdiv_rn(num, denom);
  }
  y = fminf(fmaxf(y, -1.0f), 1.0f);
  y = __fadd_rn(y, 1.0f);
  y = __fmul_rn(y, half_bins);
  return (int)y;  // truncation toward zero, like .type(torch.int32)
}

struct TokArgs {
  const neko_sample_desc* descs;
  int B, d;
  neko_tok_params p;
  float mu_denom;  // fp32(log(1 + mu*M))
  const float* fvals;
  const int32_t* ivals;
  const float* patch_emb;
  const float* embed_table;
  const float* pos_table;
  const float* sep_vec;
  int64_t* tokens;
  float* target_masks;
  float* token_masks;
  float* emb;
  int32_t* err_flag;
};

__device__ __forceinline__ long long slot_token(const TokArgs& a, const neko_sample_desc& sd, const SlotInfo& si,
                                                float* target) {
  long long id = 0;
  float tgt = 0.0f;
  switch (si.kind) {
    case SLOT_TEXT:
      id = a.ivals[sd.text_off + si.t * sd.n_text + si.k];
      tgt = 1.0f;
      break;
    case SLOT_COBS:
      id = discretize(a.fvals[sd.cobs_off + si.t * sd.n_cobs + si.k], true, a.p.mu, a.mu_denom,
                      0.5f * (float)a.p.n_bins) + a.p.cont_start;
      break;
    case SLOT_DOBS:
      id = (long long)a.ivals[sd.dobs_off + si.t * sd.n_dobs + si.k] + a.p.disc_start;
      break;
    case SLOT_CACT:
      id = discretize(a.fvals[sd.cact_off + si.t * sd.n_cact + si.k], false, a.p.mu, a.mu_denom,
                      0.5f * (float)a.p.n_bins) + a.p.cont_start;
      tgt = 1.0f;
      break;
    case SLOT_DACT:
      id = (long long)a.ivals[sd.dact_off + si.t * sd.n_dact + si.k] + a.p.disc_start;
      tgt = 1.0f;
      break;
    default:  // pad, patch, separator: id 0, target 0
      break;
  }
  *target = tgt;
  return id;
}

// PACKED: warps still walk (b, s) of the padded grid (s < seq_len); a valid position writes row row_base + (s - seq_off)
// of the packed outputs and a padding position writes nothing.
template <bool PACKED>
__global__ void __launch_bounds__(256) tokenize_embed_kernel(TokArgs a) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int width = PACKED ? a.p.seq_len : a.p.width;
  if (warp >= a.B * width) return;
  const int b = warp / width;
  const int s = warp - b * width;
  const neko_sample_desc sd = a.descs[b];
  const SlotInfo si = locate(sd, s, a.p.seq_len);
  if (PACKED && si.kind == SLOT_PAD) return;
  const int row = PACKED ? sd.row_base + (s - sd.seq_off) : warp;
  float tgt;
  const long long id = slot_token(a, sd, si, &tgt);
  if (lane == 0) {
    a.tokens[row] = id;
    a.target_masks[row] = tgt;
    a.token_masks[row] = (si.kind == SLOT_PAD) ? 0.0f : 1.0f;
  }
  if (a.emb == nullptr) return;

  const int d = a.d;
  float4* out = reinterpret_cast<float4*>(a.emb + (size_t)row * d);
  const int nv = d >> 2;
  if (si.kind == SLOT_PAD) {
    for (int i = lane; i < nv; i += 32) out[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  const float* src;
  if (si.kind == SLOT_PATCH) {
    src = a.patch_emb + ((size_t)sd.patch_off + (size_t)si.t * sd.n_patches + si.k) * d;
  } else if (si.kind == SLOT_SEP) {
    src = a.sep_vec;
  } else {
    if (id < 0 || id >= a.p.vocab) {
      if (lane == 0 && a.err_flag) atomicExch(a.err_flag, 1);
      for (int i = lane; i < nv; i += 32) out[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      return;
    }
    src = a.embed_table + (size_t)id * d;
  }
  const bool add_pos = a.p.use_pos && si.kind >= SLOT_PATCH && si.kind <= SLOT_DOBS;
  const float4* s4 = reinterpret_cast<const float4*>(src);
  if (add_pos) {
    const float4* p4 = reinterpret_cast<const float4*>(a.pos_table + (size_t)si.j * d);
    for (int i = lane; i < nv; i += 32) {
      float4 v = __ldg(s4 + i);
      const float4 q = __ldg(p4 + i);
      v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
      out[i] = v;
    }
  } else {
    for (int i = lane; i < nv; i += 32) out[i] = __ldg(s4 + i);
  }
}

// Backward: each warp routes one position's gradient row.
struct EmbBwdArgs {
  const neko_sample_desc* descs;
  int B, d;
  neko_tok_params p;
  const int64_t* tokens;
  const float* d_emb;
  float* d_embed_table;
  float* d_pos_table;
  float* d_sep;
  float* d_patch_emb;
};

template <bool PACKED>
__global__ void __launch_bounds__(256) embed_bwd_kernel(EmbBwdArgs a) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int width = PACKED ? a.p.seq_len : a.p.width;
  if (warp >= a.B * width) return;
  const int b = warp / width;
  const int s = warp - b * width;
  const neko_sample_desc sd = a.descs[b];
  const SlotInfo si = locate(sd, s, a.p.seq_len);
  if (si.kind == SLOT_PAD) return;
  const int row = PACKED ? sd.row_base + (s - sd.seq_off) : warp;
  const int d = a.d;
  const float* g = a.d_emb + (size_t)row * d;
  float* dst = nullptr;
  bool atomic = true;
  if (si.kind == SLOT_PATCH) {
    if (a.d_patch_emb) {
      dst = a.d_patch_emb + ((size_t)sd.patch_off + (size_t)si.t * sd.n_patches + si.k) * d;
      atomic = false;  // each patch row is used by exactly one position
    }
  } else if (si.kind == SLOT_SEP) {
    dst = a.d_sep;
  } else {
    const long long id = a.tokens[row];
    if (id >= 0 && id < a.p.vocab) dst = a.d_embed_table + (size_t)id * d;
  }
  const bool add_pos = a.p.use_pos && si.kind >= SLOT_PATCH && si.kind <= SLOT_DOBS;
  float* pos = add_pos ? a.d_pos_table + (size_t)si.j * d : nullptr;
  for (int i = lane; i < d; i += 32) {
    const float v = g[i];
    if (dst) {
      if (atomic) atomicAdd(dst + i, v); else dst[i] = v;
    }
    if (pos) atomicAdd(pos + i, v);
  }
}

template <bool PACKED>
static int tokenize_embed(const neko_sample_desc* descs, int B, int d, const neko_tok_params* hp, const float* fvals,
                          const int32_t* ivals, const float* patch_emb, const float* embed_table, const float* pos_table,
                          const float* sep_vec, int64_t* tokens, float* target_masks, float* token_masks,
                          float* token_embeddings, int32_t* err_flag, void* stream) {
  NEKO_REQUIRE(descs && hp && tokens && target_masks && token_masks, "tokenize: null pointer");
  NEKO_REQUIRE(B > 0 && hp->width >= hp->seq_len && hp->seq_len > 0, "tokenize: bad B/seq_len/width");
  if (token_embeddings) {
    NEKO_REQUIRE(d > 0 && d % 4 == 0, "tokenize: embed_dim must be a multiple of 4 (got %d)", d);
    NEKO_REQUIRE(embed_table && sep_vec && (pos_table || !hp->use_pos), "tokenize: null table pointer");
  }
  TokArgs a;
  a.descs = descs; a.B = B; a.d = d; a.p = *hp;
  a.mu_denom = (float)log(1.0 + (double)hp->mu * (double)hp->M);
  a.fvals = fvals; a.ivals = ivals; a.patch_emb = patch_emb; a.embed_table = embed_table;
  a.pos_table = pos_table; a.sep_vec = sep_vec; a.tokens = tokens; a.target_masks = target_masks;
  a.token_masks = token_masks; a.emb = token_embeddings; a.err_flag = err_flag;
  const long long warps = (long long)B * (PACKED ? hp->seq_len : hp->width);
  const int threads = 256;
  const long long blocks = (warps * 32 + threads - 1) / threads;
  tokenize_embed_kernel<PACKED><<<(unsigned)blocks, threads, 0, as_stream(stream)>>>(a);
  NEKO_LAUNCH_CHECK("tokenize_embed_kernel");
  return NEKO_OK;
}

template <bool PACKED>
static int embed_bwd(const neko_sample_desc* descs, int B, int d, const neko_tok_params* hp, const int64_t* tokens,
                     const float* d_token_embeddings, float* d_embed_table, float* d_pos_table, float* d_sep,
                     float* d_patch_emb, void* stream) {
  NEKO_REQUIRE(descs && hp && tokens && d_token_embeddings && d_embed_table && d_sep, "embed_bwd: null pointer");
  NEKO_REQUIRE(d_pos_table || !hp->use_pos, "embed_bwd: null d_pos_table");
  EmbBwdArgs a;
  a.descs = descs; a.B = B; a.d = d; a.p = *hp; a.tokens = tokens; a.d_emb = d_token_embeddings;
  a.d_embed_table = d_embed_table; a.d_pos_table = d_pos_table; a.d_sep = d_sep; a.d_patch_emb = d_patch_emb;
  const long long warps = (long long)B * (PACKED ? hp->seq_len : hp->width);
  const int threads = 256;
  const long long blocks = (warps * 32 + threads - 1) / threads;
  embed_bwd_kernel<PACKED><<<(unsigned)blocks, threads, 0, as_stream(stream)>>>(a);
  NEKO_LAUNCH_CHECK("embed_bwd_kernel");
  return NEKO_OK;
}

// Ordered backward (deterministic mode): one warp per grid position writes two sort keys -- [0, n) the table row (embed_token
// row id, or vocab for the separator), [n, 2n) the position-table row (vocab + 1 + j) -- with the position's gradient row as
// value; positions without a target get the sentinel key.  Patch rows are copied (one writer per row).  The sorted segments
// are then summed in ascending source-row order (ordered.cu).
template <bool PACKED>
__global__ void __launch_bounds__(256) embed_keys_kernel(EmbBwdArgs a, unsigned* __restrict__ keys, int* __restrict__ vals) {
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int width = PACKED ? a.p.seq_len : a.p.width;
  const long long n = (long long)a.B * width;
  if (warp >= n) return;
  const int b = (int)(warp / width);
  const int s = (int)(warp - (long long)b * width);
  const neko_sample_desc sd = a.descs[b];
  const SlotInfo si = locate(sd, s, a.p.seq_len);
  const unsigned sentinel = (unsigned)(a.p.vocab + 1 + a.p.ctx_rows);
  unsigned tk = sentinel, pk = sentinel;
  int row = 0;
  if (si.kind != SLOT_PAD) {
    row = PACKED ? sd.row_base + (s - sd.seq_off) : (int)warp;
    if (si.kind == SLOT_PATCH) {
      if (a.d_patch_emb) {
        const float4* g = reinterpret_cast<const float4*>(a.d_emb + (size_t)row * a.d);
        float4* dst = reinterpret_cast<float4*>(a.d_patch_emb + ((size_t)sd.patch_off + (size_t)si.t * sd.n_patches + si.k) * a.d);
        for (int i = lane; i < (a.d >> 2); i += 32) dst[i] = g[i];
      }
    } else if (si.kind == SLOT_SEP) {
      tk = (unsigned)a.p.vocab;
    } else {
      const long long id = a.tokens[row];
      if (id >= 0 && id < a.p.vocab) tk = (unsigned)id;
    }
    if (a.p.use_pos && si.kind >= SLOT_PATCH && si.kind <= SLOT_DOBS && si.j < a.p.ctx_rows) pk = (unsigned)(a.p.vocab + 1 + si.j);
  }
  if (lane == 0) {
    keys[warp] = tk; vals[warp] = row;
    keys[n + warp] = pk; vals[n + warp] = row;
  }
}

static int embed_ord_check(const neko_tok_params* hp, int B) {
  NEKO_REQUIRE(hp && B > 0 && hp->seq_len > 0 && hp->width >= hp->seq_len && hp->vocab > 0 && hp->ctx_rows >= 0,
               "embed_bwd_ordered: bad B / seq_len / width / vocab / ctx_rows");
  NEKO_REQUIRE((long long)B * hp->width <= (1LL << 29) && (long long)hp->vocab + hp->ctx_rows < (1LL << 30),
               "embed_bwd_ordered: problem too large");
  return NEKO_OK;
}

template <bool PACKED>
static int embed_bwd_ordered(const neko_sample_desc* descs, int B, int d, const neko_tok_params* hp, const int64_t* tokens,
                             const float* d_token_embeddings, float* d_embed_table, float* d_pos_table, float* d_sep,
                             float* d_patch_emb, void* workspace, int64_t workspace_bytes, void* stream) {
  NEKO_REQUIRE(descs && hp && tokens && d_token_embeddings && d_embed_table && d_sep && workspace, "embed_bwd_ordered: null pointer");
  NEKO_REQUIRE(d_pos_table || !hp->use_pos, "embed_bwd_ordered: null d_pos_table");
  int rc = embed_ord_check(hp, B);
  if (rc != NEKO_OK) return rc;
  NEKO_REQUIRE(d > 0 && d % 4 == 0, "embed_bwd_ordered: embed_dim must be a multiple of 4 (got %d)", d);
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  NEKO_REQUIRE(al16(d_token_embeddings) && al16(d_embed_table) && al16(d_pos_table) && al16(d_sep) && al16(d_patch_emb) &&
               (reinterpret_cast<uintptr_t>(workspace) & 255) == 0,
               "embed_bwd_ordered: gradient buffers must be 16-byte aligned, the workspace 256-byte aligned");
  const long long n = (long long)B * (PACKED ? hp->seq_len : hp->width);
  const int end_bit = key_bits((unsigned)(hp->vocab + 1 + hp->ctx_rows));
  SortWs s;
  rc = sort_ws_layout(2 * n, end_bit, workspace, s);
  if (rc != NEKO_OK) return rc;
  NEKO_REQUIRE(workspace_bytes >= (int64_t)s.total, "embed_bwd_ordered: workspace of %lld bytes, need %lld", (long long)workspace_bytes,
               (long long)s.total);
  EmbBwdArgs a;
  a.descs = descs; a.B = B; a.d = d; a.p = *hp; a.tokens = tokens; a.d_emb = d_token_embeddings;
  a.d_embed_table = d_embed_table; a.d_pos_table = d_pos_table; a.d_sep = d_sep; a.d_patch_emb = d_patch_emb;
  embed_keys_kernel<PACKED><<<(unsigned)((n * 32 + 255) / 256), 256, 0, as_stream(stream)>>>(a, s.kin, s.vin);
  NEKO_LAUNCH_CHECK("embed_keys_kernel");
  SegDst dst{};
  dst.p[0] = d_embed_table; dst.p[1] = d_sep; dst.p[2] = d_pos_table;
  dst.off[0] = 0; dst.off[1] = hp->vocab; dst.off[2] = hp->vocab + 1; dst.off[3] = hp->vocab + 1 + hp->ctx_rows;
  return sort_and_segsum(s, 2 * n, end_bit, d_token_embeddings, d, dst, as_stream(stream));
}

}  // namespace neko

extern "C" {

int64_t neko_embed_bwd_ordered_workspace_bytes(int B, const neko_tok_params* host_params) {
  using namespace neko;
  const int rc = embed_ord_check(host_params, B);
  if (rc != NEKO_OK) return rc;
  SortWs s;
  const int r2 = sort_ws_layout(2LL * B * host_params->width, key_bits((unsigned)(host_params->vocab + 1 + host_params->ctx_rows)), nullptr, s);
  if (r2 != NEKO_OK) return r2;
  return (int64_t)s.total;
}

int neko_embed_bwd_ordered(const neko_sample_desc* descs, int B, int d, const neko_tok_params* hp, const int64_t* tokens,
                           const float* d_token_embeddings, float* d_embed_table, float* d_pos_table, float* d_sep, float* d_patch_emb,
                           void* workspace, int64_t workspace_bytes, void* stream) {
  return neko::embed_bwd_ordered<false>(descs, B, d, hp, tokens, d_token_embeddings, d_embed_table, d_pos_table, d_sep, d_patch_emb,
                                        workspace, workspace_bytes, stream);
}

int neko_embed_packed_bwd_ordered(const neko_sample_desc* descs, int B, int d, const neko_tok_params* hp, const int64_t* tokens,
                                  const float* d_token_embeddings, float* d_embed_table, float* d_pos_table, float* d_sep,
                                  float* d_patch_emb, void* workspace, int64_t workspace_bytes, void* stream) {
  return neko::embed_bwd_ordered<true>(descs, B, d, hp, tokens, d_token_embeddings, d_embed_table, d_pos_table, d_sep, d_patch_emb,
                                       workspace, workspace_bytes, stream);
}

int neko_tokenize_embed_fwd(const neko_sample_desc* descs, int B, int d, const neko_tok_params* hp,
                            const float* fvals, const int32_t* ivals, const float* patch_emb,
                            const float* embed_table, const float* pos_table, const float* sep_vec,
                            int64_t* tokens, float* target_masks, float* token_masks,
                            float* token_embeddings, int32_t* err_flag, void* stream) {
  return neko::tokenize_embed<false>(descs, B, d, hp, fvals, ivals, patch_emb, embed_table, pos_table, sep_vec, tokens,
                                     target_masks, token_masks, token_embeddings, err_flag, stream);
}

int neko_tokenize_embed_packed_fwd(const neko_sample_desc* descs, int B, int d, const neko_tok_params* hp,
                                   const float* fvals, const int32_t* ivals, const float* patch_emb,
                                   const float* embed_table, const float* pos_table, const float* sep_vec,
                                   int64_t* tokens, float* target_masks, float* token_masks,
                                   float* token_embeddings, int32_t* err_flag, void* stream) {
  return neko::tokenize_embed<true>(descs, B, d, hp, fvals, ivals, patch_emb, embed_table, pos_table, sep_vec, tokens,
                                    target_masks, token_masks, token_embeddings, err_flag, stream);
}

int neko_embed_bwd(const neko_sample_desc* descs, int B, int d, const neko_tok_params* hp,
                   const int64_t* tokens, const float* d_token_embeddings, float* d_embed_table,
                   float* d_pos_table, float* d_sep, float* d_patch_emb, void* stream) {
  return neko::embed_bwd<false>(descs, B, d, hp, tokens, d_token_embeddings, d_embed_table, d_pos_table, d_sep, d_patch_emb, stream);
}

int neko_embed_packed_bwd(const neko_sample_desc* descs, int B, int d, const neko_tok_params* hp,
                          const int64_t* tokens, const float* d_token_embeddings, float* d_embed_table,
                          float* d_pos_table, float* d_sep, float* d_patch_emb, void* stream) {
  return neko::embed_bwd<true>(descs, B, d, hp, tokens, d_token_embeddings, d_embed_table, d_pos_table, d_sep, d_patch_emb, stream);
}

}  // extern "C"
