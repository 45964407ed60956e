// kernels_encode.cu -- board -> network input planes, move -> policy index, and the deterministic test
// evaluator.
//
// Replaces netencoder.get_game_state (netencoder.py:13-91) and the uci_dict gather of
// AgentDistributed.predict_policy (agentdistributed.py:31-32, 80-82).
//
// Plane layout written here: bf16 [row][8][8][128] NHWC, row 0 = rank 8, column 0 = file a; channel
// 14*s + {0: no black piece, 1..6: black P N B R Q K, 7: no white piece, 8..13: white P..K} for state s
// (s = 0 current position, s = 1..8 after undoing s plies, all-zero when the move stack is shorter),
// channel 126 = side to move (1 = white), channel 127 = zero padding so K is a multiple of 64 for the
// tcgen05 convolution.  HBM-bound: 580 B read, 16,384 B written per position, 16-byte stores, a full
// 2 KB contiguous span per block-wide store.
#include "engine.cuh"
#include "hash_eval.cuh"
#include "search_targets.cuh"

namespace crl {

static constexpr int ENC_THREADS = 128;

struct EncShared {
  u64 bb[9][8];
  int avail;   // number of states present (1 + min(8, ply))
  int turn;
};

// All threads of the block write the 64 x 128 plane tile of one position.
// Step 1: one thread per square folds the 9 states into a 128-bit channel mask (14 bits per state: "no black piece",
// six black piece bits, "no white piece", six white piece bits; bit 126 = side to move).  Step 2: all threads expand
// mask bytes to bf16 and store 16 bytes each, 2 KB contiguous per block-wide store -- the kernel is then bound by the
// 16 KB it writes per position, not by bit fiddling.
// OutT = uint8_t: e4m3 planes for the fp8 tower (1.0 = 0x38), 8 KB per position.
template <int T, class OutT = __nv_bfloat16>
__device__ __forceinline__ void write_planes(const EncShared& s, unsigned (*s_mask)[4],
                                             OutT* __restrict__ out) {
  if (threadIdx.x < 64) {
    const int cell = threadIdx.x;
    const int sq = (7 - (cell >> 3)) * 8 + (cell & 7);
    u64 lo = 0, hi = 0;
    for (int st = 0; st < s.avail; ++st) {
      const unsigned ob = (unsigned)((s.bb[st][OCC_B] >> sq) & 1), ow = (unsigned)((s.bb[st][OCC_W] >> sq) & 1);
      unsigned pt = 0;
#pragma unroll
      for (int k = 0; k < 6; ++k) pt |= (unsigned)((s.bb[st][k] >> sq) & 1) << k;
      const u64 m14 = (u64)((ob ^ 1u) | ((ob ? pt : 0u) << 1) | ((ow ^ 1u) << 7) | ((ow ? pt : 0u) << 8));
      const int o = 14 * st;
      if (o < 64) {
        lo |= m14 << o;
        if (o > 50) hi |= m14 >> (64 - o);
      } else {
        hi |= m14 << (o - 64);
      }
    }
    hi |= (u64)(s.turn & 1) << 62;   // channel 126
    s_mask[cell][0] = (unsigned)lo;
    s_mask[cell][1] = (unsigned)(lo >> 32);
    s_mask[cell][2] = (unsigned)hi;
    s_mask[cell][3] = (unsigned)(hi >> 32);
  }
  __syncthreads();
  uint4* dst = reinterpret_cast<uint4*>(out);
  if constexpr (sizeof(OutT) == 1) {
#pragma unroll
    for (int j = 0; j < 512 / T; ++j) {
      const int id = j * T + threadIdx.x;           // 16-byte chunk id: 64 squares x 8 chunks of 16 channels
      const int cell = id >> 3, chunk = id & 7;
      const unsigned bits = (s_mask[cell][chunk >> 1] >> ((chunk & 1) * 16)) & 0xFFFFu;
      uint32_t w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        w[k] = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) w[k] |= ((bits >> (4 * k + b)) & 1u) ? (0x38u << (8 * b)) : 0u;
      }
      dst[id] = make_uint4(w[0], w[1], w[2], w[3]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 1024 / T; ++j) {
      const int id = j * T + threadIdx.x;             // 16-byte chunk id: 64 squares x 16 chunks of 8 channels
      const int cell = id >> 4, chunk = id & 15;
      const unsigned bits = (s_mask[cell][chunk >> 2] >> ((chunk & 3) * 8)) & 0xFFu;
      uint4 q;
      q.x = ((bits & 1) ? 0x3F80u : 0u) | ((bits & 2) ? 0x3F800000u : 0u);
      q.y = ((bits & 4) ? 0x3F80u : 0u) | ((bits & 8) ? 0x3F800000u : 0u);
      q.z = ((bits & 16) ? 0x3F80u : 0u) | ((bits & 32) ? 0x3F800000u : 0u);
      q.w = ((bits & 64) ? 0x3F80u : 0u) | ((bits & 128) ? 0x3F800000u : 0u);
      dst[id] = q;
    }
  }
}

// stateless: boards + explicit history arrays
__global__ void __launch_bounds__(ENC_THREADS) k_encode_boards(const u64* __restrict__ boards,
                                                               const u64* __restrict__ hist,
                                                               const u8* __restrict__ hist_len, int n,
                                                               __nv_bfloat16* __restrict__ planes) {
  __shared__ EncShared s;
  __shared__ unsigned s_mask[64][4];
  const int i = blockIdx.x;
  if (threadIdx.x < 72) {
    const int st = threadIdx.x >> 3, k = threadIdx.x & 7;
    const int hl = (hist && hist_len) ? min((int)hist_len[i], 8) : 0;
    u64 v = 0;
    if (st == 0) v = boards[(long long)k * n + i];
    else if (st - 1 < hl) v = hist[((long long)(st - 1) * 8 + k) * n + i];
    s.bb[st][k] = v;
    if (threadIdx.x == 0) {
      s.avail = 1 + hl;
      s.turn = (int)(boards[8LL * n + i] & 1);
    }
  }
  __syncthreads();
  write_planes<ENC_THREADS>(s, s_mask, planes + (long long)i * 64 * 128);
}

// tree / game batches: row r -> slot eval_list[r] (game = slot / K); position = (s_node[slot], which) or the root
// when which==0.  64 threads per row: the history walk is a short pointer chase by one thread, and with 32 resident
// blocks per SM a whole 4,096-row batch is one wave, so every chase overlaps the other rows' stores.
static constexpr int ENC_ROW_THREADS = 64;
template <class OutT>
__global__ void __launch_bounds__(ENC_ROW_THREADS) k_encode_rows(Pools P, int which, OutT* __restrict__ planes) {
  __shared__ EncShared s;
  __shared__ unsigned s_mask[64][4];
  const int r = blockIdx.x;
  if (r >= *P.eval_n) return;
  const int slot = P.eval_list[r];
  const int g = slot / P.K;
  if (threadIdx.x == 0) {
    const int node = which == 0 ? 0 : P.s_node[slot];
    const int w = which == 0 ? 2 : which;
    const NodeRec& nr = P.nodes[(long long)g * P.NN + node];
    const u64 meta = (w == 2 ? nr.p2 : nr.p1)[8];
    Cursor c{node, w, meta_ply(meta)};
    cursor_bitboards(P, g, c, s.bb[0]);
    int cnt = 1;
    while (cnt < 9 && cursor_prev(P, g, c)) {
      cursor_bitboards(P, g, c, s.bb[cnt]);
      ++cnt;
    }
    s.avail = cnt;
    s.turn = (int)(meta & 1);
  }
  __syncthreads();
  write_planes<ENC_ROW_THREADS, OutT>(s, s_mask, planes + (long long)r * 64 * 128);
}

__global__ void k_policy_index(const u16* __restrict__ moves, const int* __restrict__ counts, int n,
                               const int16_t* __restrict__ label_of, int16_t* __restrict__ idx) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * MAX_MOVES) return;
  const int i = (int)(t / MAX_MOVES), k = (int)(t % MAX_MOVES);
  int16_t v = -1;
  if (k < counts[i]) {
    u16 m = moves[t];
    if (m != MOVE_NONE && mv_promo(m) < 5) v = label_of[(int)mv_promo(m) * 4096 + mv_from(m) * 64 + mv_to(m)];
  }
  idx[t] = v;
}

// ---- search targets (crl_search_targets, DESIGN.md 3.8) -----------------------------------------------------
// One block per row.  Thread 0 regenerates the legal moves into shared memory and reduces best and the sum in
// generation order (search_targets.cuh); meanwhile the block zero-fills the row.  After the barrier each thread
// scatters some of the n probabilities.  A row's bits depend on its own inputs only.
static constexpr int ST_THREADS = 128;
__global__ void __launch_bounds__(ST_THREADS) k_search_targets(const u64* __restrict__ boards,
                                                               const int* __restrict__ scores,
                                                               const int* __restrict__ offsets, int n,
                                                               float temperature, const int16_t* __restrict__ label_of,
                                                               float* __restrict__ policy,
                                                               float* __restrict__ score_value,
                                                               int* __restrict__ legal_count) {
  __shared__ u16 s_moves[MAX_MOVES];
  __shared__ SearchRowStats s_r;
  __shared__ int s_n;
  const int i = blockIdx.x;
  const int o = offsets[i], ns = offsets[i + 1] - o;
  const int* s = scores + o;
  float* row = policy + (long long)i * CRL_N_LABELS;
  if (threadIdx.x == 0) {
    const Board b = load_soa(boards, n, i);
    StoreSink sink{s_moves, 0};
    generate_legal(b, sink);
    legal_count[i] = sink.n;
    float v = 0.0f;
    int use = 0;                                       // a count mismatch leaves the row zero (the caller reports it)
    if (sink.n == ns && ns > 0) {
      s_r = search_row_stats(s, ns, temperature);
      v = search_score_value(s_r.best, meta_turn(b.meta));
      use = ns;
    }
    s_n = use;
    score_value[i] = v;
  }
  for (int l = threadIdx.x; l < CRL_N_LABELS; l += ST_THREADS) row[l] = 0.0f;
  __syncthreads();
  for (int k = threadIdx.x; k < s_n; k += ST_THREADS) {
    const int l = search_label(label_of, s_moves[k]);
    if (l >= 0) row[l] = search_prob(s[k], s_r, temperature);
  }
}

int launch_search_targets(crl_engine_impl* e, const u64* boards, const int* scores, const int* offsets, int n,
                          float temperature, float* policy, float* score_value, int* legal_count) {
  if (n <= 0) return CRL_OK;
  LaunchScope ls(e, KC_ENCODE);
  k_search_targets<<<n, ST_THREADS, 0, e->stream>>>(boards, scores, offsets, n, temperature, e->d_label_of, policy,
                                                     score_value, legal_count);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}

// ---- deterministic test evaluator ---------------------------------------------------------------------
__device__ __forceinline__ void hash_eval_row(const Board& b, u64 seed, int bits, float* __restrict__ policy_row,
                                              float* __restrict__ value) {
  const u64 h = eval_hash(b, seed);
  for (int l = threadIdx.x; l < CRL_N_LABELS; l += blockDim.x) policy_row[l] = hash_policy(h, l, bits);
  if (threadIdx.x == 0) *value = hash_value(h);
}

__global__ void __launch_bounds__(256) k_hash_eval_boards(const u64* __restrict__ boards, int n, u64 seed,
                                                          int bits, float* __restrict__ policy,
                                                          float* __restrict__ value) {
  const int i = blockIdx.x;
  Board b = load_soa(boards, n, i);
  hash_eval_row(b, seed, bits, policy + (long long)i * CRL_N_LABELS, value + i);
}

__global__ void __launch_bounds__(256) k_hash_eval_rows(Pools P, int which, u64 seed, int bits,
                                                        float* __restrict__ policy, float* __restrict__ value) {
  const int r = blockIdx.x;
  if (r >= *P.eval_n) return;
  const int slot = P.eval_list[r];
  const int g = slot / P.K;
  const int node = which == 0 ? 0 : P.s_node[slot];
  const NodeRec& nr = P.nodes[(long long)g * P.NN + node];
  Board b = load_rec((which == 1) ? nr.p1 : nr.p2);
  hash_eval_row(b, seed, bits, policy + (long long)r * CRL_N_LABELS, value + r);
}

int launch_encode_boards(crl_engine_impl* e, const u64* boards, const u64* hist, const u8* hist_len, int n,
                         __nv_bfloat16* planes) {
  if (n <= 0) return CRL_OK;
  LaunchScope ls(e, KC_ENCODE);
  k_encode_boards<<<n, ENC_THREADS, 0, e->stream>>>(boards, hist, hist_len, n, planes);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}
int launch_policy_index(crl_engine_impl* e, const u16* moves, const int* counts, int n, int16_t* idx) {
  if (n <= 0) return CRL_OK;
  LaunchScope ls(e, KC_ENCODE);
  k_policy_index<<<div_up((long long)n * MAX_MOVES, 256), 256, 0, e->stream>>>(moves, counts, n, e->d_label_of, idx);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}
int launch_hash_eval_boards(crl_engine_impl* e, const u64* boards, int n, u64 seed, int bits, float* policy,
                            float* value) {
  if (n <= 0) return CRL_OK;
  LaunchScope ls(e, KC_HASHEVAL);
  k_hash_eval_boards<<<n, 256, 0, e->stream>>>(boards, n, seed, bits, policy, value);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}

// Encodes the positions named by P.eval_list (which: 0 root, 1 state after our move, 2 node state) and runs
// the configured evaluator on them; results land in e->d_policy / e->d_value, row r <-> game eval_list[r].
// With two network slots in the search, each slot's share of the batch (its list and row count, at rows
// k * slot_stride + r) is encoded in the slot's plane dtype and evaluated by the slot's evaluator; the search reads
// both shares through slot 0's view, at their rows.
int launch_eval_batch(crl_engine_impl* e, int which) {
  for (int k = 0; k < e->search_slots; ++k) {
    Pools P = e->P;
    const long long off = (long long)k * e->slot_stride;
    P.eval_list += off;
    P.eval_n += SLOT_N_STRIDE * k;
    float* policy = e->d_policy + off * CRL_N_LABELS;
    float* value = e->d_value + off;
    PolicyView view;
    if (e->eval_kind[k] == CRL_EVAL_HASH) {
      LaunchScope ls(e, KC_HASHEVAL);
      k_hash_eval_rows<<<e->cur_rows, 256, 0, e->stream>>>(P, which, e->eval_seed[k], e->eval_bits[k], policy, value);
      CRL_CUDA(cudaGetLastError());
      view = PolicyView{e->d_policy, CRL_N_LABELS, nullptr};
    } else {
      void* planes = net_planes_buf(e, k);
      if (!planes) {
        set_error("network slot %d has no weights (crl_net_load_host)", k);
        return CRL_ESTATE;
      }
      {
        LaunchScope ls(e, KC_ENCODE);
        if (net_fp8(e, k))   // the fp8 tower reads e4m3 rows from the same buffer
          k_encode_rows<uint8_t><<<e->cur_rows, ENC_ROW_THREADS, 0, e->stream>>>(P, which, (uint8_t*)planes);
        else
          k_encode_rows<__nv_bfloat16><<<e->cur_rows, ENC_ROW_THREADS, 0, e->stream>>>(P, which, (__nv_bfloat16*)planes);
        CRL_CUDA(cudaGetLastError());
      }
      int rc = net_forward_slot(e, k, planes, e->cur_rows, P.eval_n, policy, value, &view);
      if (rc != CRL_OK) return rc;
    }
    if (k == 0) e->pview = view;
  }
  return CRL_OK;
}

}  // namespace crl
