// Device building blocks of the CTC prefix beam search, shared by the whole-call decoder (ctc_decode.cu) and the
// streaming keyword spotter (kws_stream.cu).  Bit-exact restatement of wekws/model/loss.py:229-306 and its per-frame
// twin wekws/bin/stream_kws_ctc.py:124-215, including the parts that only exist because of Python object semantics:
//   * probabilities are float32 values promoted to double, every update is the same sequence of double multiplies and
//     adds (no FMA contraction), `math.isclose(p, 0.0, abs_tol=1e-6)` is |p| <= 1e-6;
//   * path nodes are dict OBJECTS shared between hypotheses by the shallow `cur_nodes.copy()`: `nodes[-1]['prob'] = ps`
//     (loss.py:273-275) is visible through every list that holds the same dict.  Nodes therefore live in a pool and the
//     hypotheses hold node ids; "pop + append" (loss.py:296-297) allocates a fresh node;
//   * `next_hyps` is a dict in insertion order and `sorted(..., reverse=True)` is stable: ties keep insertion order;
//   * is_sublist never tests the last possible offset when the prefix is longer than the keyword (score_ctc.py:95).
#pragma once
#include <math.h>

#include "../../include/wekws_b200.h"

namespace wekws {
namespace beam {

constexpr int ML = WEKWS_CTC_MAX_PREFIX;      // longest prefix / node list kept (overflow is flagged)
constexpr int PBM = WEKWS_CTC_MAX_PATH_BEAM;  // path_beam_size limit
constexpr int SBM = WEKWS_CTC_MAX_SCORE_BEAM; // score_beam_size limit
constexpr int NEXTM = PBM * (SBM + 1);        // keys next_hyps can hold: old prefixes + one extension per token
constexpr int POOLM = PBM * ML + PBM * SBM + 8;

struct Hyp {
  double pb, pnb;
  int32_t len, nlen;          // prefix length, node-list length (equal except transiently empty lists)
  int16_t tok[ML];
  int16_t node[ML];
};

struct Work {                 // one utterance's decoder state (shared memory)
  Hyp cur[PBM];
  Hyp next[NEXTM];
  int32_t nframe[POOLM];      // node pool: frame, prob, token
  float nprob[POOLM];
  int16_t ntok[POOLM];
  int16_t remap[POOLM];
  int32_t ncur, npool, overflow;
  uint8_t order[NEXTM];
};

__device__ __forceinline__ bool close0(double p) { return fabs(p) <= 1e-6; }   // math.isclose(p, 0.0, abs_tol=1e-6)

// cur_hyps = [(tuple(), (1.0, 0.0, []))]; the node pool is emptied, the overflow flag is kept
__device__ __forceinline__ void init_hyps(Work& w) {
  w.ncur = 1; w.npool = 0;
  w.cur[0].pb = 1.0; w.cur[0].pnb = 0.0; w.cur[0].len = 0; w.cur[0].nlen = 0;
}

// find the entry with this prefix (tok[0..len) [+ extra]) or insert an empty one -- defaultdict((0.0, 0.0, []))
__device__ inline int find_or_insert(Work& w, int& nnext, const int16_t* tok, int len, int extra /* -1 = none */) {
  const int L = len + (extra >= 0 ? 1 : 0);
  for (int e = 0; e < nnext; ++e) {
    const Hyp& h = w.next[e];
    if (h.len != L) continue;
    bool same = true;
    for (int i = 0; i < len && same; ++i) same = h.tok[i] == tok[i];
    if (same && extra >= 0) same = h.tok[len] == (int16_t)extra;
    if (same) return e;
  }
  if (nnext >= NEXTM) return -1;
  Hyp& h = w.next[nnext];
  h.pb = 0.0; h.pnb = 0.0; h.len = L; h.nlen = 0;
  for (int i = 0; i < len; ++i) h.tok[i] = tok[i];
  if (extra >= 0) h.tok[len] = (int16_t)extra;
  return nnext++;
}

__device__ __forceinline__ void copy_nodes(Hyp& dst, const Hyp& src) {            // nodes = cur_nodes.copy()
  dst.nlen = src.nlen;
  for (int i = 0; i < src.nlen; ++i) dst.node[i] = src.node[i];
}

__device__ __forceinline__ int new_node(Work& w, int tok, int frame, float prob) {
  if (w.npool >= POOLM) { w.overflow = 1; return POOLM - 1; }
  const int id = w.npool++;
  w.ntok[id] = (int16_t)tok; w.nframe[id] = frame; w.nprob[id] = prob;
  return id;
}

// one frame of loss.py:229-306 / stream_kws_ctc.py:140-213 for the filtered tokens s[0..ns) with probabilities ps[]
__device__ inline void advance(Work& w, int t, const int* s_idx, const float* s_prob, int ns, int path_beam) {
  int nnext = 0;
  for (int k = 0; k < ns; ++k) {
    const int s = s_idx[k];
    const float psf = s_prob[k];
    const double ps = (double)psf;
    for (int hi = 0; hi < w.ncur; ++hi) {
      const Hyp& c = w.cur[hi];
      const int last = c.len > 0 ? c.tok[c.len - 1] : -1;
      const double pb = c.pb, pnb = c.pnb;
      if (s == 0) {                                               // blank
        const int e = find_or_insert(w, nnext, c.tok, c.len, -1);
        if (e < 0) { w.overflow = 1; continue; }
        Hyp& n = w.next[e];
        n.pb = __dadd_rn(__dadd_rn(n.pb, __dmul_rn(pb, ps)), __dmul_rn(pnb, ps));
        copy_nodes(n, c);
      } else if (s == last) {
        if (!close0(pnb)) {                                       // *ss -> *s
          const int e = find_or_insert(w, nnext, c.tok, c.len, -1);
          if (e < 0) { w.overflow = 1; continue; }
          Hyp& n = w.next[e];
          n.pnb = __dadd_rn(n.pnb, __dmul_rn(pnb, ps));
          copy_nodes(n, c);
          const int id = n.node[n.nlen - 1];
          if (psf > w.nprob[id]) { w.nprob[id] = psf; w.nframe[id] = t; }   // the shared dict is updated in place
        }
        if (!close0(pb)) {                                        // *s-s -> *ss
          if (c.len >= ML) { w.overflow = 1; continue; }
          const int e = find_or_insert(w, nnext, c.tok, c.len, s);
          if (e < 0) { w.overflow = 1; continue; }
          Hyp& n = w.next[e];
          n.pnb = __dadd_rn(n.pnb, __dmul_rn(pb, ps));
          copy_nodes(n, c);
          n.node[n.nlen++] = (int16_t)new_node(w, s, t, psf);
        }
      } else {
        if (c.len >= ML) { w.overflow = 1; continue; }
        const int e = find_or_insert(w, nnext, c.tok, c.len, s);
        if (e < 0) { w.overflow = 1; continue; }
        Hyp& n = w.next[e];
        if (n.nlen > 0) {
          if (psf > w.nprob[n.node[n.nlen - 1]]) n.node[n.nlen - 1] = (int16_t)new_node(w, s, t, psf);   // pop + append
        } else {
          copy_nodes(n, c);
          n.node[n.nlen++] = (int16_t)new_node(w, s, t, psf);
        }
        n.pnb = __dadd_rn(__dadd_rn(n.pnb, __dmul_rn(pb, ps)), __dmul_rn(pnb, ps));
      }
    }
  }
  // stable sort by pb + pnb, descending (insertion sort on an index array keeps ties in insertion order)
  for (int e = 0; e < nnext; ++e) {
    const double key = __dadd_rn(w.next[e].pb, w.next[e].pnb);
    int p = e;
    while (p > 0) {
      const Hyp& o = w.next[w.order[p - 1]];
      if (__dadd_rn(o.pb, o.pnb) >= key) break;
      w.order[p] = w.order[p - 1];
      --p;
    }
    w.order[p] = (uint8_t)e;
  }
  const int keep = nnext < path_beam ? nnext : path_beam;
  // garbage-collect the node pool: keep the nodes the surviving hypotheses reference, ids stay in ascending order
  for (int i = 0; i < w.npool; ++i) w.remap[i] = 0;
  for (int r = 0; r < keep; ++r) {
    const Hyp& h = w.next[w.order[r]];
    for (int i = 0; i < h.nlen; ++i) w.remap[h.node[i]] = 1;
  }
  int live = 0;
  for (int i = 0; i < w.npool; ++i) {
    if (w.remap[i]) {
      w.ntok[live] = w.ntok[i]; w.nframe[live] = w.nframe[i]; w.nprob[live] = w.nprob[i];
      w.remap[i] = (int16_t)live++;
    }
  }
  w.npool = live;
  for (int r = 0; r < keep; ++r) {
    const Hyp& h = w.next[w.order[r]];
    Hyp& d = w.cur[r];
    d.pb = h.pb; d.pnb = h.pnb; d.len = h.len; d.nlen = h.nlen;
    for (int i = 0; i < h.len; ++i) d.tok[i] = h.tok[i];
    for (int i = 0; i < h.nlen; ++i) d.node[i] = w.remap[h.node[i]];
  }
  w.ncur = keep;
}

// keyword-token bitmap over V in shared memory (n_allowed == 0: every token passes); the whole warp calls this
__device__ __forceinline__ void build_allow(uint32_t* allow, int V, const int32_t* allowed, int n_allowed, int lane) {
  const int nwords = (V + 31) / 32;
  for (int i = lane; i < nwords; i += 32) allow[i] = n_allowed > 0 ? 0u : 0xffffffffu;
  __syncwarp();
  if (lane == 0) {
    for (int i = 0; i < n_allowed; ++i) {
      const int tkn = allowed[i];
      if (tkn >= 0 && tkn < V) allow[tkn >> 5] |= 1u << (tkn & 31);
    }
  }
}

// probs.topk(score_beam) of one frame p[0..V) followed by the filter "prob > 0.05 and token in the keyword set"
// (loss.py:243-255 / stream_kws_ctc.py:145-158).  Per-lane candidates, then SB rounds of warp arg-max (ties: lower
// index first).  The whole warp calls this; every lane gets the same (s_idx, s_prob, return value = count).
__device__ __forceinline__ int warp_topk_filter(const float* p, int V, int SB, const uint32_t* allow, int lane,
                                                int* s_idx, float* s_prob) {
  float bv[SBM];
  int bi[SBM];
#pragma unroll
  for (int k = 0; k < SBM; ++k) { bv[k] = -INFINITY; bi[k] = 0x7fffffff; }
  for (int i = lane; i < V; i += 32) {
    const float v = __ldg(p + i);
    if (v > bv[SBM - 1]) {                     // strictly greater: an equal later index never displaces an earlier one
      bv[SBM - 1] = v; bi[SBM - 1] = i;
#pragma unroll
      for (int k = SBM - 1; k > 0; --k) {
        if (bv[k] > bv[k - 1]) {
          const float tv = bv[k]; bv[k] = bv[k - 1]; bv[k - 1] = tv;
          const int ti = bi[k]; bi[k] = bi[k - 1]; bi[k - 1] = ti;
        }
      }
    }
  }
  int ns = 0;
  for (int k = 0; k < SB; ++k) {
    float mv = bv[0];
    int mi = bi[0];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, mv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
      if (ov > mv || (ov == mv && oi < mi)) { mv = ov; mi = oi; }
    }
    if (bi[0] == mi && mi != 0x7fffffff) {     // the winning lane pops its head
#pragma unroll
      for (int q = 0; q < SBM - 1; ++q) { bv[q] = bv[q + 1]; bi[q] = bi[q + 1]; }
      bv[SBM - 1] = -INFINITY; bi[SBM - 1] = 0x7fffffff;
    }
    // filter: prob > 0.05 (Python float compare of the float32 value) and token in the keyword set
    if (mi != 0x7fffffff && (double)mv > 0.05 && ((allow[mi >> 5] >> (mi & 31)) & 1u)) {
      s_idx[ns] = mi; s_prob[ns] = mv; ++ns;
    }
  }
  return ns;
}

// score_ctc.py:88-103 (identical copy in stream_kws_ctc.py:105-120), quirk included: for a longer main list the loop
// runs over range(len(main) - len(check)) and never tests the last offset
template <typename T>
__device__ inline int is_sublist(const T* main_list, int nm, const int32_t* check, int nc) {
  if (nm < nc) return -1;
  if (nm == nc) {
    for (int i = 0; i < nc; ++i)
      if ((int32_t)main_list[i] != check[i]) return -1;
    return 0;
  }
  for (int i = 0; i < nm - nc; ++i) {
    if ((int32_t)main_list[i] == check[0]) {
      int j = 0;
      while (j < nc && (int32_t)main_list[i + j] == check[j]) ++j;
      if (j == nc) return i;
    }
  }
  return -1;
}

}  // namespace beam
}  // namespace wekws
