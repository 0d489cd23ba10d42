// Stage (c): per-joint top-k (k = max_num_people) of the NMS'd heatmap with the tie order of
// the reference's CPU run (grouping.py:147-170).
//
// torch's CPU topk for k*64 <= n is std::partial_sort over (value, index) pairs with a
// value-only comparator (aten/src/ATen/native/TopKImpl.h), i.e. libstdc++'s __heap_select +
// __sort_heap: a k-entry heap whose top is the smallest kept value, fed by the stream in index
// order; an element enters only if it is STRICTLY greater than the current top.  Among equal
// values the final order is therefore a function of the heap's history, not of the indices
// (SURVEY.md App. A.4).  Per (image, joint) row:
//   * the heap top never decreases, so the row is streamed through the per-word maxima of the NMS'd
//     values written by the aggregation kernel (32 words = 1024 pixels per step); only words that can
//     still contain an entering element are expanded (one coalesced 128-byte line of the heatmap + the
//     survivor mask word, up to 8 words per batch of loads);
//   * floor mode: the word maxima also give a lower bound of the M-th largest value before the row is
//     streamed; a sorted-across-the-lanes sink started at that floor yields the M largest values, which is
//     the answer whenever it is free of ties;
//   * otherwise the heap history is replayed exactly: the libstdc++ heap with slot i in lane i
//     (WarpHeap), or -- force_generic bit 0 -- the literal __adjust_heap / __push_heap code run by lane 0
//     on shared memory (HeapSink), kept as the anchor the other two are tested against.
// One warp per row (topk_kernel) or, for small batches, 8 warps per row (topk_split_kernel).
// The NMS'd value of a suppressed pixel is x*0 (sign of x): zeros do enter while the top is
// negative and their indices are part of the bit-exact contract.
#include "common.cuh"
#ifdef HPD_TOPK_PROFILE
#include <cstdio>
#endif

namespace hpd {

namespace {

// -DHPD_TOPK_PROFILE: the first few tied rows print clock64() per phase of topk_tied_rows_kernel (development aid)
#ifdef HPD_TOPK_PROFILE
__device__ int tp_printed = 0;
#define TP_MARK(i) do { tp[i] = clock64(); } while (0)
#else
#define TP_MARK(i)
#endif

constexpr int kTopkWarps = 4;

struct HeapRef {
  float* v;
  int* i;
};

// comp(a, b) of the reference's lambda: a.value > b.value (finite inputs)
__device__ __forceinline__ bool comp_gt(float a, float b) { return a > b; }

// libstdc++ std::__push_heap
__device__ __forceinline__ void push_heap(HeapRef h, int hole, int top, float val, int idx) {
  int parent = (hole - 1) / 2;
  while (hole > top && comp_gt(h.v[parent], val)) {
    h.v[hole] = h.v[parent];
    h.i[hole] = h.i[parent];
    hole = parent;
    parent = (hole - 1) / 2;
  }
  h.v[hole] = val;
  h.i[hole] = idx;
}

// libstdc++ std::__adjust_heap
__device__ __forceinline__ void adjust_heap(HeapRef h, int hole, int len, float val, int idx) {
  const int top = hole;
  int child = hole;
  while (child < (len - 1) / 2) {
    child = 2 * (child + 1);
    if (comp_gt(h.v[child], h.v[child - 1])) --child;
    h.v[hole] = h.v[child];
    h.i[hole] = h.i[child];
    hole = child;
  }
  if ((len & 1) == 0 && child == (len - 2) / 2) {
    child = 2 * (child + 1);
    h.v[hole] = h.v[child - 1];
    h.i[hole] = h.i[child - 1];
    hole = child - 1;
  }
  push_heap(h, hole, top, val, idx);
}

__device__ __forceinline__ void make_heap(HeapRef h, int len) {
  if (len < 2) return;
  int parent = (len - 2) / 2;
  while (true) {
    const float v = h.v[parent];
    const int i = h.i[parent];
    adjust_heap(h, parent, len, v, i);
    if (parent == 0) return;
    --parent;
  }
}

__device__ __forceinline__ void sort_heap(HeapRef h, int len) {
  int last = len;
  while (last > 1) {
    --last;
    const float v = h.v[last];
    const int i = h.i[last];
    h.v[last] = h.v[0];
    h.i[last] = h.i[0];
    adjust_heap(h, 0, last, v, i);
  }
}

// ---- exact sink: the libstdc++ heap in shared memory, edited by lane 0 -----------------------------
struct HeapSink {
  HeapRef h;
  int M, lane;
  float top;
  __device__ __forceinline__ void init(float nv) {   // lane < M holds element `lane` of the row
    if (lane < M) { h.v[lane] = nv; h.i[lane] = lane; }
    __syncwarp();
    if (lane == 0) make_heap(h, M);
    __syncwarp();
    top = h.v[0];
  }
  __device__ __forceinline__ void insert(float cv, int idx) {   // std::__heap_select: __pop_heap(first, middle, i)
    if (lane == 0) adjust_heap(h, 0, M, cv, idx);
    __syncwarp();
    top = h.v[0];
  }
  template <bool EQ>
  __device__ __forceinline__ void feed(float cv, int idx) {
    if (cv > top) insert(cv, idx);
  }
};

// ---- exact sink, warp-wide: the same libstdc++ heap with slot i held by lane i --------------------------
// __adjust_heap walks down choosing, per level, between two siblings, then __push_heap walks back up
// comparing the value with the elements of that path.  Both kinds of comparison are made for the whole
// heap at once -- lane k compares node k's two children, every lane compares its element with the value
// -- and collected by two ballots; the walk itself is then scalar bit arithmetic, and all element moves
// along the path are one shuffle.  Same comparisons, same outcome as the functions above, ~3x fewer
// cycles per insertion than lane 0 editing shared memory.
struct WarpHeap {
  int lane;
  unsigned anc;   // ancestors of this lane's node below the root, the node itself included (bit k for node k)
  float v;
  int i;
  __device__ __forceinline__ void setup(int lane_) {
    lane = lane_;
    anc = 0;
    for (int k = lane_; k >= 1; k = (k - 1) >> 1) anc |= 1u << k;
  }
  __device__ __forceinline__ void adjust(int hole, int len, float val, int idx) {
    const int lc = min(2 * lane + 1, 31), rc = min(2 * lane + 2, 31);
    const float right = __shfl_sync(kFull, v, rc), left = __shfl_sync(kFull, v, lc);
    const unsigned take_left = __ballot_sync(kFull, comp_gt(right, left));   // bit k: comp(first[2k+2], first[2k+1])
    const unsigned above = __ballot_sync(kFull, comp_gt(v, val));            // bit n: comp(first[n], value)
    int p[7];
    p[0] = hole;
    int n = 0, child = hole;
    bool finished = false;
#pragma unroll
    for (int k = 1; k <= 6; ++k) {
      p[k] = 0;
      if (!finished) {
        if (child < (len - 1) / 2) {
          int c = 2 * (child + 1);
          if ((take_left >> child) & 1u) --c;
          p[k] = c; n = k; child = c;
        } else {
          if ((len & 1) == 0 && child == (len - 2) / 2) { p[k] = 2 * (child + 1) - 1; n = k; }
          finished = true;
        }
      }
    }
    // __push_heap from the leaf: climbs while the element above (the one just moved up) is greater
    int j = n;
#pragma unroll
    for (int k = 6; k >= 1; --k)
      if (k <= n && j == k && ((above >> p[k]) & 1u)) j = k - 1;
    int src = lane;
#pragma unroll
    for (int k = 0; k < 6; ++k)
      if (k < j && lane == p[k]) src = p[k + 1];
    const float nv = __shfl_sync(kFull, v, src);
    const int ni = __shfl_sync(kFull, i, src);
    v = nv; i = ni;
    int pj = p[0];
#pragma unroll
    for (int k = 1; k <= 6; ++k)
      if (k == j) pj = p[k];
    if (lane == pj) { v = val; i = idx; }
  }
  // __adjust_heap(first, 0, len, value) -- the call __heap_select and __sort_heap make -- without the level-by-level
  // walk.  Node k lies on the sift-down path iff every node from k up to (not including) the root was the child
  // its parent chose, and "was chosen" is one comparison with the sibling: a left child (odd k) is taken when
  // comp(right, left) or when it has no right sibling (the lone child of an even-length heap), a right child
  // otherwise.  One ballot collects those bits, one AND against the lane's ancestor mask says whether the lane is
  // on the path, and since children have larger indices than parents the path in depth order is the path mask in
  // bit order: __push_heap stops at the deepest path node whose element is not greater than the value (highest
  // such bit), every path node above it takes its path child's element (one shuffle), that node takes the value.
  // Same comparisons, same outcome as adjust(0, len, ...); ~3 ballots + 2 shuffles deep instead of a 6-level chain.
  // GUARDED: the sift happens only if comp(value, first[0]), i.e. value > top -- __heap_select's test -- decided
  // inside by a ballot that is issued together with the others instead of ahead of them (no branch on the way).
  template <bool GUARDED = false>
  __device__ __forceinline__ void adjust_root(int len, float val, int idx) {
    const int sib = (lane & 1) ? lane + 1 : lane - 1;
    const float sv = __shfl_sync(kFull, v, sib & 31);
    bool chosen = false;
    if (lane >= 1 && lane < len) {
      if (lane & 1) chosen = (lane + 1 < len) ? comp_gt(sv, v) : true;   // left child: comp(right, left), or alone
      else chosen = !comp_gt(v, sv);                                    // right child: !comp(right, left)
    }
    const unsigned sel = __ballot_sync(kFull, chosen);
    const bool on_path = lane >= 1 && (sel & anc) == anc;
    const unsigned path = __ballot_sync(kFull, on_path);               // nodes of the path below the root
    const unsigned above = __ballot_sync(kFull, comp_gt(v, val));      // bit n: comp(first[n], value)
    const bool enter = !GUARDED || (__ballot_sync(kFull, lane == 0 && comp_gt(val, v)) != 0u);
    const unsigned stop = path & ~above;
    const int t = stop ? 31 - __clz(stop) : 0;                         // where the value lands
    int src = lane;
    if (enter && (lane == 0 || on_path) && lane < t) src = ((path >> (2 * lane + 1)) & 1u) ? 2 * lane + 1 : 2 * lane + 2;
    const float nv = __shfl_sync(kFull, v, src);
    const int ni = __shfl_sync(kFull, i, src);
    v = nv; i = ni;
    if (enter && lane == t) { v = val; i = idx; }
  }
  __device__ __forceinline__ void make(int len) {
    if (len < 2) return;
    for (int parent = (len - 2) / 2; parent >= 0; --parent)
      adjust(parent, len, __shfl_sync(kFull, v, parent), __shfl_sync(kFull, i, parent));
  }
  __device__ __forceinline__ void sort(int len) {
    for (int last = len - 1; last >= 1; --last) {
      const float val = __shfl_sync(kFull, v, last), v0 = __shfl_sync(kFull, v, 0);
      const int idx = __shfl_sync(kFull, i, last), i0 = __shfl_sync(kFull, i, 0);
      if (lane == last) { v = v0; i = i0; }
      adjust_root(last, val, idx);
    }
  }
};

struct WarpHeapSink {
  WarpHeap h;
  int M, lane;
  float top;
  __device__ __forceinline__ void init(float nv) {   // lane < M holds element `lane` of the row
    h.setup(lane);
    h.v = nv;
    h.i = lane;
    h.make(M);
    top = __shfl_sync(kFull, h.v, 0);
  }
  __device__ __forceinline__ void insert(float cv, int idx) {
    h.adjust_root(M, cv, idx);
    top = __shfl_sync(kFull, h.v, 0);
  }
  template <bool EQ>
  __device__ __forceinline__ void feed(float cv, int idx) {
    if (cv > top) insert(cv, idx);
  }
};

// ---- fast sink: the M kept elements sorted by value across the lanes of the warp ---------------------
// The heap's VALUE dynamics do not depend on its arrangement (an element enters iff it is strictly
// greater than the smallest kept value, and a smallest-valued element leaves), so a sorted register
// array evolves through the same multisets.  Which of several EQUAL elements leaves, and the final
// order of equal elements, is where the heap arrangement matters; `ambiguous()` detects every such
// case (two equal values among the final M, or an evicted value equal to the final minimum -- the
// +-0 tail of a channel with fewer than M positive peaks always lands here) and the row is then
// replayed with the exact sink.  Otherwise the result (distinct values, descending) is what
// sort_heap produces from any arrangement.
struct SortedSink {
  int M, lane;
  float sv;       // lane i < M: i-th largest kept value (lanes >= M: -inf)
  int si;
  float top;      // smallest kept value
  float evicted;  // value of the last evicted element (evictions are non-decreasing)
  bool any_evicted;
  // log of the entering elements, in order: the exact sink goes through the same VALUE history, so a
  // replay only has to feed it this list instead of scanning the row again
  float* log_v;
  int* log_i;
  int n_log, log_cap;
  float rej_eq;   // merge only: largest value that arrived equal to the then-smallest kept value
  __device__ __forceinline__ void init_empty() {   // M slots of -inf: the first M arrivals fill them
    n_log = 0;
    sv = -INFINITY;
    si = -1;
    top = -INFINITY;
    evicted = -INFINITY;
    rej_eq = -INFINITY;
    any_evicted = false;
  }
  // M placeholders of value `floor_v` (index -1): for a row known to hold at least M elements above
  // floor_v the placeholders are all evicted by the end, and nothing at or below floor_v is ever looked at
  __device__ __forceinline__ void init_floor(float floor_v) {
    n_log = 0;
    sv = lane < M ? floor_v : -INFINITY;
    si = -1;
    top = floor_v;
    evicted = -INFINITY;
    rej_eq = -INFINITY;
    any_evicted = false;
  }
  __device__ __forceinline__ void offer(float cv, int idx) {   // any value may be offered
    if (cv > top) insert(cv, idx);
    else if (cv == top) rej_eq = cv;
  }
  template <bool EQ>
  __device__ __forceinline__ void feed(float cv, int idx) {
    if (EQ) offer(cv, idx);
    else if (cv > top) insert(cv, idx);
  }
  __device__ __forceinline__ void init(float nv) {
    n_log = 0;
    rej_eq = -INFINITY;
    sv = lane < M ? nv : -INFINITY;
    si = lane;
    // bitonic sort, descending by value
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
      for (int j = k >> 1; j > 0; j >>= 1) {
        const float ov = __shfl_xor_sync(kFull, sv, j);
        const int oi = __shfl_xor_sync(kFull, si, j);
        const bool up = ((lane & k) == 0);          // this k-block sorts descending
        const bool lower = ((lane & j) == 0);       // this lane keeps the larger (if up) element
        const bool take = (lower == up) ? (ov > sv) : (ov < sv);
        if (take) { sv = ov; si = oi; }
      }
    }
    top = __shfl_sync(kFull, sv, M - 1);
    evicted = -INFINITY;
    any_evicted = false;
  }
  __device__ __forceinline__ void insert(float cv, int idx) {   // requires cv > top
    const int pos = __popc(__ballot_sync(kFull, lane < M && sv >= cv));
    const float uv = __shfl_up_sync(kFull, sv, 1);
    const int ui = __shfl_up_sync(kFull, si, 1);
    evicted = top;
    any_evicted = true;
    if (lane == 0 && n_log < log_cap) { log_v[n_log] = cv; log_i[n_log] = idx; }
    ++n_log;
    if (lane < M) {
      if (lane > pos) { sv = uv; si = ui; }
      else if (lane == pos) { sv = cv; si = idx; }
    }
    top = __shfl_sync(kFull, sv, M - 1);
  }
  __device__ __forceinline__ bool ambiguous() const {
    const float nxt = __shfl_down_sync(kFull, sv, 1);
    const bool tie = __ballot_sync(kFull, lane < M - 1 && sv == nxt) != 0u;
    return tie || (any_evicted && evicted == top) || rej_eq == top;
  }
};

// Stream one row through a sink in index order.  The per-word maxima are scanned 128 words at a time
// (the next 128 are prefetched while this group is processed); words that can still hold an
// entering element are expanded up to 8 at a time so that their heatmap lines and mask words are
// fetched together instead of one DRAM round trip each.
// EQ: elements EQUAL to the sink's smallest kept value are fed too (the floor mode needs to see them to
// know whether its result is free of ties); otherwise only strictly greater ones, as the heap admits.
// row_max: an upper bound of every word maximum in the range; once the sink's smallest kept value has reached it
// nothing can enter any more and the scan stops (a channel without positive peaks is done after its first words).
template <typename Sink, bool EQ = false>
__device__ __forceinline__ void scan_range(Sink& sink, const float* __restrict__ hm, const uint32_t* __restrict__ mk,
                                           const float* __restrict__ wm, int W, int wpr, int w_begin, int w_end,
                                           int first_idx, int lane, float row_max = INFINITY) {
  // words [w_begin, w_end) of the row; pixels with flat index < first_idx are not offered (they are the
  // initial heap of the sequential algorithm)
  const int nwords = w_end;
  constexpr int kGroup = 4, kSlots = 8, kAhead = 4;
  // word maxima are loaded kAhead groups (of 128 words) ahead of their use
  float ring[kAhead][kGroup];
#pragma unroll
  for (int a = 0; a < kAhead; ++a)
#pragma unroll
    for (int u = 0; u < kGroup; ++u) {
      const int wd = w_begin + 32 * (a * kGroup + u) + lane;
      ring[a][u] = wd < nwords ? wm[wd] : -INFINITY;
    }
  for (int base = w_begin; base < nwords; base += 32 * kGroup) {
    if (!(EQ ? (row_max >= sink.top) : (row_max > sink.top))) return;
    float cur[kGroup];
#pragma unroll
    for (int u = 0; u < kGroup; ++u) {
      cur[u] = ring[0][u];
#pragma unroll
      for (int a = 0; a + 1 < kAhead; ++a) ring[a][u] = ring[a + 1][u];
      const int wd = base + 32 * (kAhead * kGroup + u) + lane;
      ring[kAhead - 1][u] = wd < nwords ? wm[wd] : -INFINITY;
    }
#pragma unroll
    for (int u = 0; u < kGroup; ++u) {
      const int cbase = base + 32 * u;
      uint32_t pass = __ballot_sync(kFull, EQ ? (cur[u] >= sink.top) : (cur[u] > sink.top));
      while (pass) {
        float hv[kSlots];
        uint32_t mw[kSlots];
        int wl[kSlots];
#pragma unroll
        for (int s = 0; s < kSlots; ++s) {
          wl[s] = -1;
          hv[s] = 0.f;
          mw[s] = 0u;
          if (pass) {
            const int l = __ffs(pass) - 1;
            pass &= pass - 1;
            wl[s] = l;
            const int w2 = cbase + l;
            const int y = w2 / wpr, x = (w2 - y * wpr) * 32 + lane;
            const int idx = y * W + x;
            if (x < W && idx >= first_idx) hv[s] = hm[idx];
            mw[s] = mk[w2];
          }
        }
#pragma unroll
        for (int s = 0; s < kSlots; ++s) {
          if (wl[s] < 0) break;
          const float wmx = __shfl_sync(kFull, cur[u], wl[s]);
          if (!(EQ ? (wmx >= sink.top) : (wmx > sink.top))) continue;   // the top may have risen meanwhile
          const int w2 = cbase + wl[s];
          const int y = w2 / wpr, x0 = (w2 - y * wpr) * 32;
          const bool valid = (x0 + lane < W) && (y * W + x0 + lane >= first_idx);
          const bool keep = (mw[s] >> lane) & 1u;
          const float nv = keep ? hv[s] : __fmul_rn(hv[s], 0.0f);
          uint32_t cand = __ballot_sync(kFull, valid && (EQ ? (nv >= sink.top) : (nv > sink.top)));
          while (cand) {
            const int j = __ffs(cand) - 1;
            cand &= cand - 1;
            const float cv = __shfl_sync(kFull, nv, j);
            sink.template feed<EQ>(cv, y * W + x0 + j);
          }
        }
      }
    }
  }
}

// ---- a floor for the M-th largest value of words [w_begin, w_end) -------------------------------------
// Every word maximum is the NMS'd value of a distinct pixel, so the M-th largest of any set of word
// maxima is a lower bound of the M-th largest pixel value.  Each lane keeps the 4 largest of the maxima it
// streams (the true top M are spread over the lanes, so the 128 candidates nearly always contain them);
// pop() removes the largest candidate of the warp.
struct WordMaxCandidates {
  float t0, t1, t2, t3;   // descending
  __device__ __forceinline__ void feed(float x) {
    const float a = fminf(t0, x); t0 = fmaxf(t0, x);
    const float b = fminf(t1, a); t1 = fmaxf(t1, a);
    const float c = fminf(t2, b); t2 = fmaxf(t2, b);
    t3 = fmaxf(t3, c);
  }
  __device__ __forceinline__ void scan(const float* __restrict__ wm, int w_begin, int w_end, int lane) {
    t0 = t1 = t2 = t3 = -INFINITY;
    constexpr int U = 8;
    if ((reinterpret_cast<uintptr_t>(wm + w_begin) & 15) == 0) {
      // 16-byte loads, 8 in flight per lane: 4 KB of word maxima per warp and round trip (the maxima of a
      // 512x512 plane are 32 KB that the aggregation kernel's map writes have pushed out of L2)
      for (int base = w_begin; base < w_end; base += 128 * U) {
        float4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          // which lane reads which 16 bytes of a 128-word chunk rotates from chunk to chunk: maps with regular
          // structure (a border column, artefacts with a period of a few rows) would otherwise put all their large
          // maxima into the same few lanes, and a lane keeps only four
          const int chunk = ((base - w_begin) >> 7) + u;
          const int wd = base + 128 * u + 4 * ((lane + 5 * chunk) & 31);
          if (wd + 3 < w_end) {
            v[u] = *reinterpret_cast<const float4*>(wm + wd);
          } else {
            v[u].x = wd < w_end ? wm[wd] : -INFINITY;
            v[u].y = wd + 1 < w_end ? wm[wd + 1] : -INFINITY;
            v[u].z = wd + 2 < w_end ? wm[wd + 2] : -INFINITY;
            v[u].w = -INFINITY;
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) { feed(v[u].x); feed(v[u].y); feed(v[u].z); feed(v[u].w); }
      }
      return;
    }
    for (int base = w_begin; base < w_end; base += 32 * U) {
      float v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int wd = base + 32 * u + lane;
        v[u] = wd < w_end ? wm[wd] : -INFINITY;
      }
#pragma unroll
      for (int u = 0; u < U; ++u) feed(v[u]);
    }
  }
  __device__ __forceinline__ float pop(int lane) {
    // order-preserving float -> unsigned map, warp max, the lowest lane holding it drops its head
    const unsigned bits = __float_as_uint(t0);
    const unsigned key = bits ^ ((bits >> 31) ? 0xffffffffu : 0x80000000u);
    const unsigned mx = __reduce_max_sync(kFull, key);
    const unsigned owners = __ballot_sync(kFull, key == mx);
    if (lane == __ffs(owners) - 1) { t0 = t1; t1 = t2; t2 = t3; t3 = -INFINITY; }
    const unsigned ob = mx ^ ((mx >> 31) ? 0x80000000u : 0xffffffffu);
    return __uint_as_float(ob);
  }
};

// largest float below a positive finite x
__device__ __forceinline__ float next_below(float x) { return __uint_as_float(__float_as_uint(x) - 1u); }

// NMS'd value of flat element `lane` (the sequential algorithm's initial heap is elements 0..M-1)
__device__ __forceinline__ float first_element(const float* __restrict__ hm, const uint32_t* __restrict__ mk, int W,
                                               int wpr, int M, int lane) {
  float nv = 0.f;
  if (lane < M) {
    const int y = lane / W, x = lane % W;
    const float v = hm[lane];
    const bool keep = (mk[(size_t)y * wpr + (x >> 5)] >> (x & 31)) & 1u;
    nv = keep ? v : __fmul_rn(v, 0.0f);
  }
  return nv;
}

// Floor mode's second pass over a whole row: only a few dozen words can hold an element at or above the floor.
// Streaming them through scan_range costs one DRAM round trip per 32-word group that has one (they are spread
// all over the row); here their indices are first compacted into a shared-memory list (the word maxima were read
// a moment ago, so this pass hits the cache) and then expanded eight at a time with all sixteen loads in flight.
// Returns false -- nothing fed, the sink untouched -- when the list does not fit (the caller then streams the row).
constexpr int kListCap = 256;

__device__ __forceinline__ bool scan_listed(SortedSink& sink, const float* __restrict__ hm, const uint32_t* __restrict__ mk,
                                            const float* __restrict__ wm, int W, int wpr, int nwords, int* __restrict__ list_w,
                                            float* __restrict__ list_m, int lane) {
  const float top0 = sink.top;
  int cnt = 0;
  constexpr int U = 8;
  for (int base = 0; base < nwords; base += 32 * U) {
    float v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int wd = base + 32 * u + lane;
      v[u] = wd < nwords ? wm[wd] : -INFINITY;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const bool hit = v[u] >= top0;
      const unsigned m = __ballot_sync(kFull, hit);
      if (m) {
        const int pos = cnt + __popc(m & ((1u << lane) - 1u));
        if (hit && pos < kListCap) { list_w[pos] = base + 32 * u + lane; list_m[pos] = v[u]; }
        cnt += __popc(m);
      }
    }
    if (cnt > kListCap) return false;
  }
  __syncwarp();
  if (cnt > 2 * sink.M) {
    // The floor came from four candidates per lane and can be loose.  The list holds EVERY word maximum at or above
    // it, the M largest included, so the M-th largest of (a per-lane top-4 of) the list is a better floor; listed
    // words below it are dropped before anything is loaded.
    WordMaxCandidates c2;
    c2.t0 = c2.t1 = c2.t2 = c2.t3 = -INFINITY;
    for (int i = lane; i < cnt; i += 32) c2.feed(list_m[i]);
    float f2 = -INFINITY;
    for (int r = 0; r < sink.M; ++r) f2 = c2.pop(lane);
    if (f2 > 0.f && next_below(f2) > sink.top) {
      sink.init_floor(next_below(f2));
      int kept = 0;
      for (int base = 0; base < cnt; base += 32) {
        const int i = base + lane;
        const int wv = i < cnt ? list_w[i] : 0;
        const float mv = i < cnt ? list_m[i] : -INFINITY;
        const bool hit = mv >= sink.top;
        const unsigned m = __ballot_sync(kFull, hit);
        __syncwarp();
        if (hit) {
          const int pos = kept + __popc(m & ((1u << lane) - 1u));
          list_w[pos] = wv; list_m[pos] = mv;
        }
        kept += __popc(m);
        __syncwarp();
      }
      cnt = kept;
    }
  }
  constexpr int kSlots = 8;
  for (int b0 = 0; b0 < cnt; b0 += kSlots) {
    float hv[kSlots];
    uint32_t mw[kSlots];
    int w2[kSlots];
#pragma unroll
    for (int s2 = 0; s2 < kSlots; ++s2) {
      w2[s2] = -1; hv[s2] = 0.f; mw[s2] = 0u;
      if (b0 + s2 < cnt) {
        w2[s2] = list_w[b0 + s2];
        const int y = w2[s2] / wpr, x = (w2[s2] - y * wpr) * 32 + lane;
        if (x < W) hv[s2] = hm[y * W + x];
        mw[s2] = mk[w2[s2]];
      }
    }
#pragma unroll
    for (int s2 = 0; s2 < kSlots; ++s2) {
      if (w2[s2] < 0) break;
      if (!(list_m[b0 + s2] >= sink.top)) continue;          // the top may have risen meanwhile
      const int y = w2[s2] / wpr, x0 = (w2[s2] - y * wpr) * 32;
      const bool keep = (mw[s2] >> lane) & 1u;
      const float nv = keep ? hv[s2] : __fmul_rn(hv[s2], 0.0f);
      uint32_t cand = __ballot_sync(kFull, (x0 + lane < W) && nv >= sink.top);
      while (cand) {
        const int j = __ffs(cand) - 1;
        cand &= cand - 1;
        sink.offer(__shfl_sync(kFull, nv, j), y * W + x0 + j);
      }
    }
  }
  return true;
}

template <typename Sink>
__device__ __forceinline__ void scan_row(Sink& sink, const float* __restrict__ hm, const uint32_t* __restrict__ mk,
                                         const float* __restrict__ wm, int H, int W, int wpr, int M, int lane,
                                         float row_max = INFINITY) {
  sink.init(first_element(hm, mk, W, wpr, M, lane));
  scan_range(sink, hm, mk, wm, W, wpr, 0, H * wpr, M, lane, row_max);
}

__global__ void __launch_bounds__(kTopkWarps * 32, 1) topk_kernel(const float* __restrict__ agg_hm,
                                                              const TagSource tags,
                                                              const uint32_t* __restrict__ mask,
                                                              const float* __restrict__ wmax, int rows, int H, int W,
                                                              int wpr, int E, int M, int force_exact, int defer_ties,
                                                              float* __restrict__ scores_k,
                                                              int32_t* __restrict__ idx_k,
                                                              int32_t* __restrict__ coords_k,
                                                              float* __restrict__ tags_k) {
  __shared__ float s_v[kTopkWarps][32];
  __shared__ int s_i[kTopkWarps][32];
  __shared__ int s_list_w[kTopkWarps][kListCap];
  __shared__ float s_list_m[kTopkWarps][kListCap];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * kTopkWarps + warp;
  if (row >= rows) return;
  const float* hm = agg_hm + (size_t)row * H * W;
  const uint32_t* mk = mask + (size_t)row * H * wpr;
  const float* wm = wmax + (size_t)row * H * wpr;

  float out_v = 0.f;
  int out_i = 0;
  bool done = false;
  float row_max = INFINITY;
#ifdef HPD_TOPK_PROFILE
  long long tp[8];
  int path = 0;
  float floor_dbg = 0.f;
#endif
  TP_MARK(0);
  if (!force_exact) {
    // Floor mode: with M word maxima above a positive floor the row holds M positive peaks, the stream can
    // start at that floor instead of at the row's first M elements, and only a few dozen words are ever
    // expanded.  Its value history is not the heap's, so it is only final when the result is free of ties
    // (distinct kept values, nothing else in the row equal to the smallest) -- then the M largest values in
    // descending order are what any history produces.
    WordMaxCandidates cand;
    cand.scan(wm, 0, H * wpr, lane);
    float floor_v = 0.f;
    for (int i = 0; i < M; ++i) {
      floor_v = cand.pop(lane);
      if (i == 0) row_max = floor_v;          // every lane's head is its true maximum: this is the row's largest
    }
    TP_MARK(1);
#ifdef HPD_TOPK_PROFILE
    floor_dbg = floor_v;
#endif
    if (floor_v > 0.f) {
      SortedSink fl;
      fl.M = M; fl.lane = lane;
      fl.log_v = nullptr; fl.log_i = nullptr; fl.log_cap = 0;
      fl.init_floor(next_below(floor_v));
      if (!scan_listed(fl, hm, mk, wm, W, wpr, H * wpr, s_list_w[warp], s_list_m[warp], lane)) {
#ifdef HPD_TOPK_PROFILE
        path |= 8;
#endif
        scan_range<SortedSink, true>(fl, hm, mk, wm, W, wpr, 0, H * wpr, 0, lane);
      }
#ifdef HPD_TOPK_PROFILE
      path |= 1;
#endif
      if (!fl.ambiguous()) { out_v = fl.sv; out_i = fl.si; done = true; }
      else if (defer_ties) {
        // Ties among M positive peaks (say, a peak on the image border, which the clamped bilinear taps
        // duplicate): the order among the equal values is the heap's history, ~M*ln(n/M) insertions.  One warp
        // would stream them for ~0.3 ms while the other thousand rows are long done, so the row is only marked
        // here and topk_tied_rows_kernel gives it eight warps.
        if (lane == 0) idx_k[(size_t)row * M] = -1;
        return;
      }
    }
  }
  if (!done && !force_exact) {
    // ties in play (always so for a channel with fewer than M positive peaks: its +-0 tail): stream the
    // row through the exact heap, slot i in lane i
    WarpHeapSink exact;
    exact.M = M; exact.lane = lane;
    scan_row(exact, hm, mk, wm, H, W, wpr, M, lane, row_max);
    exact.h.sort(M);
    out_v = exact.h.v; out_i = exact.h.i;
    done = true;
#ifdef HPD_TOPK_PROFILE
    path |= 2;
#endif
  }
#ifdef HPD_TOPK_PROFILE
  TP_MARK(2);
  if (lane == 0 && tp[2] - tp[0] > 60000)
    printf("slow row %d: floor %g path %d: maxima+pops %lld, rest %lld cycles\n", row, floor_dbg, path, tp[1] - tp[0], tp[2] - tp[1]);
#endif
  if (!done) {   // force_exact: the literal libstdc++ control flow, lane 0 editing shared memory
    HeapSink exact;
    exact.h = HeapRef{s_v[warp], s_i[warp]};
    exact.M = M; exact.lane = lane;
    scan_row(exact, hm, mk, wm, H, W, wpr, M, lane);
    __syncwarp();
    if (lane == 0) sort_heap(exact.h, M);
    __syncwarp();
    if (lane < M) { out_v = exact.h.v[lane]; out_i = exact.h.i[lane]; }
  }
  if (lane < M) {
    const size_t o = (size_t)row * M + lane;
    scores_k[o] = out_v;
    idx_k[o] = out_i;
    coords_k[o * 2 + 0] = out_i % W;
    coords_k[o * 2 + 1] = out_i / W;
    float tv[HPD_MAX_EMB];
    tag_value(tags, row, out_i, tv);
    tags_k[o * E] = tv[0];
    if (E > 1) tags_k[o * E + 1] = tv[1];
  }
}

// Small batches: kSplitWarps warps per (image, joint) row.  Every warp streams one contiguous segment of
// the row through its own sorted sink, started empty (a segment's smallest kept value never exceeds the
// sequential algorithm's at the same position, so the segment keeps and logs a superset of what enters
// there); warp 0 merges the segment lists.  The merged top M is final iff it is free of ties (no equal
// values among the top M, no other listed element equal to the M-th value, no segment evicted an element
// equal to it); otherwise warp 0 replays the concatenated segment logs, which are in index order, through
// the exact libstdc++ heap.
constexpr int kSplitWarps = 8;
constexpr int kSegLogCap = 320;

__global__ void __launch_bounds__(kSplitWarps * 32, 1) topk_split_kernel(const float* __restrict__ agg_hm,
                                                                     const TagSource tags,
                                                                     const uint32_t* __restrict__ mask,
                                                                     const float* __restrict__ wmax, int H, int W,
                                                                     int wpr, int E, int M, int force_exact,
                                                                     float* __restrict__ scores_k,
                                                                     int32_t* __restrict__ idx_k,
                                                                     int32_t* __restrict__ coords_k,
                                                                     float* __restrict__ tags_k) {
  __shared__ float s_v[kSplitWarps][32];
  __shared__ int s_i[kSplitWarps][32];
  __shared__ float s_logv[kSplitWarps][kSegLogCap];
  __shared__ int s_logi[kSplitWarps][kSegLogCap];
  __shared__ float s_evicted[kSplitWarps];
  __shared__ float s_rej[kSplitWarps];
  __shared__ int s_nlog[kSplitWarps];
  __shared__ float s_cand[kSplitWarps][8];
  __shared__ int s_floor_done;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x;
  const float* hm = agg_hm + (size_t)row * H * W;
  const uint32_t* mk = mask + (size_t)row * H * wpr;
  const float* wm = wmax + (size_t)row * H * wpr;
  const int nwords = H * wpr;
  const int groups = (nwords + 127) / 128;   // segment bounds in whole groups of 128 words
  const int gb = (groups * warp) / kSplitWarps, ge = (groups * (warp + 1)) / kSplitWarps;

  if (!force_exact) {
    // Floor mode (see topk_kernel): the floor is the M-th largest of the 8 largest word maxima of every
    // segment; each segment then keeps its elements above it and warp 0 merges.  Final only when free of
    // ties: distinct values, and no segment saw, evicted or turned away another element equal to the M-th.
    WordMaxCandidates cand;
    cand.scan(wm, gb * 128, min(ge * 128, nwords), lane);
    for (int r = 0; r < 8; ++r) {
      const float x = cand.pop(lane);
      if (lane == 0) s_cand[warp][r] = x;
    }
    if (threadIdx.x == 0) s_floor_done = 0;
    __syncthreads();
    static_assert(kSplitWarps * 8 == 64, "two candidates per lane below");
    const float c0 = (&s_cand[0][0])[2 * lane], c1 = (&s_cand[0][0])[2 * lane + 1];
    cand.t0 = fmaxf(c0, c1); cand.t1 = fminf(c0, c1); cand.t2 = cand.t3 = -INFINITY;
    float floor_v = 0.f;
    for (int r = 0; r < M; ++r) floor_v = cand.pop(lane);
    if (floor_v > 0.f) {   // uniform over the CTA
      SortedSink seg;
      seg.M = M; seg.lane = lane;
      seg.log_v = nullptr; seg.log_i = nullptr; seg.log_cap = 0;
      seg.init_floor(next_below(floor_v));
      scan_range<SortedSink, true>(seg, hm, mk, wm, W, wpr, gb * 128, min(ge * 128, nwords), 0, lane);
      s_v[warp][lane] = seg.sv;
      s_i[warp][lane] = seg.si;
      if (lane == 0) {
        s_evicted[warp] = seg.any_evicted ? seg.evicted : -INFINITY;
        s_rej[warp] = seg.rej_eq;
      }
      __syncthreads();
      if (warp == 0) {
        SortedSink all;
        all.M = M; all.lane = lane;
        all.log_v = nullptr; all.log_i = nullptr; all.log_cap = 0;
        all.init_empty();
        for (int w = 0; w < kSplitWarps; ++w) {
          const float cvl = s_v[w][lane];
          const int cil = s_i[w][lane];
          for (int j = 0; j < M; ++j) {           // descending; placeholders (index -1) come last
            const float cv = __shfl_sync(kFull, cvl, j);
            const int ci = __shfl_sync(kFull, cil, j);
            if (ci < 0 || cv < all.top) break;
            all.offer(cv, ci);
          }
        }
        bool amb = all.ambiguous();
        for (int w = 0; w < kSplitWarps; ++w) amb = amb || (s_evicted[w] == all.top) || (s_rej[w] == all.top);
        if (!amb) {
          if (lane < M) {
            const size_t o = (size_t)row * M + lane;
            scores_k[o] = all.sv;
            idx_k[o] = all.si;
            coords_k[o * 2 + 0] = all.si % W;
            coords_k[o * 2 + 1] = all.si / W;
            float tv[HPD_MAX_EMB];
            tag_value(tags, row, all.si, tv);
            tags_k[o * E] = tv[0];
            if (E > 1) tags_k[o * E + 1] = tv[1];
          }
          if (lane == 0) s_floor_done = 1;
        }
      }
      __syncthreads();
      if (s_floor_done) return;
    }
    SortedSink seg;
    seg.M = M; seg.lane = lane;
    seg.log_v = s_logv[warp]; seg.log_i = s_logi[warp]; seg.log_cap = kSegLogCap;
    seg.init_empty();
    scan_range(seg, hm, mk, wm, W, wpr, gb * 128, min(ge * 128, nwords), 0, lane);
    s_v[warp][lane] = seg.sv;
    s_i[warp][lane] = seg.si;
    if (lane == 0) {
      s_evicted[warp] = seg.any_evicted ? seg.evicted : -INFINITY;
      s_nlog[warp] = seg.n_log;
    }
  }
  __syncthreads();
  if (warp != 0) return;

  float out_v = 0.f;
  int out_i = 0;
  bool done = false, logs_ok = !force_exact;
  if (!force_exact) {
    SortedSink all;
    all.M = M; all.lane = lane;
    all.log_v = nullptr; all.log_i = nullptr; all.log_cap = 0;
    all.init_empty();
    for (int w = 0; w < kSplitWarps; ++w) {
      const float cvl = s_v[w][lane];
      const int cil = s_i[w][lane];
      for (int j = 0; j < M; ++j) {           // descending: stop at the first value that cannot matter
        const float cv = __shfl_sync(kFull, cvl, j);
        if (cv < all.top || cv == -INFINITY) break;
        all.offer(cv, __shfl_sync(kFull, cil, j));
      }
      logs_ok = logs_ok && s_nlog[w] <= kSegLogCap;
    }
    bool amb = all.ambiguous();
    for (int w = 0; w < kSplitWarps; ++w) amb = amb || (s_evicted[w] == all.top);
    if (!amb) { out_v = all.sv; out_i = all.si; done = true; }
  }
  if (!done && logs_ok) {
    // the logs hold a superset of the entering elements in index order: filter 32 entries at a time
    // against the live top, replay the survivors one by one through the exact heap (slot i in lane i)
    WarpHeapSink exact;
    exact.M = M; exact.lane = lane;
    exact.init(first_element(hm, mk, W, wpr, M, lane));
    for (int w = 0; w < kSplitWarps; ++w) {
      const int n = s_nlog[w];
      for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + lane;
        const float cv = i < n ? s_logv[w][i] : -INFINITY;
        const int ci = i < n ? s_logi[w][i] : 0;
        uint32_t pass = __ballot_sync(kFull, i < n && ci >= M && cv > exact.top);
        while (pass) {
          const int j = __ffs(pass) - 1;
          pass &= pass - 1;
          const float cvj = __shfl_sync(kFull, cv, j);
          const int cij = __shfl_sync(kFull, ci, j);
          if (cvj > exact.top) exact.insert(cvj, cij);
        }
      }
    }
    exact.h.sort(M);
    out_v = exact.h.v; out_i = exact.h.i;
    done = true;
  }
  if (!done) {   // force_exact, or a log overflowed: the literal libstdc++ control flow over the whole row
    HeapSink exact;
    exact.h = HeapRef{s_v[0], s_i[0]};
    exact.M = M; exact.lane = lane;
    scan_row(exact, hm, mk, wm, H, W, wpr, M, lane);
    __syncwarp();
    if (lane == 0) sort_heap(exact.h, M);
    __syncwarp();
    if (lane < M) { out_v = exact.h.v[lane]; out_i = exact.h.i[lane]; }
  }
  if (lane < M) {
    const size_t o = (size_t)row * M + lane;
    scores_k[o] = out_v;
    idx_k[o] = out_i;
    coords_k[o * 2 + 0] = out_i % W;
    coords_k[o * 2 + 1] = out_i / W;
    float tv[HPD_MAX_EMB];
    tag_value(tags, row, out_i, tv);
    tags_k[o * E] = tv[0];
    if (E > 1) tags_k[o * E + 1] = tv[1];
  }
}

// Second launch of the large-batch path: one CTA of kSplitWarps warps per row, rows not marked by topk_kernel
// leave at once.  The sequential algorithm admits element i iff its value exceeds the M-th largest value before it,
// so WHICH elements enter can be found in parallel and only the entering elements (~M*ln(n/M), a few hundred)
// have to go through the exact heap one by one:
//   1. the row is cut into segments that grow geometrically (the entries thin out like M/i, so every segment logs a
//      few dozen of them);
//   2. warp s takes the M-th largest word maximum of the words BEFORE its segment -- word maxima are values of
//      distinct pixels, so this is a lower bound of the heap top at the segment's start -- seeds a sorted sink with M
//      placeholders at that value and logs every element of its segment that enters the sink: a superset of what
//      enters the heap there, in index order;
//   3. warp 0 owns the libstdc++ heap (slot i in lane i): it streams its own segment -- the first pixels of the row --
//      straight through it, then replays the logs of the other segments in order, each as soon as it is complete,
//      filtering against the live top, and sorts.
constexpr int kTiedLogCap = 512;
// segment s covers [kSegFrac[s], kSegFrac[s+1]) / 1024 of the row's words (rounded up to multiples of 8 words): with
// ~M/i entries per element every segment logs a few dozen, the first one (which warp 0 both logs and replays) the fewest
__constant__ int kSegFrac[kSplitWarps + 1] = {0, 1, 4, 16, 64, 128, 256, 512, 1024};

__global__ void __launch_bounds__(kSplitWarps * 32, 1) topk_tied_rows_kernel(const float* __restrict__ agg_hm,
                                                                         const TagSource tags,
                                                                         const uint32_t* __restrict__ mask,
                                                                         const float* __restrict__ wmax, int H, int W,
                                                                         int wpr, int E, int M,
                                                                         float* __restrict__ scores_k,
                                                                         int32_t* __restrict__ idx_k,
                                                                         int32_t* __restrict__ coords_k,
                                                                         float* __restrict__ tags_k) {
  const int row = blockIdx.x;
  if (idx_k[(size_t)row * M] != -1) return;
  __shared__ float s_v[32];
  __shared__ int s_i[32];
  __shared__ float s_logv[kSplitWarps][kTiedLogCap];
  __shared__ int s_logi[kSplitWarps][kTiedLogCap];
  __shared__ int s_nlog[kSplitWarps];
  __shared__ int s_ready[kSplitWarps];      // segment s's log is complete (warp 0 replays the logs as they arrive)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x < kSplitWarps) s_ready[threadIdx.x] = 0;
  __syncthreads();
  const float* hm = agg_hm + (size_t)row * H * W;
  const uint32_t* mk = mask + (size_t)row * H * wpr;
  const float* wm = wmax + (size_t)row * H * wpr;
  const int nwords = H * wpr;
  const int noct = (nwords + 7) / 8;
  const int w_begin = min(nwords, 8 * (int)(((long long)noct * kSegFrac[warp] + 1023) / 1024));
  const int w_end = warp == kSplitWarps - 1 ? nwords : min(nwords, 8 * (int)(((long long)noct * kSegFrac[warp + 1] + 1023) / 1024));
#ifdef HPD_TOPK_PROFILE
  long long tp[8];
  __shared__ long long s_tp[kSplitWarps][4];
#endif
  TP_MARK(0);

  // lower bound of the heap top at the start of this segment: the M-th largest word maximum of the prefix
  float floor_s = -INFINITY;
  if (w_begin >= M) {
    WordMaxCandidates cand;
    cand.scan(wm, 0, w_begin, lane);
    TP_MARK(1);
    for (int r = 0; r < M; ++r) floor_s = cand.pop(lane);
  } else {
    TP_MARK(1);
  }
  if (warp != 0) {
    SortedSink seg;
    seg.M = M; seg.lane = lane;
    seg.log_v = s_logv[warp]; seg.log_i = s_logi[warp]; seg.log_cap = kTiedLogCap;
    if (floor_s > -INFINITY) seg.init_floor(floor_s);
    else seg.init_empty();
    TP_MARK(2);
    scan_range(seg, hm, mk, wm, W, wpr, w_begin, w_end, 0, lane);
    TP_MARK(3);
#ifdef HPD_TOPK_PROFILE
    if (lane == 0) { s_tp[warp][0] = tp[1] - tp[0]; s_tp[warp][1] = tp[2] - tp[1]; s_tp[warp][2] = tp[3] - tp[2]; }
#endif
    __syncwarp();
    if (lane == 0) {
      s_nlog[warp] = seg.n_log;
      __threadfence_block();
      *(volatile int*)&s_ready[warp] = 1;
    }
    return;
  }
  TP_MARK(2);

  // Warp 0 owns the heap.  Its own segment -- the first pixels of the row, where most of the entries are -- goes
  // through the exact heap directly (no log in between); then it replays segment after segment, each as soon as its
  // warp has finished logging it (the later segments are still being streamed meanwhile).
  float out_v = 0.f;
  int out_i = 0;
  bool logs_ok = true;
  WarpHeapSink exact;
  exact.M = M; exact.lane = lane;
  exact.init(first_element(hm, mk, W, wpr, M, lane));
  scan_range(exact, hm, mk, wm, W, wpr, w_begin, w_end, M, lane);
  TP_MARK(3);
  TP_MARK(4);
  for (int w = 1; w < kSplitWarps && logs_ok; ++w) {
    while (*(volatile int*)&s_ready[w] == 0) {}
    __threadfence_block();
    const int n = *(volatile int*)&s_nlog[w];
    if (n > kTiedLogCap) { logs_ok = false; break; }
    for (int i0 = 0; i0 < n; i0 += 32) {
      const int i = i0 + lane;
      const float cv = i < n ? s_logv[w][i] : -INFINITY;
      const int ci = i < n ? s_logi[w][i] : 0;
      const float top = __shfl_sync(kFull, exact.h.v, 0);
      uint32_t pass = __ballot_sync(kFull, i < n && ci >= M && cv > top);
      // (the next candidate is read -- one broadcast shared-memory load -- while the current one sifts)
      int j = pass ? __ffs(pass) - 1 : 0;
      float cvj = s_logv[w][i0 + j];
      int cij = s_logi[w][i0 + j];
      while (pass) {
        pass &= pass - 1;
        const float cur_v = cvj;
        const int cur_i = cij;
        j = pass ? __ffs(pass) - 1 : j;
        cvj = s_logv[w][i0 + j];
        cij = s_logi[w][i0 + j];
        // comp(*i, *first): the element enters iff it is greater than the heap's top right now (tested inside)
        exact.h.adjust_root<true>(M, cur_v, cur_i);
      }
    }
  }
  if (logs_ok) {
    TP_MARK(5);
    exact.h.sort(M);
    TP_MARK(6);
#ifdef HPD_TOPK_PROFILE
    if (lane == 0 && atomicAdd(&tp_printed, 1) < 80) {
      int tot = 0;
      for (int w = 1; w < kSplitWarps; ++w) tot += s_nlog[w];
      printf("tied row %d: own segment %lld, replay+wait %lld, sort %lld, total %lld cycles; %d log entries\n", row, tp[3] - tp[0],
             tp[5] - tp[4], tp[6] - tp[5], tp[6] - tp[0], tot);
    }
#endif
    out_v = exact.h.v; out_i = exact.h.i;
  } else {   // a log overflowed: the literal libstdc++ control flow over the whole row
#ifdef HPD_TOPK_PROFILE
    if (lane == 0) printf("tied row %d: LOG OVERFLOW\n", row);
#endif
    HeapSink exact;
    exact.h = HeapRef{s_v, s_i};
    exact.M = M; exact.lane = lane;
    scan_row(exact, hm, mk, wm, H, W, wpr, M, lane);
    __syncwarp();
    if (lane == 0) sort_heap(exact.h, M);
    __syncwarp();
    if (lane < M) { out_v = exact.h.v[lane]; out_i = exact.h.i[lane]; }
  }
  if (lane < M) {
    const size_t o = (size_t)row * M + lane;
    scores_k[o] = out_v;
    idx_k[o] = out_i;
    coords_k[o * 2 + 0] = out_i % W;
    coords_k[o * 2 + 1] = out_i / W;
    float tv[HPD_MAX_EMB];
    tag_value(tags, row, out_i, tv);
    tags_k[o * E] = tv[0];
    if (E > 1) tags_k[o * E + 1] = tv[1];
  }
}

}  // namespace

int launch_topk(const HpdParams* p, const HpdBuffers* buf, cudaStream_t st) {
  if (!buf->agg_hm || !buf->nms_mask || !buf->nms_wmax || !buf->scores_k || !buf->idx_k || !buf->coords_k ||
      !buf->tags_k) {
    set_error("hpd_topk: agg_hm, nms_mask, nms_wmax, scores_k, idx_k, coords_k, tags_k are required");
    return HPD_EINVAL;
  }
  TagSource tags;
  if (int rc = make_tag_source(p, buf, &tags, "hpd_topk")) return rc;
  const int rows = p->batch * p->num_kpts;
  const int wpr = (p->out_w + 31) / 32;
  // small batches: kSplitWarps warps per row cut the per-row latency; large ones fill the GPU with one warp per row
  const bool split = rows <= 512 && (long long)p->out_h * wpr >= 128 * kSplitWarps && !(p->force_generic & 2) &&
                     p->batches_in_flight < 8;
  if (split)
    topk_split_kernel<<<rows, kSplitWarps * 32, 0, st>>>(buf->agg_hm, tags, buf->nms_mask, buf->nms_wmax, p->out_h,
                                                         p->out_w, wpr, p->emb, p->max_people, p->force_generic & 1,
                                                         buf->scores_k, buf->idx_k, buf->coords_k, buf->tags_k);
  else {
    // force_generic bit 2 (testing): rows with ties stay in topk_kernel's own one-warp exact stream
    const bool defer = !(p->force_generic & 1) && !(p->force_generic & 4) && (long long)p->out_h * wpr >= 128 * kSplitWarps;
    topk_kernel<<<(rows + kTopkWarps - 1) / kTopkWarps, kTopkWarps * 32, 0, st>>>(
        buf->agg_hm, tags, buf->nms_mask, buf->nms_wmax, rows, p->out_h, p->out_w, wpr, p->emb, p->max_people,
        p->force_generic & 1, defer ? 1 : 0, buf->scores_k, buf->idx_k, buf->coords_k, buf->tags_k);
    if (defer) {
      count_launch();
      if (int rc = check_launch("topk_kernel")) return rc;
      topk_tied_rows_kernel<<<rows, kSplitWarps * 32, 0, st>>>(buf->agg_hm, tags, buf->nms_mask, buf->nms_wmax,
                                                               p->out_h, p->out_w, wpr, p->emb, p->max_people, buf->scores_k,
                                                               buf->idx_k, buf->coords_k, buf->tags_k);
    }
  }
  count_launch();
  return check_launch("topk_kernel");
}

}  // namespace hpd
