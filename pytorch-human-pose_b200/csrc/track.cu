// Person tracking across frames (include/hpdecode.h: hpd_track): each frame's persons are matched greedily to the
// tracks of earlier frames by OKS.  The NumPy statement of the definition is oracle/track_oracle.py.
//
//   track_kernel  one CTA walks the call's frames in order, reading the result records in place.  Per frame, in
//                 shared memory: the persons' joints, visibility and areas; their score ranks, counted as
//                 coco_image_kernel ranks detections; the OKS of every (person, live track) pair, one thread each;
//                 the greedy pass, one warp with one arg-max per person over the live, unclaimed tracks; then the
//                 update and compaction of the track table.
//
// Tracks sit in slots of a table of C = max_people * max_age entries (no more can be live at once: a frame adds or
// refreshes at most max_people, and a track unclaimed for max_age frames is dropped).  `live` lists the slots of the
// live tracks in id order, so that its position order is the id order the tie rule needs, and compaction moves
// slot indices, not poses.  Between calls the state holds the live tracks compacted to slots 0..n_live-1.
//
// Like hpd_coco_eval, every float64 operation is spelled out and exp() is CUDA's, within 1 ulp of NumPy's.
//
// track_kernel<true> (hpd_track_smooth) also runs a One-Euro filter per (track, joint); oracle/smooth_oracle.py states
// it.  Its state (FilterTable) is too large for shared memory next to the table, so it stays in the state buffer in
// global memory, indexed by slot, and is touched only for the frame's claimed and new tracks, one thread per (person,
// joint).  The end-of-call compaction moves tracks to slots 0..n_live-1; the filter region is double-buffered so that
// it can follow: the call reads and updates buffer `buf` by slot, then copies the live slots in live order to the
// other buffer and flips `buf`.
#include <math.h>

#include "common.cuh"

namespace hpd {
namespace {

constexpr int kTrackThreads = 256;

struct TrackHeader {
  int32_t n_live, next_id;
  uint32_t frame, buf;   // hpd_track_smooth only: frames filtered so far (mod 2^32); the filter buffer in use (bit 0)
};

// Track slots; the same layout in the state (after TrackHeader) and in shared memory.
struct TrackTable {
  double *x, *y;       // [C][K] the pose that last matched the track, COCO-section coordinates
  double* area;        // [C]
  uint32_t* vis;       // [C] bit k: joint k visible
  int32_t *id, *age;   // [C]
};

__host__ __device__ inline size_t table_bytes(int C, int K) { return (size_t)C * (16 * K + 8 + 3 * 4); }

__host__ __device__ inline TrackTable carve_table(uint8_t* base, int C, int K) {
  TrackTable t;
  t.x = reinterpret_cast<double*>(base);
  t.y = t.x + (size_t)C * K;
  t.area = t.y + (size_t)C * K;
  t.vis = reinterpret_cast<uint32_t*>(t.area + C);
  t.id = reinterpret_cast<int32_t*>(t.vis + C);
  t.age = t.id + C;
  return t;
}

// One-Euro filter state of the track slots, C x K entries per buffer: the filtered position and speed, the frame the joint
// was last filtered (so a gap of g frames gives te = g / fps) and whether it was seen since the track began.
struct FilterTable {
  double *x, *y, *dx, *dy;   // [C][K]
  uint32_t *last, *seen;     // [C][K]
};

__host__ __device__ inline size_t filter_bytes(int C, int K) { return (size_t)C * K * (4 * 8 + 2 * 4); }
__host__ __device__ inline size_t filter_offset(int C, int K) { return (sizeof(TrackHeader) + table_bytes(C, K) + 7) / 8 * 8; }

__host__ __device__ inline FilterTable carve_filter(uint8_t* base, int C, int K) {
  FilterTable t;
  const size_t n = (size_t)C * K;
  t.x = reinterpret_cast<double*>(base);
  t.y = t.x + n;
  t.dx = t.y + n;
  t.dy = t.dx + n;
  t.last = reinterpret_cast<uint32_t*>(t.dy + n);
  t.seen = t.last + n;
  return t;
}

struct TrackSmem {
  double* oks;                 // [M][C] person x live position
  double *px, *py;             // [M][K]
  double* parea;               // [M]
  TrackTable t;                // C slots
  uint32_t* pvis;              // [M]
  float* pscore;               // [M]
  int32_t *pnvis, *order, *assign, *pid, *nslot;   // [M] assign: live position, -1 new track, -2 none
  int32_t *live, *live2, *free_slot, *used;        // [C]
};

// Carves the kernel's dynamic shared memory (base == nullptr: only the size); returns its bytes.  float64 arrays first.
__host__ __device__ inline size_t carve_smem(uint8_t* base, int M, int C, int K, TrackSmem* s) {
  size_t off = 0;
  auto take = [&](size_t bytes) {
    uint8_t* q = base ? base + off : nullptr;
    off += bytes;
    return q;
  };
  s->oks = reinterpret_cast<double*>(take(8 * (size_t)M * C));
  s->px = reinterpret_cast<double*>(take(8 * (size_t)M * K));
  s->py = reinterpret_cast<double*>(take(8 * (size_t)M * K));
  s->parea = reinterpret_cast<double*>(take(8 * (size_t)M));
  uint8_t* t = take(table_bytes(C, K));
  if (base) s->t = carve_table(t, C, K);
  s->pvis = reinterpret_cast<uint32_t*>(take(4 * (size_t)M));
  s->pscore = reinterpret_cast<float*>(take(4 * (size_t)M));
  int32_t** per_person[] = {&s->pnvis, &s->order, &s->assign, &s->pid, &s->nslot};
  for (int32_t** a : per_person) *a = reinterpret_cast<int32_t*>(take(4 * (size_t)M));
  int32_t** per_slot[] = {&s->live, &s->live2, &s->free_slot, &s->used};
  for (int32_t** a : per_slot) *a = reinterpret_cast<int32_t*>(take(4 * (size_t)C));
  return off;
}

size_t track_smem_bytes(int M, int C, int K) {
  TrackSmem s;
  return carve_smem(nullptr, M, C, K, &s);
}

// OKS of person d against track t over the joints visible in both: np.sum(np.exp(-e)) / |J| with
// e = (dx**2 + dy**2) / vars / ((area_d + area_t) / 2 + np.spacing(1)) / 2
__device__ __forceinline__ double track_oks(const double* xd, const double* yd, uint32_t vd, double ad,
                                            const double* xt, const double* yt, uint32_t vt, double at,
                                            const double* vars, int K) {
  const uint32_t J = vd & vt;
  const int n = __popc(J);
  if (n == 0) return 0.0;
  const double den = __dadd_rn(__ddiv_rn(__dadd_rn(ad, at), 2.0), 0x1p-52);
  NpSumF64 acc(n);
  for (int k = 0; k < K; ++k) {
    if (!((J >> k) & 1u)) continue;
    const double dx = __dsub_rn(xd[k], xt[k]), dy = __dsub_rn(yd[k], yt[k]);
    double e = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
    e = __ddiv_rn(__ddiv_rn(__ddiv_rn(e, vars[k]), den), 2.0);
    acc.add(exp(-e));
  }
  return __ddiv_rn(acc.sum(), (double)n);
}

constexpr double kTwoPi = 2.0 * 3.141592653589793;   // Python's 2 * math.pi

// One filter step of one coordinate (include/hpdecode.h: hpd_track_smooth), each operation rounded once, no FMA:
// updates the filtered speed dxh and position xh from the raw x and returns the new position.
__device__ __forceinline__ double one_euro(double x, double& xh, double& dxh, double te, double ad,
                                           const HpdSmoothParams& sp) {
  const double dx = __ddiv_rn(__dsub_rn(x, xh), te);
  dxh = __dadd_rn(__dmul_rn(ad, dx), __dmul_rn(__dsub_rn(1.0, ad), dxh));
  const double c = __dadd_rn(sp.min_cutoff, __dmul_rn(sp.beta, fabs(dxh)));
  const double r = __dmul_rn(__dmul_rn(kTwoPi, c), te);
  const double a = __ddiv_rn(r, __dadd_rn(r, 1.0));
  xh = __dadd_rn(__dmul_rn(a, x), __dmul_rn(__dsub_rn(1.0, a), xh));
  return xh;
}

// SMOOTH's parameters follow the others, so that track_kernel<false> compiles to the instructions of the untemplated
// kernel it replaced.
template <bool SMOOTH>
__global__ void __launch_bounds__(kTrackThreads) track_kernel(HpdTrackParams p, const uint8_t* __restrict__ records,
                                                              int n_frames, HpdRecordLayout L, uint8_t* state,
                                                              int32_t* __restrict__ ids, HpdSmoothParams sp,
                                                              double* __restrict__ coords) {
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ double s_vars[HPD_MAX_KPTS];
  __shared__ int s_n_live, s_next_id;
  const int K = p.num_kpts, M = p.max_people, C = M * p.max_age, D = 3 + p.emb;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  TrackSmem s;
  carve_smem(smem, M, C, K, &s);
  TrackHeader* hdr = reinterpret_cast<TrackHeader*>(state);
  const TrackTable g = carve_table(state + sizeof(TrackHeader), C, K);
  uint32_t frame0 = 0, buf = 0;
  FilterTable fz;
  if constexpr (SMOOTH) {
    frame0 = hdr->frame;
    buf = hdr->buf & 1u;
    fz = carve_filter(state + filter_offset(C, K) + buf * filter_bytes(C, K), C, K);
  }

  // the state's live tracks are compacted: live position j is slot j
  const int n_live0 = min(max(hdr->n_live, 0), C);
  for (int i = tid; i < n_live0 * K; i += kTrackThreads) {
    s.t.x[i] = g.x[i];
    s.t.y[i] = g.y[i];
  }
  for (int j = tid; j < n_live0; j += kTrackThreads) {
    s.t.area[j] = g.area[j];
    s.t.vis[j] = g.vis[j];
    s.t.id[j] = g.id[j];
    s.t.age[j] = g.age[j];
    s.live[j] = j;
  }
  for (int k = tid; k < K; k += kTrackThreads) s_vars[k] = p.kpt_vars[k];
  if (tid == 0) {
    s_n_live = n_live0;
    s_next_id = hdr->next_id;
  }
  int32_t *live = s.live, *live2 = s.live2;

  for (int f = 0; f < n_frames; ++f) {
    const uint8_t* r = records + (size_t)f * L.row_bytes;
    int n = min(max(*reinterpret_cast<const int32_t*>(r + L.off_n_person), 0), M);
    if (*reinterpret_cast<const int32_t*>(r + L.off_flags) & 1) n = 0;   // the empty-scene fallback's pseudo-person
    const double* coco = reinterpret_cast<const double*>(r + L.off_coco);
    const float* poses = reinterpret_cast<const float*>(r + L.off_poses);
    const float* scores = reinterpret_cast<const float*>(r + L.off_person_scores);
    int32_t* out = ids + (size_t)f * M;
    __syncthreads();   // the previous frame (or the load) is complete
    const int n_live = s_n_live;

    for (int i = tid; i < n * K; i += kTrackThreads) {
      const int q = i / K, k = i % K;
      s.px[i] = coco[(size_t)q * L.coco_stride + 3 * k];
      s.py[i] = coco[(size_t)q * L.coco_stride + 3 * k + 1];
    }
    for (int q = tid; q < M; q += kTrackThreads) {
      if (q < n) s.pscore[q] = scores[q];
      else out[q] = -1;
      s.order[q] = -1;     // stays -1 only for ranks a NaN score leaves unfilled
      s.assign[q] = -2;
      s.pid[q] = -1;
    }
    __syncthreads();

    // visibility, area of the visible joints' box, and the score rank (descending, ties: lower index)
    for (int q = tid; q < n; q += kTrackThreads) {
      uint32_t vis = 0;
      int nv = 0;
      double x0 = 0, x1 = 0, y0 = 0, y1 = 0;
      for (int k = 0; k < K; ++k) {
        if (!(poses[((size_t)q * K + k) * D + 2] > 0.f)) continue;
        const double x = s.px[q * K + k], y = s.py[q * K + k];
        if (nv == 0) {
          x0 = x1 = x;
          y0 = y1 = y;
        } else {
          x0 = x < x0 ? x : x0;
          x1 = x > x1 ? x : x1;
          y0 = y < y0 ? y : y0;
          y1 = y > y1 ? y : y1;
        }
        vis |= 1u << k;
        ++nv;
      }
      s.pvis[q] = vis;
      s.pnvis[q] = nv;
      s.parea[q] = nv >= 2 ? __dmul_rn(__dsub_rn(x1, x0), __dsub_rn(y1, y0)) : 0.0;
      const float sc = s.pscore[q];
      int rank = 0;
      for (int o = 0; o < n; ++o) {
        const float so = s.pscore[o];
        rank += (so > sc) || (so == sc && o < q);
      }
      if (rank < n) s.order[rank] = q;
    }
    __syncthreads();

    for (int i = tid; i < n * n_live; i += kTrackThreads) {
      const int q = i / n_live, j = i % n_live, t = live[j];
      s.oks[(size_t)q * C + j] = track_oks(s.px + q * K, s.py + q * K, s.pvis[q], s.parea[q], s.t.x + (size_t)t * K,
                                           s.t.y + (size_t)t * K, s.t.vis[t], s.t.area[t], s_vars, K);
    }
    __syncthreads();

    // greedy pass: lane l holds live positions l, l + 32, ... (C <= 256: 8 bits of `claimed`)
    if (warp == 0) {
      uint32_t claimed = 0;
      int next_id = s_next_id;
      for (int rk = 0; rk < n; ++rk) {
        const int q = s.order[rk];
        if (q < 0) continue;
        double best = 0.0;
        int bj = -1;
        for (int i = 0, j = lane; j < n_live; ++i, j += 32) {
          if ((claimed >> i) & 1u) continue;
          const double v = s.oks[(size_t)q * C + j];
          if (bj < 0 || v > best) {   // ascending j: an equal OKS keeps the smaller position, i.e. the smaller id
            best = v;
            bj = j;
          }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
          const double ov = __shfl_xor_sync(kFull, best, off);
          const int oj = __shfl_xor_sync(kFull, bj, off);
          if (oj >= 0 && (bj < 0 || ov > best || (ov == best && oj < bj))) {
            best = ov;
            bj = oj;
          }
        }
        int a, id;
        if (bj >= 0 && best > p.oks_thr) {
          a = bj;
          id = s.t.id[live[bj]];
          if ((bj & 31) == lane) claimed |= 1u << (bj >> 5);
        } else if (s.pnvis[q] >= p.min_keypoints) {
          a = -1;
          id = next_id++;
        } else {
          a = -2;
          id = -1;
        }
        if (lane == 0) {
          s.assign[q] = a;
          s.pid[q] = id;
        }
      }
      // unclaimed tracks age; `used` marks the slots of the survivors below
      for (int i = 0, j = lane; j < n_live; ++i, j += 32)
        if (!((claimed >> i) & 1u)) s.t.age[live[j]] += 1;
      if (lane == 0) s_next_id = next_id;
    }
    for (int sl = tid; sl < C; sl += kTrackThreads) s.used[sl] = 0;
    __syncthreads();

    // ids out; claimed tracks take their person's pose
    for (int q = tid; q < n; q += kTrackThreads) {
      out[q] = s.pid[q];
      const int a = s.assign[q];
      if (a >= 0) {
        const int t = live[a];
        s.t.vis[t] = s.pvis[q];
        s.t.area[t] = s.parea[q];
        s.t.age[t] = 0;
      }
    }
    for (int i = tid; i < n * K; i += kTrackThreads) {
      const int a = s.assign[i / K];
      if (a >= 0) {
        const size_t t = live[a];
        s.t.x[t * K + i % K] = s.px[i];
        s.t.y[t * K + i % K] = s.py[i];
      }
    }
    __syncthreads();

    // compaction (warp 0): survivors keep their order, new tracks follow in id order (= rank order) in free slots
    if (warp == 0) {
      const uint32_t lt = (1u << lane) - 1u;
      int m = 0;
      for (int base = 0; base < n_live; base += 32) {
        const int j = base + lane;
        const bool keep = j < n_live && s.t.age[live[j]] < p.max_age;
        const uint32_t b = __ballot_sync(kFull, keep);
        if (keep) {
          live2[m + __popc(b & lt)] = live[j];
          s.used[live[j]] = 1;
        }
        m += __popc(b);
      }
      __syncwarp();
      int nf = 0;
      for (int base = 0; base < C; base += 32) {
        const int sl = base + lane;
        const bool fr = sl < C && !s.used[sl];
        const uint32_t b = __ballot_sync(kFull, fr);
        if (fr) s.free_slot[nf + __popc(b & lt)] = sl;
        nf += __popc(b);
      }
      __syncwarp();
      const int q = lane < n ? s.order[lane] : -1;     // n <= 32
      const bool fresh = q >= 0 && s.assign[q] == -1;
      const uint32_t b = __ballot_sync(kFull, fresh);
      if (fresh) {
        const int idx = __popc(b & lt), sl = s.free_slot[idx];
        live2[m + idx] = sl;
        s.nslot[q] = sl;
        s.t.id[sl] = s.pid[q];
        s.t.age[sl] = 0;
        s.t.vis[sl] = s.pvis[q];
        s.t.area[sl] = s.parea[q];
      }
      if (lane == 0) s_n_live = m + __popc(b);
    }
    __syncthreads();
    for (int i = tid; i < n * K; i += kTrackThreads) {
      const int q = i / K;
      if (s.assign[q] == -1) {
        const size_t sl = s.nslot[q];
        s.t.x[sl * K + i % K] = s.px[i];
        s.t.y[sl * K + i % K] = s.py[i];
      }
    }
    if constexpr (SMOOTH) {
      // every row of the frame: tracked persons' visible joints filtered, other persons raw, rows past n_person 0
      const int n_rec = min(max(*reinterpret_cast<const int32_t*>(r + L.off_n_person), 0), M);
      const uint32_t fr = frame0 + (uint32_t)f;
      double* co = coords + (size_t)f * M * K * 2;
      for (int i = tid; i < M * K; i += kTrackThreads) {
        const int q = i / K, k = i % K;
        double x = 0.0, y = 0.0;
        if (q < n_rec) {
          x = coco[(size_t)q * L.coco_stride + 3 * k];
          y = coco[(size_t)q * L.coco_stride + 3 * k + 1];
        }
        const int a = q < n ? s.assign[q] : -2;
        if (a != -2) {   // the person has a track: claimed (a >= 0, the pose update above) or new (slot nslot)
          const size_t e = (size_t)(a >= 0 ? live[a] : s.nslot[q]) * K + k;
          const bool vis = (s.pvis[q] >> k) & 1u;
          if (vis) {
            double xh = x, yh = y, dxh = 0.0, dyh = 0.0;
            if (a >= 0 && fz.seen[e]) {
              xh = fz.x[e];
              yh = fz.y[e];
              dxh = fz.dx[e];
              dyh = fz.dy[e];
              const double te = __ddiv_rn((double)(fr - fz.last[e]), sp.fps);
              const double rd = __dmul_rn(__dmul_rn(kTwoPi, sp.d_cutoff), te);
              const double ad = __ddiv_rn(rd, __dadd_rn(rd, 1.0));
              x = one_euro(x, xh, dxh, te, ad, sp);
              y = one_euro(y, yh, dyh, te, ad, sp);
            }
            fz.x[e] = xh;
            fz.y[e] = yh;
            fz.dx[e] = dxh;
            fz.dy[e] = dyh;
            fz.last[e] = fr;
          }
          if (vis || a == -1) fz.seen[e] = vis;   // a new track in a reused slot starts unseeded
        }
        co[2 * i] = x;
        co[2 * i + 1] = y;
      }
    }
    int32_t* tmp = live;
    live = live2;
    live2 = tmp;
  }
  __syncthreads();

  const int n_live = s_n_live;
  for (int i = tid; i < n_live * K; i += kTrackThreads) {
    const size_t t = live[i / K];
    g.x[i] = s.t.x[t * K + i % K];
    g.y[i] = s.t.y[t * K + i % K];
  }
  for (int j = tid; j < n_live; j += kTrackThreads) {
    const int t = live[j];
    g.area[j] = s.t.area[t];
    g.vis[j] = s.t.vis[t];
    g.id[j] = s.t.id[t];
    g.age[j] = s.t.age[t];
  }
  if (tid == 0) {
    hdr->n_live = n_live;
    hdr->next_id = s_next_id;
  }
  if constexpr (SMOOTH) {   // the filter follows the compaction into the other buffer
    const FilterTable to = carve_filter(state + filter_offset(C, K) + (buf ^ 1u) * filter_bytes(C, K), C, K);
    for (int i = tid; i < n_live * K; i += kTrackThreads) {
      const size_t e = (size_t)live[i / K] * K + i % K;
      to.x[i] = fz.x[e];
      to.y[i] = fz.y[e];
      to.dx[i] = fz.dx[e];
      to.dy[i] = fz.dy[e];
      to.last[i] = fz.last[e];
      to.seen[i] = fz.seen[e];
    }
    if (tid == 0) {
      hdr->frame = frame0 + (uint32_t)n_frames;
      hdr->buf = buf ^ 1u;
    }
  }
}

size_t state_bytes_of(const HpdTrackParams* p) {
  return sizeof(TrackHeader) + table_bytes(p->max_people * p->max_age, p->num_kpts);
}

size_t smooth_state_bytes_of(const HpdTrackParams* p) {
  const int C = p->max_people * p->max_age, K = p->num_kpts;
  return filter_offset(C, K) + 2 * filter_bytes(C, K);
}

int check_state(const void* state, size_t state_bytes, size_t need, const char* who) {
  if (!state) { set_error("%s: state is NULL", who); return HPD_EINVAL; }
  if ((uintptr_t)state % 8) { set_error("%s: state must be 8-byte aligned", who); return HPD_EINVAL; }
  if (state_bytes < need) {
    set_error("%s: state too small (%zu < %zu bytes)", who, state_bytes, need);
    return HPD_EINVAL;
  }
  return HPD_OK;
}

}  // namespace

int validate_track_params(const HpdTrackParams* p, const char* who) {
  if (!p) { set_error("%s: params pointer is NULL", who); return HPD_EINVAL; }
  if (p->num_kpts < 1 || p->num_kpts > HPD_MAX_KPTS) {
    set_error("%s: num_kpts must be in [1,%d] (got %d)", who, HPD_MAX_KPTS, p->num_kpts);
    return HPD_EINVAL;
  }
  if (p->max_people < 1 || p->max_people > HPD_MAX_PEOPLE) {
    set_error("%s: max_people must be in [1,%d] (got %d)", who, HPD_MAX_PEOPLE, p->max_people);
    return HPD_EINVAL;
  }
  if (p->emb < 1 || p->emb > HPD_MAX_EMB) { set_error("%s: emb must be 1 or 2 (got %d)", who, p->emb); return HPD_EINVAL; }
  if (p->max_age < 1 || p->max_age > HPD_TRACK_MAX_AGE) {
    set_error("%s: max_age must be in [1,%d] (got %d)", who, HPD_TRACK_MAX_AGE, p->max_age);
    return HPD_EINVAL;
  }
  if (p->min_keypoints < 0 || p->min_keypoints > p->num_kpts) {
    set_error("%s: min_keypoints must be in [0,num_kpts=%d] (got %d)", who, p->num_kpts, p->min_keypoints);
    return HPD_EINVAL;
  }
  if (!isfinite(p->oks_thr)) { set_error("%s: oks_thr must be finite", who); return HPD_EINVAL; }
  for (int k = 0; k < p->num_kpts; ++k) {
    if (!(isfinite(p->kpt_vars[k]) && p->kpt_vars[k] > 0.0)) {
      set_error("%s: kpt_vars[%d] must be finite and > 0", who, k);
      return HPD_EINVAL;
    }
  }
  return HPD_OK;
}

int validate_smooth_params(const HpdSmoothParams* sp, const char* who) {
  if (!sp) { set_error("%s: smooth params pointer is NULL", who); return HPD_EINVAL; }
  const struct { const char* name; double v, lo, hi; bool lo_open; } f[] = {
      {"min_cutoff", sp->min_cutoff, 0.0, 1e6, true}, {"beta", sp->beta, 0.0, 1e6, false},
      {"d_cutoff", sp->d_cutoff, 0.0, 1e6, true}, {"fps", sp->fps, 1e-3, 1e6, false}};
  for (const auto& x : f) {
    if (!(isfinite(x.v) && (x.lo_open ? x.v > x.lo : x.v >= x.lo) && x.v <= x.hi)) {
      set_error("%s: %s must be finite and in %c%g, %g] (got %g)", who, x.name, x.lo_open ? '(' : '[', x.lo, x.hi, x.v);
      return HPD_EINVAL;
    }
  }
  return HPD_OK;
}

size_t track_state_bytes(const HpdTrackParams* p) { return state_bytes_of(p); }

size_t track_smooth_state_bytes(const HpdTrackParams* p) { return smooth_state_bytes_of(p); }

int launch_track_reset(const HpdTrackParams* p, void* state, size_t state_bytes, int clear_ids, cudaStream_t st) {
  int rc = check_state(state, state_bytes, state_bytes_of(p), "hpd_track_reset");
  if (rc) return rc;
  // n_live = 0 drops the tracks, and with them their filters; clear_ids zeroes the whole header: next_id restarts at
  // 0, and a smoothing state's frame counter and buffer bit start from known values
  const cudaError_t e = cudaMemsetAsync(state, 0, clear_ids ? sizeof(TrackHeader) : sizeof(int32_t), st);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("hpd_track_reset: %s", cudaGetErrorString(e));
    return HPD_ECUDA;
  }
  return HPD_OK;
}

int launch_track(const HpdTrackParams* p, const uint8_t* records, int n_frames, void* state, size_t state_bytes,
                 int32_t* track_ids, cudaStream_t st) {
  if (!records) { set_error("hpd_track: records is NULL"); return HPD_EINVAL; }
  if ((uintptr_t)records % 8) { set_error("hpd_track: records must be 8-byte aligned"); return HPD_EINVAL; }
  if (n_frames < 1) { set_error("hpd_track: n_frames must be >= 1 (got %d)", n_frames); return HPD_EINVAL; }
  if (!track_ids) { set_error("hpd_track: track_ids is NULL"); return HPD_EINVAL; }
  if ((uintptr_t)track_ids % 4) { set_error("hpd_track: track_ids must be 4-byte aligned"); return HPD_EINVAL; }
  int rc = check_state(state, state_bytes, state_bytes_of(p), "hpd_track");
  if (rc) return rc;
  const int C = p->max_people * p->max_age;
  const size_t smem = track_smem_bytes(p->max_people, C, p->num_kpts);
  if ((rc = ensure_dynamic_smem((const void*)track_kernel<false>, smem, "hpd_track"))) return rc;
  track_kernel<false><<<1, kTrackThreads, smem, st>>>(*p, records, n_frames,
                                                      record_layout(p->num_kpts, p->max_people, p->emb),
                                                      (uint8_t*)state, track_ids, HpdSmoothParams{}, nullptr);
  count_launch();
  return check_launch("track_kernel");
}

int launch_track_smooth(const HpdTrackParams* p, const HpdSmoothParams* sp, const uint8_t* records, int n_frames,
                        void* state, size_t state_bytes, int32_t* track_ids, double* coords, cudaStream_t st) {
  int rc = validate_smooth_params(sp, "hpd_track_smooth");
  if (rc) return rc;
  if (!records) { set_error("hpd_track_smooth: records is NULL"); return HPD_EINVAL; }
  if ((uintptr_t)records % 8) { set_error("hpd_track_smooth: records must be 8-byte aligned"); return HPD_EINVAL; }
  if (n_frames < 1) { set_error("hpd_track_smooth: n_frames must be >= 1 (got %d)", n_frames); return HPD_EINVAL; }
  if (!track_ids) { set_error("hpd_track_smooth: track_ids is NULL"); return HPD_EINVAL; }
  if ((uintptr_t)track_ids % 4) { set_error("hpd_track_smooth: track_ids must be 4-byte aligned"); return HPD_EINVAL; }
  if (!coords) { set_error("hpd_track_smooth: coords is NULL"); return HPD_EINVAL; }
  if ((uintptr_t)coords % 8) { set_error("hpd_track_smooth: coords must be 8-byte aligned"); return HPD_EINVAL; }
  if ((rc = check_state(state, state_bytes, smooth_state_bytes_of(p), "hpd_track_smooth"))) return rc;
  const int C = p->max_people * p->max_age;
  const size_t smem = track_smem_bytes(p->max_people, C, p->num_kpts);
  if ((rc = ensure_dynamic_smem((const void*)track_kernel<true>, smem, "hpd_track_smooth"))) return rc;
  track_kernel<true><<<1, kTrackThreads, smem, st>>>(*p, records, n_frames,
                                                     record_layout(p->num_kpts, p->max_people, p->emb),
                                                     (uint8_t*)state, track_ids, *sp, coords);
  count_launch();
  return check_launch("track_kernel<true>");
}

}  // namespace hpd
