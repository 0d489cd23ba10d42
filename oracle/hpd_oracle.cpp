// TEST INFRASTRUCTURE ONLY -- CPU oracle for the HigherHRNet bottom-up decode path.
//
// A plain C++ restatement (host only, no CUDA, no torch) of what the reference
// computes for this path.  Only tests/, __graft_entry__.smoke() and bench.py's
// cpu_baseline / --impl reference legs may load it; the product (libhpdecode.so
// and the hpdecode python package) never does.
//
// PARITY STATUS: pinned against the reference's own python code executed in the
// build container (oracle/gen_golden.py imports the unmodified
// /root/reference/src/keypoints/grouping.py and replays results.py/model.py's
// torch calls; tests/golden/*.npz hold the recorded outputs) for everything
// except the Hungarian solver, whose upstream package (munkres 1.1.4, un-vendored,
// not installable offline) is restated from its published algorithm: that one
// piece is PARITY UNPINNED (see oracle/refshim/munkres.py and DESIGN.md).
//
// Reference lines followed (all paths relative to /root/reference):
//   flip averaging            src/keypoints/model.py:85-96, transforms.py:11
//   bilinear resize           src/keypoints/results.py:46-67  (torch F.interpolate, align_corners=False)
//   stage mean / tag stack    src/keypoints/results.py:225-230
//   nms                       src/keypoints/grouping.py:74,80-83
//   top_k                     src/keypoints/grouping.py:147-170 (torch CPU topk == std::partial_sort)
//   match_by_tag              src/keypoints/grouping.py:85-145
//   py_max_match / munkres    src/keypoints/grouping.py:55-59 (munkres 1.1.4 Munkres.compute)
//   adjust                    src/keypoints/grouping.py:172-191
//   refine                    src/keypoints/grouping.py:193-250
//   parse                     src/keypoints/grouping.py:252-283
//
// Build: oracle/Makefile (g++ -O2 -ffp-contract=off -mfma).  Every fused
// multiply-add below is an explicit fmaf(); nothing else may be contracted.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <utility>
#include <vector>

#define HPO_API extern "C" __attribute__((visibility("default")))

namespace {

constexpr int kMaxPeople = 32;   // the warp-wide device solver handles n <= 32
constexpr int kMaxKpts = 32;
constexpr int kMaxEmb = 2;

// ---------------------------------------------------------------------------
// bilinear resize, torch CPU semantics (results.py:51,59,65)
// ---------------------------------------------------------------------------
struct AxisTap { int i0, i1; float w0, w1; };

inline AxisTap axis_tap(float scale, int o, int in_size, int out_size) {
    AxisTap t;
    if (in_size == out_size) { t.i0 = t.i1 = o; t.w0 = 1.f; t.w1 = 0.f; return t; }
    float src = fmaf(scale, (float)o + 0.5f, -0.5f);
    if (src < 0.f) src = 0.f;
    int i0 = (int)src;                       // src >= 0 -> truncation == floor
    if (i0 > in_size - 1) i0 = in_size - 1;
    float l1 = src - (float)i0;
    l1 = std::min(std::max(l1, 0.f), 1.f);
    t.i0 = i0;
    t.i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
    t.w1 = l1;
    t.w0 = 1.f - l1;
    return t;
}

void resize_plane(const float* in, int ih, int iw, float* out, int oh, int ow) {
    const float sy = (float)ih / (float)oh, sx = (float)iw / (float)ow;
    std::vector<AxisTap> tx(ow);
    for (int x = 0; x < ow; ++x) tx[x] = axis_tap(sx, x, iw, ow);
    for (int y = 0; y < oh; ++y) {
        const AxisTap ty = axis_tap(sy, y, ih, oh);
        const float* r0 = in + (size_t)ty.i0 * iw;
        const float* r1 = in + (size_t)ty.i1 * iw;
        float* o = out + (size_t)y * ow;
        for (int x = 0; x < ow; ++x) {
            const AxisTap& t = tx[x];
            const float top = fmaf(t.w0, r0[t.i0], t.w1 * r0[t.i1]);
            const float bot = fmaf(t.w0, r1[t.i0], t.w1 * r1[t.i1]);
            o[x] = fmaf(ty.w0, top, ty.w1 * bot);
        }
    }
}

const int kFlipDefault[17] = {0, 2, 1, 4, 3, 6, 5, 8, 7, 10, 9, 12, 11, 14, 13, 16, 15};

// (a + flipW(b)) * 0.5 for one plane (model.py:90)
void flip_average_plane(const float* a, const float* b, int h, int w, float* out) {
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x)
            out[(size_t)y * w + x] = (a[(size_t)y * w + x] + b[(size_t)y * w + (w - 1 - x)]) * 0.5f;
}

// ---------------------------------------------------------------------------
// munkres 1.1.4 Munkres.compute, restated (see oracle/refshim/munkres.py)
// rows <= cols == n.  C is n x n row-major with the pad rows already zero.
// ---------------------------------------------------------------------------
struct Munkres {
    int n;
    double* C;
    bool rowc[kMaxPeople], colc[kMaxPeople];
    int8_t mark[kMaxPeople][kMaxPeople];
    int z0r, z0c;

    double& at(int i, int j) { return C[(size_t)i * n + j]; }

    void clear_covers() { for (int i = 0; i < n; ++i) rowc[i] = colc[i] = false; }

    // the zero-selection policy: rows cyclic from i0, in-row columns cyclic from
    // j0, LAST uncovered zero of the first row that has one.
    void find_a_zero(int i0, int j0, int& row, int& col) {
        row = col = -1;
        int i = i0;
        bool done = false;
        while (!done) {
            int j = j0;
            while (true) {
                if (at(i, j) == 0.0 && !rowc[i] && !colc[j]) { row = i; col = j; done = true; }
                j = (j + 1) % n;
                if (j == j0) break;
            }
            i = (i + 1) % n;
            if (i == i0) done = true;
        }
    }
    int find_in_row(int r, int m) { for (int j = 0; j < n; ++j) if (mark[r][j] == m) return j; return -1; }
    int find_in_col(int c, int m) { for (int i = 0; i < n; ++i) if (mark[i][c] == m) return i; return -1; }

    // Returns false when the step-6 cap stopped it (see hpo_match_by_tag's cost guard).
    bool run() {
        const int cap = n * (n + 1);
        int n6 = 0;
        std::memset(mark, 0, sizeof(mark));
        clear_covers();
        // step 1
        for (int i = 0; i < n; ++i) {
            double m = at(i, 0);
            for (int j = 1; j < n; ++j) if (at(i, j) < m) m = at(i, j);
            for (int j = 0; j < n; ++j) at(i, j) -= m;
        }
        // step 2
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j)
                if (at(i, j) == 0.0 && !colc[j] && !rowc[i]) { mark[i][j] = 1; colc[j] = rowc[i] = true; break; }
        clear_covers();
        int step = 3;
        while (true) {
            if (step == 3) {
                int count = 0;
                for (int i = 0; i < n; ++i)
                    for (int j = 0; j < n; ++j)
                        if (mark[i][j] == 1 && !colc[j]) { colc[j] = true; ++count; }
                if (count >= n) return true;
                step = 4;
            } else if (step == 4) {
                int row = 0, col = 0;
                while (true) {
                    find_a_zero(row, col, row, col);
                    if (row < 0) { step = 6; break; }
                    mark[row][col] = 2;
                    const int sc = find_in_row(row, 1);
                    if (sc >= 0) { col = sc; rowc[row] = true; colc[col] = false; }
                    else { z0r = row; z0c = col; step = 5; break; }
                }
            } else if (step == 5) {
                int pr[2 * kMaxPeople + 2], pc[2 * kMaxPeople + 2];
                int count = 0;
                pr[0] = z0r; pc[0] = z0c;
                while (true) {
                    const int r = find_in_col(pc[count], 1);
                    if (r < 0) break;
                    ++count; pr[count] = r; pc[count] = pc[count - 1];
                    const int c = find_in_row(pr[count], 2);
                    ++count; pr[count] = pr[count - 1]; pc[count] = c;
                }
                for (int k = 0; k <= count; ++k) mark[pr[k]][pc[k]] = (mark[pr[k]][pc[k]] == 1) ? 0 : 1;
                clear_covers();
                for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) if (mark[i][j] == 2) mark[i][j] = 0;
                step = 3;
            } else {  // step 6
                if (++n6 > cap) return false;
                double m = 9.223372036854775807e18;  // sys.maxsize
                for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j)
                    if (!rowc[i] && !colc[j] && m > at(i, j)) m = at(i, j);
                for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) {
                    if (rowc[i]) at(i, j) += m;
                    if (!colc[j]) at(i, j) -= m;
                }
                step = 4;
            }
        }
    }
};

// numpy float32 np.mean(list_of_vectors, axis=0) (grouping.py:114,213)
// E == 1 -> contiguous reduction -> pairwise-8 summation; E == 2 -> sequential.
inline float np_sum_pairwise8(const float* a, int n, int stride) {
    if (n < 8) {
        float r = -0.0f;
        for (int i = 0; i < n; ++i) r += a[i * stride];
        return r;
    }
    float r[8];
    for (int j = 0; j < 8; ++j) r[j] = a[j * stride];
    int i = 8;
    for (; i < n - (n % 8); i += 8)
        for (int j = 0; j < 8; ++j) r[j] += a[(i + j) * stride];
    float res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res += a[i * stride];
    return res;
}
inline void np_mean_vectors(const float* v /*[n][E]*/, int n, int E, float* out) {
    if (E == 1) {
        out[0] = (0.0f + np_sum_pairwise8(v, n, 1)) / (float)n;
    } else {
        for (int e = 0; e < E; ++e) {
            float s = 0.0f;
            for (int i = 0; i < n; ++i) s += v[i * E + e];
            out[e] = s / (float)n;
        }
    }
}

}  // namespace

// ===========================================================================
// exported C entry points (ctypes)
// ===========================================================================

HPO_API int hpo_abi_version() { return 1; }

HPO_API void hpo_resize_bilinear(const float* in, int planes, int ih, int iw, float* out, int oh, int ow) {
    for (int p = 0; p < planes; ++p)
        resize_plane(in + (size_t)p * ih * iw, ih, iw, out + (size_t)p * oh * ow, oh, ow);
}

// One image, one scale: network outputs -> stage mean resized to (H, W).
//   hm_lo [K,lh,lw], hm_hi [K,hh,hw]; *_f = outputs of the flipped run or NULL.
// out [K,H,W].
HPO_API void hpo_aggregate_heatmaps_scale(const float* hm_lo, const float* hm_hi,
                                          const float* hm_lo_f, const float* hm_hi_f,
                                          const int* flip_index, int K, int lh, int lw, int hh, int hw,
                                          int H, int W, float* out) {
    std::vector<float> lo((size_t)lh * lw), hi((size_t)hh * hw), up((size_t)hh * hw);
    for (int k = 0; k < K; ++k) {
        const int kf = flip_index ? flip_index[k] : (k < 17 ? kFlipDefault[k] : k);
        const float* plo = hm_lo + (size_t)k * lh * lw;
        const float* phi = hm_hi + (size_t)k * hh * hw;
        if (hm_lo_f) {
            flip_average_plane(plo, hm_lo_f + (size_t)kf * lh * lw, lh, lw, lo.data());
            flip_average_plane(phi, hm_hi_f + (size_t)kf * hh * hw, hh, hw, hi.data());
            plo = lo.data(); phi = hi.data();
        }
        resize_plane(plo, lh, lw, up.data(), hh, hw);                       // results.py:225
        for (size_t i = 0; i < (size_t)hh * hw; ++i) up[i] = (up[i] + phi[i]) * 0.5f;   // results.py:226
        resize_plane(up.data(), hh, hw, out + (size_t)k * H * W, H, W);     // results.py:227
    }
}

// mean over n_s per-scale maps: torch.stack(scales).mean(0) == sequential sum / n_s
HPO_API void hpo_scale_mean(const float* const* maps, int n_s, size_t count, float* out) {
    if (n_s == 1) { std::memcpy(out, maps[0], count * sizeof(float)); return; }
    for (size_t i = 0; i < count; ++i) {
        float s = maps[0][i];
        for (int k = 1; k < n_s; ++k) s += maps[k][i];
        out[i] = s / (float)n_s;
    }
}

// tags: E maps resized x? and stacked E-innermost (results.py:229-230, model.py:91-94)
//   tag [K,th,tw]; tag_f = flipped run (-> E = 2) or NULL (E = 1).  out [K,H,W,E]
HPO_API void hpo_aggregate_tags(const float* tag, const float* tag_f, const int* flip_index, int K,
                                int th, int tw, int H, int W, float* out) {
    const int E = tag_f ? 2 : 1;
    std::vector<float> src((size_t)th * tw), dst((size_t)H * W);
    for (int k = 0; k < K; ++k) {
        for (int e = 0; e < E; ++e) {
            const float* p;
            if (e == 0) p = tag + (size_t)k * th * tw;
            else {
                const int kf = flip_index ? flip_index[k] : (k < 17 ? kFlipDefault[k] : k);
                const float* q = tag_f + (size_t)kf * th * tw;
                for (int y = 0; y < th; ++y) for (int x = 0; x < tw; ++x)
                    src[(size_t)y * tw + x] = q[(size_t)y * tw + (tw - 1 - x)];
                p = src.data();
            }
            resize_plane(p, th, tw, dst.data(), H, W);
            float* o = out + (size_t)k * H * W * E + e;
            for (size_t i = 0; i < (size_t)H * W; ++i) o[i * E] = dst[i];
        }
    }
}

// grouping.py:80-83.  5x5 max with -inf padding; out = x*1 or x*0 (keeps x's sign on zeros)
HPO_API void hpo_nms(const float* hm, int planes, int H, int W, float* out, uint8_t* keep_out) {
    const float ninf = -std::numeric_limits<float>::infinity();
    std::vector<float> rowmax((size_t)H * W);
    for (int p = 0; p < planes; ++p) {
        const float* a = hm + (size_t)p * H * W;
        for (int y = 0; y < H; ++y) for (int x = 0; x < W; ++x) {
            float m = ninf;
            for (int dx = -2; dx <= 2; ++dx) { const int xx = x + dx; if (xx >= 0 && xx < W) m = std::max(m, a[(size_t)y * W + xx]); }
            rowmax[(size_t)y * W + x] = m;
        }
        for (int y = 0; y < H; ++y) for (int x = 0; x < W; ++x) {
            float m = ninf;
            for (int dy = -2; dy <= 2; ++dy) { const int yy = y + dy; if (yy >= 0 && yy < H) m = std::max(m, rowmax[(size_t)yy * W + x]); }
            const float v = a[(size_t)y * W + x];
            const bool keep = (m == v);
            if (out) out[(size_t)p * H * W + (size_t)y * W + x] = v * (keep ? 1.0f : 0.0f);
            if (keep_out) keep_out[(size_t)p * H * W + (size_t)y * W + x] = keep ? 1 : 0;
        }
    }
}

// grouping.py:150-170.  nms_hm [K,H*W] already NMS'd; tags [K,H*W,E].
// torch CPU topk(k) for k*64 <= n  ==  std::partial_sort on (value,index) with a
// value-only comparator (aten/src/ATen/native/TopKImpl.h); requires H*W >= 64*M.
HPO_API int hpo_topk(const float* nms_hm, const float* tags, int K, int H, int W, int E, int M,
                     float* tags_k, int32_t* coords_k, float* scores_k, int32_t* idx_k) {
    const int n = H * W;
    if ((long long)M * 64 > n) return 1;
    std::vector<std::pair<float, int64_t>> q(n);
    for (int k = 0; k < K; ++k) {
        const float* a = nms_hm + (size_t)k * n;
        for (int i = 0; i < n; ++i) { q[i].first = a[i]; q[i].second = i; }
        std::partial_sort(q.begin(), q.begin() + M, q.end(),
                          [](const std::pair<float, int64_t>& x, const std::pair<float, int64_t>& y) {
                              return (std::isnan(x.first) && !std::isnan(y.first)) || (x.first > y.first);
                          });
        for (int j = 0; j < M; ++j) {
            const int idx = (int)q[j].second;
            scores_k[k * M + j] = q[j].first;
            if (idx_k) idx_k[k * M + j] = idx;
            coords_k[(k * M + j) * 2 + 0] = idx % W;
            coords_k[(k * M + j) * 2 + 1] = idx / W;
            for (int e = 0; e < E; ++e) tags_k[(k * M + j) * E + e] = tags[((size_t)k * n + idx) * E + e];
        }
    }
    return 0;
}

// munkres on a rows x cols (rows <= cols <= 32) float64 matrix; out_col[r] = assigned column
HPO_API int hpo_munkres(const double* cost, int rows, int cols, int32_t* out_col) {
    if (rows > cols || cols > kMaxPeople) return 1;
    std::vector<double> C((size_t)cols * cols, 0.0);
    for (int i = 0; i < rows; ++i) for (int j = 0; j < cols; ++j) C[(size_t)i * cols + j] = cost[(size_t)i * cols + j];
    Munkres m; m.n = cols; m.C = C.data();
    m.run();
    for (int i = 0; i < rows; ++i) out_col[i] = m.find_in_row(i, 1);
    return 0;
}

// grouping.py:85-145 as a flat-array algorithm.  Output poses [M][K][3+E] f32
// (zeros for missing joints), *n_person = min(#persons, M), *n_total = #persons, *flags (may be
// NULL) = hpd_group's bit 1: a cost was replaced by the guard below or a solve hit its step-6 cap.
HPO_API int hpo_match_by_tag(const float* tags_k, const int32_t* coords_k, const float* scores_k,
                             int K, int M, int E, double det_thr, double tag_thr,
                             const int* joints_order, float* poses, int32_t* n_person, int32_t* n_total,
                             int32_t* flags) {
    if (K > kMaxKpts || M > kMaxPeople || E > kMaxEmb) return 1;
    static const int kOrder17[17] = {0, 1, 2, 3, 4, 5, 6, 11, 12, 7, 8, 9, 10, 13, 14, 15, 16};
    const int D = 3 + E;
    std::memset(poses, 0, sizeof(float) * (size_t)M * K * D);
    int fl = 0;
    int P = 0;              // persons tracked (<= M)
    int Ptotal = 0;         // persons created (dict size); only the first M are ever read
    float key[kMaxPeople];
    float taglist[kMaxPeople][kMaxKpts][kMaxEmb];
    int ntag[kMaxPeople];

    auto put_joint = [&](int p, int k, int r) {
        float* d = poses + ((size_t)p * K + k) * D;
        d[0] = (float)coords_k[(k * M + r) * 2 + 0];
        d[1] = (float)coords_k[(k * M + r) * 2 + 1];
        d[2] = scores_k[k * M + r];
        for (int e = 0; e < E; ++e) d[3 + e] = tags_k[(k * M + r) * E + e];
    };
    // dict.setdefault(key) + tag_dict[key] = [tag]   (grouping.py:109-111,141-143)
    auto new_or_collide = [&](int k, int r) {
        const float* tg = tags_k + (size_t)(k * M + r) * E;
        for (int p = 0; p < P; ++p)
            if (key[p] == tg[0]) {           // float ==: +-0 collide, NaN never
                put_joint(p, k, r);
                ntag[p] = 1;
                for (int e = 0; e < E; ++e) taglist[p][0][e] = tg[e];
                return;
            }
        // keys of persons beyond the first M are never outputs nor match columns;
        // a collision with one of them only edits that discarded person.
        ++Ptotal;
        if (P < M) {
            key[P] = tg[0];
            put_joint(P, k, r);
            ntag[P] = 1;
            for (int e = 0; e < E; ++e) taglist[P][0][e] = tg[e];
            ++P;
        }
    };

    for (int it = 0; it < K; ++it) {
        const int k = joints_order ? joints_order[it] : (K == 17 ? kOrder17[it] : it);
        int rows[kMaxPeople], nr = 0;
        for (int r = 0; r < M; ++r) if ((double)scores_k[k * M + r] > det_thr) rows[nr++] = r;
        if (nr == 0) continue;
        if (it == 0 || Ptotal == 0) {
            for (int a = 0; a < nr; ++a) new_or_collide(k, rows[a]);
            continue;
        }
        const int G = P;   // min(len(dict), M): P is already capped at M
        float mean[kMaxPeople][kMaxEmb];
        // np_mean_vectors expects [n][E] packed; taglist rows are [kMaxKpts][kMaxEmb] -> repack
        for (int p = 0; p < G; ++p) {
            float packed[kMaxKpts * kMaxEmb];
            for (int i = 0; i < ntag[p]; ++i) for (int e = 0; e < E; ++e) packed[i * E + e] = taglist[p][i][e];
            np_mean_vectors(packed, ntag[p], E, mean[p]);
        }
        const int n = std::max(G, nr);
        std::vector<double> C((size_t)n * n, 0.0), dist((size_t)nr * G);
        for (int a = 0; a < nr; ++a) {
            const float* tg = tags_k + (size_t)(k * M + rows[a]) * E;
            const double sc = (double)scores_k[k * M + rows[a]];
            for (int p = 0; p < G; ++p) {
                double s = 0.0;
                for (int e = 0; e < E; ++e) {
                    const double d = (double)tg[e] - (double)mean[p][e];
                    const double sq = d * d;
                    s = (e == 0) ? sq : s + sq;
                }
                const double dn = std::sqrt(s);
                dist[(size_t)a * G + p] = dn;
                double c = std::nearbyint(dn) * 100.0 - sc;   // np.round: half to even
                // Library policy, not the reference's: munkres 1.1.4 never returns on a NaN row, nor
                // once step 6's sys.maxsize sentinel stops making zeros (costs >= 2^63).  Such costs
                // become the reference's own "cannot match" value and the image is flagged.
                if (!(std::fabs(c) < 0x1p63)) { c = 1e10; fl |= 2; }
                C[(size_t)a * n + p] = c;
            }
            for (int p = G; p < n; ++p) C[(size_t)a * n + p] = 1e10;
        }
        Munkres mk; mk.n = n; mk.C = C.data();
        const bool solved = mk.run();    // with the guard the cap is never reached; if it is, nobody matches
        if (!solved) fl |= 2;
        for (int a = 0; a < nr; ++a) {
            const int c = solved ? mk.find_in_row(a, 1) : -1;
            if (c >= 0 && c < G && dist[(size_t)a * G + c] < tag_thr) {
                put_joint(c, k, rows[a]);
                const float* tg = tags_k + (size_t)(k * M + rows[a]) * E;
                for (int e = 0; e < E; ++e) taglist[c][ntag[c]][e] = tg[e];
                ++ntag[c];
            } else {
                new_or_collide(k, rows[a]);
            }
        }
    }
    *n_person = P;
    if (n_total) *n_total = Ptotal;
    if (flags) *flags = fl;
    return 0;
}

// grouping.py:172-191 on float32 poses [P][K][D]; hm [K,H,W]
HPO_API void hpo_adjust(float* poses, int P, int K, int D, const float* hm, int H, int W) {
    for (int p = 0; p < P; ++p) for (int k = 0; k < K; ++k) {
        float* d = poses + ((size_t)p * K + k) * D;
        if (d[2] == 0.0f) continue;
        float x = d[0], y = d[1];
        const int xi = (int)x, yi = (int)y;
        const float* m = hm + (size_t)k * H * W;
        x += (m[(size_t)yi * W + std::min(xi + 1, W - 1)] > m[(size_t)yi * W + std::max(xi - 1, 0)]) ? 0.25f : -0.25f;
        y += (m[(size_t)std::min(yi + 1, H - 1) * W + xi] > m[(size_t)std::max(yi - 1, 0) * W + xi]) ? 0.25f : -0.25f;
        d[0] = x + 0.5f;
        d[1] = y + 0.5f;
    }
}

// grouping.py:276: float32 mean over K scores, numpy pairwise-8 order
HPO_API void hpo_person_scores(const float* poses, int P, int K, int D, float* out) {
    for (int p = 0; p < P; ++p)
        out[p] = (0.0f + np_sum_pairwise8(poses + (size_t)p * K * D + 2, K, D)) / (float)K;
}

// grouping.py:193-250 for one person (poses row [K][D]); hm [K,H,W], tags [K,H,W,E]
HPO_API void hpo_refine_person(const float* hm, const float* tags, int K, int H, int W, int E, float* person) {
    const int D = 3 + E;
    float tl[kMaxKpts * kMaxEmb]; int nt = 0;
    for (int k = 0; k < K; ++k) {
        const float* d = person + (size_t)k * D;
        if (d[2] > 0.0f) {
            const int x = (int)d[0], y = (int)d[1];
            for (int e = 0; e < E; ++e) tl[nt * E + e] = tags[(((size_t)k * H + y) * W + x) * E + e];
            ++nt;
        }
    }
    float T[kMaxEmb] = {0.f, 0.f};
    if (nt > 0) np_mean_vectors(tl, nt, E, T);
    else for (int e = 0; e < E; ++e) T[e] = std::numeric_limits<float>::quiet_NaN();  // np.mean([]) -> nan
    for (int k = 0; k < K; ++k) {
        float* d = person + (size_t)k * D;
        if (!(d[2] == 0.0f)) continue;      // only missing joints can be replaced (grouping.py:248)
        const float* m = hm + (size_t)k * H * W;
        const float* tg = tags + (size_t)k * H * W * E;
        float best = 0.f; int bi = -1;
        for (int i = 0; i < H * W; ++i) {
            float dd;
            if (E == 1) { const float a = tg[i] - T[0]; dd = std::sqrt(a * a); }
            else {
                const float a = tg[(size_t)i * 2] - T[0], b = tg[(size_t)i * 2 + 1] - T[1];
                const float a2 = a * a, b2 = b * b;
                dd = std::sqrt(a2 + b2);
            }
            const float v = m[i] - std::nearbyintf(dd);
            if (bi < 0 || v > best || (std::isnan(v) && !std::isnan(best))) { best = v; bi = i; }
        }
        const int y = bi / W, x = bi % W;
        const float val = m[bi];
        if (!(val > 0.0f)) continue;
        float fx = (float)x + 0.5f, fy = (float)y + 0.5f;
        fx += (m[(size_t)y * W + std::min(x + 1, W - 1)] > m[(size_t)y * W + std::max(x - 1, 0)]) ? 0.25f : -0.25f;
        fy += (m[(size_t)std::min(y + 1, H - 1) * W + x] > m[(size_t)std::max(y - 1, 0) * W + x]) ? 0.25f : -0.25f;
        d[0] = fx; d[1] = fy; d[2] = val;
    }
}

// grouping.py:252-283 on one image.  hm [K,H,W], tags [K,H,W,E] (aggregated, full res).
// poses [M][K][3+E], scores [M]; returns person count in *n_person; *fallback = 1 when the
// "take only best pred" branch (grouping.py:262-269) fired (the reference returns float64
// there with score 0.01; here the float32 image of that is produced and flagged).
HPO_API int hpo_parse(const float* hm, const float* tags, int K, int H, int W, int E, int M,
                      double det_thr, double tag_thr, int do_adjust, int do_refine,
                      float* poses, float* person_scores, int32_t* n_person, int32_t* fallback,
                      float* tags_k_out, int32_t* coords_k_out, float* scores_k_out, int32_t* idx_k_out) {
    const size_t n = (size_t)H * W;
    const int D = 3 + E;
    std::vector<float> nmsd((size_t)K * n);
    hpo_nms(hm, K, H, W, nmsd.data(), nullptr);
    std::vector<float> tags_k((size_t)K * M * E), scores_k((size_t)K * M);
    std::vector<int32_t> coords_k((size_t)K * M * 2), idx_k((size_t)K * M);
    if (hpo_topk(nmsd.data(), tags, K, H, W, E, M, tags_k.data(), coords_k.data(), scores_k.data(), idx_k.data())) return 1;
    if (tags_k_out) std::memcpy(tags_k_out, tags_k.data(), tags_k.size() * 4);
    if (coords_k_out) std::memcpy(coords_k_out, coords_k.data(), coords_k.size() * 4);
    if (scores_k_out) std::memcpy(scores_k_out, scores_k.data(), scores_k.size() * 4);
    if (idx_k_out) std::memcpy(idx_k_out, idx_k.data(), idx_k.size() * 4);
    int32_t P = 0, Pt = 0;
    if (hpo_match_by_tag(tags_k.data(), coords_k.data(), scores_k.data(), K, M, E, det_thr, tag_thr, nullptr, poses, &P, &Pt, nullptr)) return 1;
    *fallback = 0;
    if (P == 0) {
        *fallback = 1;
        P = 1;
        for (int k = 0; k < K; ++k) {
            float* d = poses + (size_t)k * D;
            d[0] = (float)coords_k[(k * M) * 2 + 0];
            d[1] = (float)coords_k[(k * M) * 2 + 1];
            d[2] = 0.01f;
            for (int e = 0; e < E; ++e) { const float t = tags_k[(size_t)(k * M) * E + e]; d[3 + e] = std::isnan(t) ? 0.f : t; }
        }
    }
    if (do_adjust) hpo_adjust(poses, P, K, D, hm, H, W);
    hpo_person_scores(poses, P, K, D, person_scores);
    if (do_refine) for (int p = 0; p < P; ++p) hpo_refine_person(hm, tags, K, H, W, E, poses + (size_t)p * K * D);
    *n_person = P;
    return 0;
}
