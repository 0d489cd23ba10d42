"""Python statement of the One-Euro smoothing of tracked joints (hpd_track_smooth, include/hpdecode.h): the 1-Euro
filter of Casiez, Roussel and Vogel (CHI 2012), per track, joint and coordinate, at a constant frame rate.

Test infrastructure only; the product never imports it.  Every step is one float64 operation (Python floats, correctly
rounded, no FMA) in the kernel's order, so the kernel's coordinates are compared bit for bit.

The filter is stated as a function of (records, ids): ids are never reused and a dropped track never returns, so state
keyed by id lives exactly as long as its track.  Fed the kernel's own ids, it is independent of the tracker's OKS
decisions.

- Frames are numbered consecutively, one per record, fallback frames included.
- Person p < n_person with id >= 0, joint k visible (poses[p][k][2] > 0), raw COCO-section coordinate x:
  the first time the joint is seen in the track, x^ = x, dx^ = 0 and the output is x; otherwise, with g frames since
  it was last seen, te = g / fps, rd = (TWO_PI * d_cutoff) * te, ad = rd / (rd + 1), dx = (x - x^) / te,
  dx^ = ad * dx + (1 - ad) * dx^, c = min_cutoff + beta * |dx^|, r = (TWO_PI * c) * te, a = r / (r + 1),
  x^ = a * x + (1 - a) * x^, output x^.
- Invisible joints, persons with id -1 and the empty-scene fallback's pseudo-person: raw.  Rows p >= n_person: 0.
"""
import math

import numpy as np

from oracle.track_oracle import record_layout

TWO_PI = 2 * math.pi


class OneEuroOracle:
    def __init__(self, K=17, M=30, E=2, fps=30.0, min_cutoff=1.0, beta=0.0, d_cutoff=1.0):
        self.K, self.M, self.E = K, M, E
        self.fps, self.min_cutoff, self.beta, self.d_cutoff = float(fps), float(min_cutoff), float(beta), float(d_cutoff)
        self.frame_no = 0
        self.state = {}       # id -> {k: [x^, y^, dx^, dy^, last frame]}

    def reset(self):
        """Drops every filter (the tracks are dropped with them)."""
        self.state = {}

    def _step(self, x, xh, dxh, te, ad):
        dx = (x - xh) / te
        dxh = ad * dx + (1.0 - ad) * dxh
        c = self.min_cutoff + self.beta * abs(dxh)
        r = (TWO_PI * c) * te
        a = r / (r + 1.0)
        return a * x + (1.0 - a) * xh, dxh

    def frame(self, raw, ids):
        """One record (uint8 [row_bytes]) and its ids (int [M]) -> coords float64 [M, K, 2]."""
        K, M = self.K, self.M
        row, oc, op, osc, on, of = record_layout(K, M, self.E)
        raw = np.ascontiguousarray(raw, np.uint8)[:row]
        n = min(max(int(raw[on:on + 4].view(np.int32)[0]), 0), M)
        fallback = int(raw[of:of + 4].view(np.int32)[0]) & 1
        coco = raw[oc:op].view(np.float64).reshape(M, 3 * K + 1)
        poses = raw[op:osc].view(np.float32).reshape(M, K, 3 + self.E)
        out = np.zeros((M, K, 2), np.float64)
        f = self.frame_no
        for p in range(n):
            tid = int(ids[p])
            for k in range(K):
                x, y = float(coco[p, 3 * k]), float(coco[p, 3 * k + 1])
                if tid >= 0 and not fallback and poses[p, k, 2] > 0:
                    joints = self.state.setdefault(tid, {})
                    st = joints.get(k)
                    if st is None:
                        joints[k] = [x, y, 0.0, 0.0, f]
                    else:
                        te = float(f - st[4]) / self.fps
                        rd = (TWO_PI * self.d_cutoff) * te
                        ad = rd / (rd + 1.0)
                        x, dxh = self._step(x, st[0], st[2], te, ad)
                        y, dyh = self._step(y, st[1], st[3], te, ad)
                        joints[k] = [x, y, dxh, dyh, f]
                out[p, k] = x, y
        self.frame_no += 1
        return out

    def update(self, records, ids):
        """uint8 [n, row_bytes] records in time order and their ids int [n, M] -> coords float64 [n, M, K, 2]."""
        return np.stack([self.frame(r, i) for r, i in zip(np.asarray(records), np.asarray(ids))])
