"""CPU model (numpy, fp32 step by step) of the bucket keys and the walk order of the bucketed NMS kernel
`nms_bucket_kernel` (faster_rcnn_pytorch_b200/csrc/nms_bucket.cu) with its (x bin, y bin, area class) keys: 8 x 4
cells of the box centre at 1024 threads with one or two CTAs per image, 8 x 1 in the other launches, 60 area classes (4 per octave, clamped to
2^-15 .. 1), class minor.

Where tests/nms_model.py restates the pruning as a mask, this model walks the bucketed arrays range by range in the
order of `bk_walk` (screen phase D: kept list against the chunk's candidates) and `bk_walk_up` (pair phase H: every
survivor against the survivors above it), so it can check that the walks visit every pair that can suppress, and
each pair among the survivors exactly once, from its lower bucketed position.  Constants and pair decisions are
nms_model's.  Test infrastructure only."""
from __future__ import annotations

import numpy as np

import nms_model as nm

f32 = np.float32
K_X, K_CLASSES = 8, 60


class Grid:
    def __init__(self, ky: int):
        self.kx, self.ky, self.kc = K_X, ky, K_CLASSES
        self.keys = self.kx * self.ky * self.kc   # key `keys`: boxes that must always be tested

    def cls(self, a):
        bits = np.asarray(a, f32).view(np.int32)
        return np.minimum(self.kc - 1, np.maximum(0, (bits >> 21) - ((127 - 15) << 2)))

    @staticmethod
    def bin(c, nb):
        with np.errstate(invalid="ignore"):
            v = np.trunc((np.asarray(c, f32) * f32(nb)).astype(f32))
        v = np.where(np.isnan(v), 0, v)
        return np.minimum(nb - 1, np.maximum(0, v.astype(np.int64)))

    def key(self, b, sa):
        cx = (f32(0.5) * (b[:, 0] + b[:, 2]).astype(f32)).astype(f32)
        cy = (f32(0.5) * (b[:, 1] + b[:, 3]).astype(f32)).astype(f32)
        k = (self.bin(cx, self.kx) * self.ky + self.bin(cy, self.ky)) * self.kc + self.cls(nm.box_area(b))
        return np.where(np.isnan(sa), self.keys, k)

    def admissible(self, b, t):
        """Per box: c_lo, c_hi, x_lo, x_hi, y_lo, y_hi (bk_admissible)."""
        a = nm.box_area(b)
        with np.errstate(invalid="ignore", over="ignore"):
            out = [self.cls((a * t["alo"]).astype(f32)), self.cls((a * t["ahi"]).astype(f32))]
            for lo, hi, nb in ((0, 2, self.kx), (1, 3, self.ky)):
                c = (f32(0.5) * (b[:, lo] + b[:, hi]).astype(f32)).astype(f32)
                r = (((t["fx"] * (b[:, hi] - b[:, lo]).astype(f32)).astype(f32) * f32(1.0001)).astype(f32)
                     + f32(2.0e-6)).astype(f32)
                out += [self.bin((c - r).astype(f32), nb), self.bin((c + r).astype(f32), nb)]
        if self.ky == 1:
            out[4][:] = 0
            out[5][:] = 0
        return np.stack(out, axis=1)

    def bucket(self, keys):
        """Bucketed order (key, then position) and the start offsets start[0 .. keys + 1]."""
        order = np.lexsort((np.arange(len(keys)), keys))
        start = np.searchsorted(keys[order], np.arange(self.keys + 2), side="left")
        return order, start

    def _cells(self, ad, xb, yb):
        """Admissible cells from (xb, yb) on, in key order (y minor): bk_walk_cells."""
        while xb <= ad[3]:
            yield xb * self.ky + yb
            yb += 1
            if yb > ad[5]:
                yb, xb = ad[4], xb + 1

    def walk(self, start, ad, every):
        """Positions bk_walk visits, in order."""
        if every:
            return [range(0, start[self.keys + 1])]
        r = [range(start[c * self.kc + ad[0]], start[c * self.kc + ad[1] + 1]) for c in self._cells(ad, ad[2], ad[4])]
        return r + [range(start[self.keys], start[self.keys + 1])]

    def walk_up(self, start, p, own_key, ad, every):
        """Positions bk_walk_up visits from bucketed position p, in order."""
        total = start[self.keys + 1]
        if every:
            return [range(p + 1, total)]
        cell = own_key // self.kc
        r = [range(p + 1, start[cell * self.kc + ad[1] + 1])]
        xb, yb = cell // self.ky, cell % self.ky + 1
        if yb > ad[5]:
            yb, xb = ad[4], xb + 1
        r += [range(start[c * self.kc + ad[0]], start[c * self.kc + ad[1] + 1]) for c in self._cells(ad, xb, yb)]
        return r + [range(start[self.keys], total)]


def _positions(ranges):
    return np.concatenate([np.arange(r.start, r.stop) for r in ranges]) if ranges else np.zeros(0, np.int64)


def nms_cells(boxes: np.ndarray, thr: float, max_keep: int, chunk_sizes=(2048,), ky: int = 4,
              stats: dict | None = None):
    """Keep list (positions, ascending) of greedy NMS over score-sorted `boxes`, first `max_keep` keeps, computed by
    walking the bucketed arrays the way the kernel walks them.  `stats` collects the pair counts of both phases and
    the walk checks: `missed_d` / `missed_h` (pairs that suppress but were not visited), `twice_h` (pairs among the
    survivors visited more than once) and `down_h` (visits to a position not above the walker's)."""
    t = nm.make_thr(thr)
    assert t["fast"], "the bucketed kernel is only selected for screenable thresholds"
    g = Grid(ky)
    boxes = np.ascontiguousarray(boxes, f32)
    n = boxes.shape[0]
    st = dict(pairs_d=0, pairs_h=0, missed_d=0, missed_h=0, twice_h=0, down_h=0)
    kept: list[int] = []
    base, ci = 0, 0
    while base < n and len(kept) < max_keep:
        kc = chunk_sizes[min(ci, len(chunk_sizes) - 1)]
        ci += 1
        cand = boxes[base:base + kc]
        m = cand.shape[0]
        sa_c = nm.screen_area(cand, t["c2"])
        ad_c = g.admissible(cand, t)
        every_c = np.isnan(sa_c)
        dead = np.zeros(m, bool)
        if kept:  # phase D: the bucketed kept list against every candidate
            kb = boxes[np.asarray(kept)]
            sa_k = nm.screen_area(kb, t["c2"])
            lorder, lstart = g.bucket(g.key(kb, sa_k))
            lb, lsa = kb[lorder], sa_k[lorder]
            hit = nm.suppress_screen(lb, lsa, cand, sa_c) & nm.suppress_exact(lb, cand, t["up"])   # [list, cand]
            for i in range(m):
                vis = _positions(g.walk(lstart, ad_c[i], every_c[i]))
                st["pairs_d"] += len(vis)
                seen = np.zeros(len(lb), bool)
                seen[vis] = True
                st["missed_d"] += int((hit[:, i] & ~seen).sum())
                dead[i] = hit[vis, i].any()
        # phase H: the survivors, bucketed by (key, chunk position), each walking the positions above its own
        surv = np.nonzero(~dead)[0]
        sorder, sstart = g.bucket(g.key(cand[surv], sa_c[surv]))
        sidx = surv[sorder]                                      # bucketed position -> chunk position
        skey = g.key(cand[sidx], sa_c[sidx])
        ns = len(sidx)
        visits = np.zeros((ns, ns), np.int32)
        for p in range(ns):
            i = sidx[p]
            vis = _positions(g.walk_up(sstart, p, skey[p], ad_c[i], every_c[i]))
            st["pairs_h"] += len(vis)
            st["down_h"] += int((vis <= p).sum())
            np.add.at(visits[p], vis, 1)
        sb, ssa = cand[sidx], sa_c[sidx]
        earlier = sidx[:, None] < sidx[None, :]                  # [p, k]: p is earlier in score order
        ex = nm.suppress_exact(sb, sb, t["up"])                  # ex[a, b]: a suppresses b if a is earlier
        sup = np.where(earlier, ex, ex.T) & (np.arange(ns)[:, None] != np.arange(ns)[None, :])
        met = visits + visits.T
        st["twice_h"] += int((met > 1).sum()) // 2
        st["missed_h"] += int((sup & (met == 0)).sum()) // 2
        scr = nm.suppress_screen(sb, ssa, sb, ssa)
        edge = (met > 0) & scr & np.where(earlier, ex, False)    # edge[p, k]: p earlier, suppresses k
        pred = np.zeros((m, m), bool)                            # pred[j, i]: chunk position j suppresses i
        pj, pk = np.nonzero(edge)
        pred[sidx[pj], sidx[pk]] = True
        state = np.where(dead, 2, 0)                             # 0 undecided, 1 kept, 2 removed
        while (state == 0).any():
            has_kept = (pred & (state == 1)[:, None]).any(axis=0)
            pending = (pred & (state == 0)[:, None]).any(axis=0)
            new = state.copy()
            new[(state == 0) & has_kept] = 2
            new[(state == 0) & ~has_kept & ~pending] = 1
            state = new
        for i in np.nonzero(state == 1)[0]:
            if len(kept) < max_keep:
                kept.append(base + int(i))
        base += m
    if stats is not None:
        stats.update(st)
    return np.asarray(kept, np.int64)
