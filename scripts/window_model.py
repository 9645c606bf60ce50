"""Estimate how the sweep's 51.7M scattered fp64 REDs would split under a dense row-window scheme (RMAT scale S, ef 16).
Mimics the library's layout: internal ids by descending in-degree, (row, block) segments, pieces of <=64 entries,
pieces ordered by (block, kind), stable -> row-ascending inside a (block, kind).  For each window size and density
threshold it also models the stream a windowed layout would read: the padding of one partial group per (dense cell, kind)
and the row bytes saved by 1-byte (256-row window) or 2-byte row offsets.  Needs about 30 GB of RAM at scale 24.

    python scripts/window_model.py [S]"""
import sys, time
import numpy as np

S = int(sys.argv[1]) if len(sys.argv) > 1 else 24
E = 16 << S
V = 1 << S
rng = np.random.default_rng(0)
t0 = time.time()
src = np.zeros(E, dtype=np.int64)
dst = np.zeros(E, dtype=np.int64)
a, b, c = 0.57, 0.19, 0.19
CH = 1 << 26
for o in range(0, E, CH):
    n = min(CH, E - o)
    s = np.zeros(n, dtype=np.int64); d = np.zeros(n, dtype=np.int64)
    for bit in range(S):
        r = rng.random(n, dtype=np.float32)
        sb = r >= a + b            # c or d quadrant -> src bit
        db = ((r >= a) & (r < a + b)) | (r >= a + b + c)
        s |= sb.astype(np.int64) << bit
        d |= db.astype(np.int64) << bit
    src[o:o + n] = s; dst[o:o + n] = d
print("gen", time.time() - t0, flush=True)
perm = rng.permutation(V)          # scramble
src = perm[src]; dst = perm[dst]
indeg = np.bincount(dst, minlength=V)
outdeg = np.bincount(src, minlength=V)
nonisol = (indeg + outdeg) > 0
# internal ids: descending in-degree among non-isolated vertices
order = np.lexsort((np.arange(V), -indeg))
order = order[nonisol[order]]
nv = order.size
internal = np.full(V, -1, dtype=np.int64); internal[order] = np.arange(nv)
src = internal[src]; dst = internal[dst]
n_cov = int((indeg > 0).sum())
print("V", nv, "n_cov", n_cov, time.time() - t0, flush=True)
W = 49088
B = (nv + W - 1) // W
blk = src // W
key = dst * B + blk                 # (row, block) segment id
del src
key.sort()
print("sort", time.time() - t0, flush=True)
brk = np.flatnonzero(np.diff(key)) + 1
starts = np.concatenate(([0], brk)); lens = np.diff(np.concatenate((starts, [E])))
seg = key[starts]; del key
row = seg // B; sb = seg % B
npieces = (lens + 63) // 64
print("segments", seg.size, "pieces", npieces.sum(), flush=True)
# pieces: full 64-entry pieces + remainder
prow = np.repeat(row, npieces); pblk = np.repeat(sb, npieces)
first = np.repeat(np.cumsum(npieces) - npieces, npieces)
j = np.arange(prow.size) - first
plen = np.minimum(64, np.repeat(lens, npieces) - 64 * j)
kind = np.where(plen == 1, 0, np.where(plen == 2, 1, np.where(plen <= 4, 2, 3 + (plen + 7) // 8 - 1)))
o = np.lexsort((prow, kind, pblk))
prow, pblk, kind = prow[o], pblk[o], kind[o]
P = prow.size
print("pieces", P, time.time() - t0, flush=True)

# current: one RED instruction per 32 consecutive pieces of a (block, kind) run (F8 hub runs collapse; ignored here)
cls = pblk * 11 + kind
cstart = np.concatenate(([0], np.flatnonzero(np.diff(cls)) + 1))
pos = np.arange(P) - np.repeat(cstart, np.diff(np.concatenate((cstart, [P]))))
warp_op = np.repeat(np.arange(cstart.size), np.diff(np.concatenate((cstart, [P])))) * (1 << 22) + pos // 32
sect = prow // 4
k2 = np.unique(warp_op * (1 << 24) + sect) if P < (1 << 31) else None
print("modelled RED sectors now:", k2.size if k2 is not None else "n/a", flush=True)
del k2, warp_op, pos

del cls, cstart


# Stream bytes of a layout whose (block, kind) runs are cut into the given classes: every class fills whole groups of its
# kind (kind_pieces per group, kind_steps step-rows of 512 bytes of ids each), rows are `row_bytes` per piece slot.
GP = np.array([256, 128, 64] + [32] * 8)
STEPS = np.array([1, 1, 1] + list(range(1, 9)))


def groups_of(n_pieces, kinds):
    return (n_pieces + GP[kinds] - 1) // GP[kinds]


def stream_bytes(groups, kinds, row_bytes):
    return int((groups * STEPS[kinds] * 512).sum()), int((groups * GP[kinds] * row_bytes).sum())


# today: one class per (block, kind)
bk = pblk * 11 + kind
u, n_bk = np.unique(bk, return_counts=True)
g_now = groups_of(n_bk, u % 11)
ids_now, rows_now = stream_bytes(g_now, u % 11, 4)
pad_now = int((g_now * GP[u % 11]).sum()) - P
print(f"today: groups {g_now.sum()}, padding pieces {pad_now}, ids {ids_now / 1e6:.1f} MB, "
      f"rows {rows_now / 1e6:.1f} MB", flush=True)
del bk, u, n_bk, g_now

for Rw in (256, 1024, 4096):
    win = prow // Rw
    k = pblk * (nv // Rw + 1) + win
    cnt_all = np.bincount(k)
    cnt = cnt_all[cnt_all > 0]
    flush = Rw * 8 // 32
    for thr in (flush, flush // 2):
        dense = cnt >= thr
        print(f"window {Rw} rows, dense if >= {thr} pieces: dense windows {dense.sum()}, pieces in them {cnt[dense].sum()} "
              f"({cnt[dense].sum()/P:.2%}), sectors {cnt[~dense].sum() + dense.sum()*flush} vs {P}", flush=True)
        # padding: dense pieces form classes (dense cell, kind); sparse pieces keep one class per (block, kind).
        # Dense rows are 1-byte offsets when the window has 256 rows, else 2-byte.
        pd = cnt_all[k] >= thr
        n_dense_pieces = int(pd.sum())
        ud, nd = np.unique(k[pd] * 11 + kind[pd], return_counts=True)
        us, ns = np.unique((pblk[~pd] * 11 + kind[~pd]), return_counts=True)
        gd, gs = groups_of(nd, ud % 11), groups_of(ns, us % 11)
        pad = int((gd * GP[ud % 11]).sum() + (gs * GP[us % 11]).sum()) - P
        ids_d, rows_d = stream_bytes(gd, ud % 11, 1 if Rw <= 256 else 2)
        ids_s, rows_s = stream_bytes(gs, us % 11, 4)
        ids_new, rows_new = ids_d + ids_s, rows_d + rows_s
        print(f"    layout: {n_dense_pieces} dense pieces in {ud.size} (cell, kind) classes; padding pieces {pad} "
              f"(today {pad_now}); ids {ids_new / 1e6:.1f} MB "
              f"({(ids_new - ids_now) / 1e6:+.1f}), rows {rows_new / 1e6:.1f} MB ({(rows_new - rows_now) / 1e6:+.1f}), "
              f"id+row stream {(ids_new + rows_new) / 1e6:.1f} MB vs {(ids_now + rows_now) / 1e6:.1f} MB today", flush=True)
        del pd, ud, nd, us, ns, gd, gs
    del win, k, cnt_all
# pieces by block range and by row range
for b0, b1 in ((0, 1), (1, 4), (4, 16), (16, 64), (64, B)):
    m = (pblk >= b0) & (pblk < b1)
    print(f"blocks [{b0},{b1}) pieces {m.sum()}  hub-row (indeg>=32) pieces {(m & (prow < int((indeg>=32).sum()))).sum()}", flush=True)
