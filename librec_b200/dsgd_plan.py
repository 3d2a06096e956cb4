"""The DSGD stratum schedule (host logic) -- the same pure functions as librec_b200/csrc/dsgd.cuh and staging.cuh (item blocks,
stream order).

World of G ranks, one per GPU.  Rank g owns a user shard for the whole run.  Items are cut into G
contiguous blocks balanced by global rating count.  In sub-epoch s rank g trains on item block
(g + s) mod G, then passes that block to rank g-1 and receives the next one from rank g+1.  After G
sub-epochs every rank holds its starting block again.  Blocks of one sub-epoch are disjoint in users
and in items, so a DSGD epoch equals a sequential walk over its strata in (sub-epoch, rank) order.
"""
import numpy as np


def block_at(rank, world, sub):
    return (rank + sub) % world


def send_peer(rank, world):
    return (rank - 1 + world) % world


def recv_peer(rank, world):
    return (rank + 1) % world


def item_bounds(item_count, world):
    """contiguous item blocks balanced by rating count: block b = [bounds[b], bounds[b+1])"""
    item_count = np.asarray(item_count, np.int64)
    I = item_count.shape[0]
    total = int(item_count.sum())
    bounds = [I] * (world + 1)
    bounds[0] = 0
    acc, b = 0, 1
    for i in range(I):
        if b >= world:
            break
        acc += int(item_count[i])
        while b < world and (acc * world >= total * b or I - (i + 1) <= world - b):
            bounds[b] = i + 1
            b += 1
    for j in range(1, world + 1):
        if bounds[j] < bounds[j - 1]:
            bounds[j] = bounds[j - 1]
    bounds[world] = I
    return bounds


RUN_MIN_DEGREE = 128          # LRK_RUN_MIN_DEGREE: items with at least this many ratings in a block shard get run tiles
_M64 = (1 << 64) - 1


def _hash32(x):
    """lrk_hash32 (csrc/staging.cuh): the splitmix64 finaliser, high word; x: uint64 array"""
    with np.errstate(over="ignore"):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        x = x ^ (x >> np.uint64(31))
    return x >> np.uint64(32)


def stream_order(rowptr, col, val, I, seed, bounds=None):
    """The staged COO stream of the SGD epoch (csrc/staging.cuh, stage_tile_keys) -> (su, si, sr, run_tiles, max_item_deg).
    Per item block (one block without bounds, otherwise the DSGD item blocks): [item-run tiles] [the rest, shuffled], i.e. one
    stable sort of entry e on  key = block:6 | is_rest:1 | hash:32 | tile or entry id:25.  An item with deg >= RUN_MIN_DEGREE
    gives deg // 32 tiles of 32 ratings, in CSR order; its remaining ratings join the rest.  seed: the handle's seed
    (+ 977 * rank on a DSGD rank).  With bounds the item ids of the stream are local to their block."""
    rowptr, col = np.asarray(rowptr, np.int64), np.asarray(col, np.int64)
    n = col.shape[0]
    row_of = np.repeat(np.arange(rowptr.shape[0] - 1), np.diff(rowptr))
    deg = np.bincount(col, minlength=I)
    runs = np.where(deg >= RUN_MIN_DEGREE, deg // 32, 0)
    run_base = np.cumsum(runs) - runs
    order = np.argsort(col, kind="stable")                          # the by-item order
    rank = np.empty(n, np.int64)
    rank[order] = np.arange(n) - (np.cumsum(deg) - deg)[col[order]]
    blk = np.searchsorted(np.asarray(bounds[1:-1]), col, side="right") if bounds is not None else np.zeros(n, np.int64)
    e = np.arange(n, dtype=np.uint64)
    tile = (run_base[col] + rank // 32).astype(np.uint64)
    in_run = rank < 32 * runs[col]
    m_tile, m_rest = np.uint64((seed * 0xA24BAED4963EE407) & _M64), np.uint64((seed * 0xD6E8FEB86659FD93) & _M64)
    low25 = np.uint64(0x1FFFFFF)
    key_tile = (_hash32(tile ^ m_tile) << np.uint64(25)) | (tile & low25)
    key_rest = np.uint64(1 << 57) | (_hash32(e ^ m_rest) << np.uint64(25)) | (e & low25)
    key = (blk.astype(np.uint64) << np.uint64(58)) | np.where(in_run, key_tile, key_rest)
    perm = np.argsort(key, kind="stable")
    si = col[perm] - (np.asarray(bounds, np.int64)[blk[perm]] if bounds is not None else 0)
    return (row_of[perm].astype(np.int32), si.astype(np.int32), np.asarray(val, np.float64)[perm].astype(np.float32),
            int(runs.sum()), int(deg.max()) if n else 0)


def segments(col, bounds):
    """per item block: indices of the CSR entries whose column falls in it (CSR order kept)"""
    col = np.asarray(col)
    blk = np.searchsorted(np.asarray(bounds[1:-1]), col, side="right")
    return [np.nonzero(blk == b)[0] for b in range(len(bounds) - 1)]


# ---- flag protocol of the experimental fused epoch kernel (csrc/dsgd_fused.cuh), restated as a step function so that the
# sequencing (who may read / overwrite which buffer when) can be exercised on the CPU under arbitrary interleavings.
class FusedRank:
    """One rank's view: two block buffers, ready[2] (written by rank+1), peer_free[2] (written by rank-1).  `step()` advances
    the rank by one protocol action if its wait condition holds and returns what it did (None = blocked)."""

    def __init__(self, rank, world, start_block):
        self.rank, self.world = rank, world
        self.buf = [start_block, None]          # block id held in each buffer (None = stale / free)
        self.ready = [0, 0]
        self.peer_free = [0, 0]
        self.cur0, self.seq0 = 0, 0
        self.t, self.phase = 0, "wait_ready"    # phases per stratum: wait_ready -> compute -> wait_free -> push
        self.trained = []                       # (seq, block) in the order the rank trained them
        self.final_wait_done = False

    def begin_epoch(self):
        self.t, self.phase, self.final_wait_done = 0, "wait_ready", False

    def finished(self):
        return self.t == self.world and self.final_wait_done

    def step(self, ranks):
        G = self.world
        prev, nxt = ranks[(self.rank - 1) % G], ranks[(self.rank + 1) % G]
        if self.t == G:                                        # the block of the next epoch's first stratum must have arrived
            b = (self.cur0 + G) & 1
            if self.ready[b] >= self.seq0 + G:
                self.final_wait_done = True
                self.cur0, self.seq0 = b, self.seq0 + G
                return "final"
            return None
        b, seq = (self.cur0 + self.t) & 1, self.seq0 + self.t
        if self.phase == "wait_ready":
            if self.ready[b] < seq:
                return None
            self.phase = "compute"
            return "ready"
        if self.phase == "compute":
            assert self.buf[b] is not None, "trained on a buffer that was never filled"
            self.trained.append((seq, self.buf[b]))
            self.phase = "wait_free"
            return "compute"
        if self.phase == "wait_free":
            if self.peer_free[b ^ 1] < seq:
                return None
            self.phase = "push"
            return "free"
        # push: copy my buffer b into prev's buffer b^1, then signal
        assert prev.phase_reads() != (b ^ 1), "pushed into a buffer its owner is still reading"
        prev.buf[b ^ 1] = self.buf[b]
        prev.ready[b ^ 1] = seq + 1
        nxt.peer_free[b] = seq + 1                             # my buffer b may be overwritten by rank+1 again
        self.buf[b] = None
        self.t += 1
        self.phase = "wait_ready"
        return "push"

    def phase_reads(self):
        """index of the buffer this rank is reading right now (computing on it or pushing from it), else -1"""
        if self.t < self.world and self.phase in ("compute", "wait_free", "push"):
            return (self.cur0 + self.t) & 1
        return -1
