"""Host model of one level of the card-set-grouped beam search (csrc/spl_m2.cuh), for tests that build rounds on
purpose: a port of the card-set hash and its inverse, the sort key and node-table home slot of a card set, a builder
of injected buy records, the run classes the dispatch (m2_group_tiny_kernel) gives a round's runs, and a plain
reference of one level with injected records.  Imports only numpy and the CPU oracle.
"""
import numpy as np

import oracle

M64 = (1 << 64) - 1
GOLDEN = 0x9E3779B97F4A7C15
MIX = 0xD6E8FEB86659FD93
MIX_INV = pow(MIX, -1, 1 << 64)
SORT_SHIFT = 34           # items are ordered, and runs cut, by the top 30 bits of the card-set hash (ITEM_KEY_LO)
TINY_ITEMS = 16           # buy-only runs of at most this many records of one card set: thread kernel
WARP_MAX_UNORDERED = 512  # candidates of a run above which the card-set-sharded round uses the CTA kernel
INJECT_ORD0 = 192         # ordinals of injected records: above the largest real fan-out (190)
MAX_SCORES = 2048         # distinct scores one level may hold in the score dictionary of the card-set-sharded cut

REC_DTYPE = np.dtype([('lo', '<u8'), ('hi', '<u8'), ('aux', '<u8'), ('link', '<u8')])


# ---------------------------------------------------------------- card-set hash (spl_common.cuh hash_key)
def hash_key(m0: int, m1: int) -> int:
    x = (m0 ^ (m1 * GOLDEN)) & M64
    x ^= x >> 32
    x = (x * MIX) & M64
    x ^= x >> 32
    x = (x * MIX) & M64
    x ^= x >> 32
    return x


def m0_for_hash(h: int, m1: int) -> int:
    """the card words m0 (cards 0..63) for which hash_key(m0, m1) == h: every step of the hash is a bijection"""
    x = h & M64
    x ^= x >> 32
    x = (x * MIX_INV) & M64
    x ^= x >> 32
    x = (x * MIX_INV) & M64
    x ^= x >> 32
    return x ^ ((m1 * GOLDEN) & M64)


def sort_key(h: int) -> int:
    return h >> SORT_SHIFT


def home_slot(h: int, nn: int) -> int:
    """umulhi(hash, nn): the node-table slot a card set's probe sequence starts at"""
    return (h * nn) >> 64


def card_words(lo: int, hi: int):
    """(m0, m1) = cards 0..63, cards 64..89 of a packed key (mask_words)"""
    m = ((int(lo) | int(hi) << 64) >> 15) & ((1 << 90) - 1)
    return m & M64, m >> 64


def set_hash(lo: int, hi: int) -> int:
    return hash_key(*card_words(lo, hi))


# ---------------------------------------------------------------- injected buy records
def legal_hand(gems) -> bool:
    return len(gems) == 5 and all(0 <= g <= 7 for g in gems) and sum(gems) <= 10


def make_record(m0: int, m1: int, gems, aux: int, q: int, ordinal: int, queue) -> tuple:
    """A buy record {key, aux, link = q << 8 | ordinal} for card set (m0, m1), as if queue state q generated it.
    Asserts what the kernels take for granted: breaking any of it indexes out of bounds on the device rather than
    giving a wrong answer."""
    assert legal_hand(gems), gems                       # gemrank of any other hand is 0xFFFF: past the node bitmap
    assert 0 <= m0 <= M64 and 0 <= m1 < 1 << 26
    key = (m0 | m1 << 64) << 15
    for i, g in enumerate(gems):
        key |= g << (3 * i)
    assert key < 1 << 105
    assert 0 <= q < len(queue)                          # the cut packs links into 8 + bitlen(queue length) bits
    assert INJECT_ORD0 <= ordinal <= 255                # never the link of a real successor (fan-out <= 190)
    assert card_words(queue['lo'][q], queue['hi'][q]) != (m0, m1)  # the warp kernel merges parents and records by rank
    return key & M64, key >> 64, int(aux), q << 8 | ordinal


def records(rows) -> np.ndarray:
    out = np.zeros(len(rows), REC_DTYPE)
    for i, r in enumerate(rows):
        out[i] = r
    return out


def random_hand(rng) -> tuple:
    while True:
        g = tuple(int(x) for x in rng.integers(0, 8, size=5))
        if sum(g) <= 10:
            return g


# ---------------------------------------------------------------- one level
def expand_queue(queue):
    """the successors of every queue state in arrival order (link = rank << 8 | ordinal) and each state's number of
    gem takes (successors that keep the card set)"""
    parts, ntk = [], np.zeros(len(queue), np.int64)
    for r in range(len(queue)):
        st = np.zeros(1, oracle.STATE_DTYPE)
        st['lo'], st['hi'], st['aux'] = queue['lo'][r], queue['hi'][r], queue['aux'][r]
        ch = oracle.expand(st)
        c = np.zeros(len(ch), REC_DTYPE)
        c['lo'], c['hi'], c['aux'] = ch['lo'], ch['hi'], ch['aux']
        c['link'] = (np.uint64(r) << np.uint64(8)) | np.arange(len(ch), dtype=np.uint64)
        same = (ch['lo'] >> np.uint64(15) == queue['lo'][r] >> np.uint64(15)) & (ch['hi'] == queue['hi'][r])
        ntk[r] = int(same.sum())
        parts.append(c)
    return (np.concatenate(parts) if parts else np.zeros(0, REC_DTYPE)), ntk


def ref_level(queue, visited: set, injected, heuristic: str, noise: str = 'const', beam: int = None, expanded=None):
    """One `while queue` iteration of the beam search with `injected` records among the candidates.

    Candidates = every successor of the queue (rank order) plus the injected records, stably sorted by link; the first
    arrival of each key not visited wins and is added to `visited` (in place); winners are scored by the oracle and
    stably sorted by score, descending; the first `beam` are the next queue.  Returns (next queue, unique)."""
    cands = expanded if expanded is not None else expand_queue(queue)[0]
    if injected is not None and len(injected):
        cands = np.concatenate([cands, np.asarray(injected, REC_DTYPE)])
    cands = cands[np.argsort(cands['link'], kind='stable')]
    win = []
    for i, (lo, hi) in enumerate(zip(cands['lo'].tolist(), cands['hi'].tolist())):
        k = (lo, hi)
        if k not in visited:
            visited.add(k)
            win.append(i)
    w = cands[np.array(win, dtype=np.int64)]
    st = np.zeros(len(w), oracle.STATE_DTYPE)
    st['lo'], st['hi'], st['aux'] = w['lo'], w['hi'], w['aux']
    sc = oracle.score(st, heuristic, noise)
    assert len(np.unique(sc)) < MAX_SCORES
    nxt = w[np.argsort(-sc, kind='stable')]
    if beam is not None:
        nxt = nxt[:beam]
    return nxt, len(w)


# ---------------------------------------------------------------- runs and their classes (m2_runs / dispatch)
def hash_np(m0, m1):
    """hash_key over uint64 arrays (products wrap mod 2^64)"""
    x = m0 ^ (m1 * np.uint64(GOLDEN))
    x ^= x >> np.uint64(32)
    x *= np.uint64(MIX)
    x ^= x >> np.uint64(32)
    x *= np.uint64(MIX)
    x ^= x >> np.uint64(32)
    return x


def card_words_np(lo, hi):
    lo, hi = np.asarray(lo, np.uint64), np.asarray(hi, np.uint64)
    return (lo >> np.uint64(15)) | (hi << np.uint64(49)), (hi & np.uint64((1 << 41) - 1)) >> np.uint64(15)


THREAD, WARP, CTA = 0, 1, 2


def predict_runs(parents, ntk, recs, warp_max: int = WARP_MAX_UNORDERED):
    """(runs, (thread, warp, cta) counts, {sort key: (class, card sets, items, candidates)}) of one round.  Items =
    the round's parents (ntk gem takes each) then the records as they arrive at the owner, stably sorted by sort key,
    so a run that holds a parent starts with one.  A buy-only run of <= TINY_ITEMS records of one card set is finished
    by the thread kernel; a run of more than warp_max candidates goes to the CTA kernel; every other run, a tiny-sized
    buy-only run of several card sets included, to the warp kernel."""
    m0, m1 = card_words_np(np.concatenate([parents['lo'], recs['lo']]), np.concatenate([parents['hi'], recs['hi']]))
    key = hash_np(m0, m1) >> np.uint64(SORT_SHIFT)
    w = np.concatenate([np.asarray(ntk, np.int64), np.ones(len(recs), np.int64)])
    is_p = np.arange(len(key)) < len(parents)
    uk, inv, cnt = np.unique(key, return_inverse=True, return_counts=True)
    wgt = np.bincount(inv, weights=w, minlength=len(uk)).astype(np.int64)
    has_p = np.bincount(inv, weights=is_p, minlength=len(uk)) > 0
    sets = np.unique(np.stack([inv.astype(np.uint64), m0, m1], axis=1), axis=0)
    n_sets = np.bincount(sets[:, 0].astype(np.int64), minlength=len(uk))
    c = np.where(~has_p & (cnt <= TINY_ITEMS), np.where(n_sets == 1, THREAD, WARP), np.where(wgt <= warp_max, WARP, CTA))
    runs = {int(k): (int(c[i]), int(n_sets[i]), int(cnt[i]), int(wgt[i])) for i, k in enumerate(uk.tolist())}
    return len(uk), tuple(int((c == q).sum()) for q in (THREAD, WARP, CTA)), runs
