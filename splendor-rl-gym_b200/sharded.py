"""Multi-GPU level-synchronous solver: the frontier is sharded across ranks (one process per GPU),
candidates are routed to the rank that owns their key (hash of the canonical key), and every
level is bit-identical to the single-GPU solver -- same states, same first-arrival `saved` and
parent links, same rank order after the beam cut (SURVEY.md 8e).

Per level (G ranks; the queue is block-distributed by global rank: rank g holds a contiguous slice):
  1. goal test: local first rank with pts >= goal, all-reduce MIN                 (src/solver.py:443)
  2. expand local parents (spl_expand_rows); global arrival index t = exscan(counts) + local index
  3. stable partition of the candidates' keys by owner (spl_route_keys) and all-to-all of the 16-byte KEYS only;
     the receive buffer, concatenated by source rank, is already in global arrival order
  4. owner: first-arrival dedup against its slice of the visited set (spl_dedup_flags)   (:447-450)
  5. one winner byte per candidate travels back (reverse all-to-all); the SOURCE rank, which still
     holds key/aux/link of its candidates in arrival order, compacts its winners (spl_compact_winners) -> the next
     queue is again block-distributed in global arrival order (pure BFS stops here)
  6. beam: scores (spl_score_rows); global radix select = the single-GPU passes with the 2048-bin
     histogram all-reduced between spl_dtopk_hist and spl_dtopk_pick; arrival-order tie quota
     split over ranks by an exclusive scan of local tie counts (stable) or key threshold (det)
  7. local cut + local rank sort (spl_dtopk_cut); global rank of every survivor = local index +
     counts against the other ranks' sorted sort-words (all-gather + spl_count_less); survivors
     are gathered (spl_move_rows) and sent to the rank that owns their global-rank block (all-to-all)  (:452-456)

The compute primitives come from a `backend` object (CudaBackend below wraps the C ABI; RCudaBackend the realistic-mode
calls spl_r*, with which RShardedSolver runs the same levels); the collectives go through torch.distributed (NCCL on
GPUs, gloo in the CPU tests).
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from ._lib import SPL_E_CAPACITY, Key as _Key, check, lib
from .engine import NOISE_IDS, TIE_IDS, Engine, Stepper, _DevArray, heuristic_id

import os
import time

SEL_BITS = 11
I64_MAX = (1 << 63) - 1
TIMING = bool(os.environ.get('SPL_TIMING'))
PHASES = {}


def _tick(name, t0):
    """phase timer (SPL_TIMING=1): synchronises the device, so only for diagnosis"""
    if not TIMING:
        return 0.0
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    PHASES[name] = PHASES.get(name, 0.0) + (t1 - t0)
    return t1


def _bitlen(x: int) -> int:
    return int(x).bit_length()


def _radix_select(comm, top, hist, pick):
    """global radix select over the `top` high bits, SEL_BITS (or the bits left) per pass, most significant first:
    hist(shift, bits, first) -> this rank's histogram of the pass (a device tensor), all-reduced here before
    pick(shift, first) narrows the selection"""
    first = True
    while top > 0:
        bits = min(SEL_BITS, top)
        shift = top - bits
        comm.all_reduce(hist(shift, bits, first), dist.ReduceOp.SUM)
        pick(shift, first)
        first = False
        top = shift


class Comm:
    """Thin wrapper over torch.distributed (world size 1 works without a process group).  Over a gloo process group the
    collectives of device tensors are staged through host memory, so that several ranks can share one GPU (a multi-rank
    check of the device code on a machine with fewer GPUs than ranks; NCCL needs one GPU per rank)."""

    def __init__(self, device):
        self.on = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        self.rank = dist.get_rank() if self.on else 0
        self.world = dist.get_world_size() if self.on else 1
        self.device = device
        self.stage = self.on and device.type == 'cuda' and dist.get_backend() == 'gloo'

    def gather_ints(self, *vals):
        """all_gather of a few python ints -> int64 array [world, len(vals)]"""
        if self.stage:
            t = torch.tensor(vals, dtype=torch.int64).reshape(1, -1)
            out = torch.empty((self.world, t.shape[1]), dtype=torch.int64)
            dist.all_gather(list(out.unbind(0)), t[0])
            return out.numpy()
        t = torch.tensor(vals, dtype=torch.int64, device=self.device).reshape(1, -1)
        if not self.on:
            return t.cpu().numpy()
        out = torch.empty((self.world, t.shape[1]), dtype=torch.int64, device=self.device)
        dist.all_gather_into_tensor(out, t) if self.device.type == 'cuda' else dist.all_gather(list(out.unbind(0)), t[0])
        return out.cpu().numpy()

    def all_reduce(self, t, op):
        if self.stage:
            h = t.cpu()
            dist.all_reduce(h, op=op)
            t.copy_(h)
        elif self.on:
            dist.all_reduce(t, op=op)
        return t

    def all_to_all_rows(self, send, send_counts, recv_counts):
        """variable all-to-all of rows (dim 0); send is grouped by destination rank"""
        if not self.on:
            return send
        src = send.contiguous().cpu() if self.stage else send.contiguous()
        out = torch.empty((int(sum(recv_counts)),) + tuple(send.shape[1:]), dtype=send.dtype, device=src.device)
        dist.all_to_all_single(out, src, [int(x) for x in recv_counts], [int(x) for x in send_counts])
        return out.to(send.device) if self.stage else out

    def all_gather_v(self, t, counts):
        """all_gather of 1-D tensors of different lengths -> list of tensors"""
        if not self.on:
            return [t]
        m = int(max(counts)) if len(counts) else 0
        dev = torch.device('cpu') if self.stage else t.device
        pad = torch.zeros(m, dtype=t.dtype, device=dev)
        pad[:t.shape[0]] = t
        outs = [torch.empty(m, dtype=t.dtype, device=dev) for _ in range(self.world)]
        dist.all_gather(outs, pad)
        return [o[:int(c)].to(t.device) for o, c in zip(outs, counts)]


class _Backend:
    """What the speedrun and realistic backends share: the row layer of a key-sharded round (route keys, dedup flags,
    compact winners, move rows) on rows of ROW_COLS and keys of KEY_COLS int64 columns through the entry points the
    backend names, and the score-generic calls of the global beam cut (distributed radix select, local cut, global
    ranks), which see only scores and sort words."""

    ROW_COLS = KEY_COLS = None
    ROUTE = DEDUP = COMPACT = MOVE = None  # C entry points (ctypes functions: class attributes, not bound methods)
    _route_cfg = ()  # leading arguments of ROUTE after the context (the realistic config)

    def __init__(self, eng: Engine):
        self.eng = eng
        self.device = eng.tdev

    # ---- row layer
    def route_keys(self, cand, world):
        """identity keys [m, KEY_COLS] of the candidates grouped by owner rank (arrival order inside a group) + per-owner
        counts"""
        m = cand.shape[0]
        send = torch.empty((max(m, 1), self.KEY_COLS), dtype=torch.int64, device=self.device)
        counts = (C.c_int64 * world)()
        check(self.ROUTE(self.eng._h, *self._route_cfg, cand.data_ptr(), m, world, send.data_ptr(), counts, self.eng._stream()),
              self.eng._h)
        return send[:m], np.array(counts[:], dtype=np.int64)

    def dedup_flags(self, keys):
        """owner side: one winner byte per received key (first arrival of a never-seen state)"""
        n = keys.shape[0]
        flags = torch.empty(max(n, 1), dtype=torch.uint8, device=self.device)
        check(self.DEDUP(self.eng._h, keys.data_ptr(), n, flags.data_ptr(), self.eng._stream()), self.eng._h)
        return flags[:n]

    def compact_winners(self, cand, flags_send_order):
        """source side: the winning rows in arrival order"""
        m = cand.shape[0]
        out = torch.empty((max(m, 1), self.ROW_COLS), dtype=torch.int64, device=self.device)
        k = C.c_int64()
        check(self.COMPACT(self.eng._h, cand.data_ptr(), m, flags_send_order.data_ptr(), out.data_ptr(), C.byref(k),
                           self.eng._stream()), self.eng._h)
        return out[:k.value]

    def scatter_into(self, dst, rows, pos):
        """dst[pos[i]] = rows[i] (dst is an existing [n, ROW_COLS] int64 tensor)"""
        check(self.MOVE(self.eng._h, rows.contiguous().data_ptr(), pos.contiguous().data_ptr(), pos.shape[0], dst.data_ptr(), 1,
                        self.eng._stream()), self.eng._h)

    def move_rows(self, rows, idx, n_out, scatter):
        """gather (out[i] = rows[idx[i]]) or scatter (out[idx[i]] = rows[i])"""
        out = torch.empty((max(n_out, 1), self.ROW_COLS), dtype=torch.int64, device=self.device)
        check(self.MOVE(self.eng._h, rows.data_ptr(), idx.data_ptr(), idx.shape[0], out.data_ptr(), int(scatter),
                        self.eng._stream()), self.eng._h)
        return out[:n_out]

    # ---- distributed top-k passes
    def dtopk_begin(self, scores, keys):
        a, b = C.c_uint64(), C.c_uint64()
        check(lib.spl_dtopk_begin(self.eng._h, scores.data_ptr(), keys.data_ptr() if keys is not None else None,
                                  scores.shape[0], C.byref(a), C.byref(b), self.eng._stream()), self.eng._h)
        return a.value, b.value

    def dtopk_hist(self, word, shift, bits, first, smin):
        p = C.c_void_p()
        check(lib.spl_dtopk_hist(self.eng._h, word, shift, bits, int(first), smin, C.byref(p), self.eng._stream()), self.eng._h)
        if getattr(self, '_hist_ptr', None) != p.value:  # the histogram lives at a fixed address inside the context
            self._hist_ptr = p.value
            self._hist = torch.as_tensor(_DevArray(p.value, (1 << SEL_BITS,), '<i4'), device=self.device)
        return self._hist

    def dtopk_pick(self, word, shift, first, init_k, k):
        check(lib.spl_dtopk_pick(self.eng._h, word, shift, int(first), int(init_k), k, self.eng._stream()), self.eng._h)

    def dtopk_get(self):
        st = (C.c_uint64 * 6)()
        check(lib.spl_dtopk_get(self.eng._h, st, self.eng._stream()), self.eng._h)
        return list(st)

    def dtopk_set(self, state):
        check(lib.spl_dtopk_set(self.eng._h, (C.c_uint64 * 6)(*state), self.eng._stream()), self.eng._h)

    def dtopk_cut(self, tie, keep_all, all_ties, smin, smax, n):
        det = tie in ('det', 'det_ordered')
        idx = torch.empty(max(n, 1), dtype=torch.int64, device=self.device)
        y = torch.empty(max(n, 1), dtype=torch.int64, device=self.device)
        kl = torch.empty(max(n, 1) if det else 1, dtype=torch.int64, device=self.device)
        kh = torch.empty(max(n, 1) if det else 1, dtype=torch.int64, device=self.device)
        kept = C.c_int64()
        check(lib.spl_dtopk_cut(self.eng._h, TIE_IDS[tie], int(keep_all), int(all_ties), smin, smax, idx.data_ptr(),
                                y.data_ptr(), kl.data_ptr() if det else None, kh.data_ptr() if det else None,
                                C.byref(kept), self.eng._stream()), self.eng._h)
        m = kept.value
        return idx[:m], y[:m], (kl[:m] if det else None), (kh[:m] if det else None)

    def count_less(self, words, inclusive, a, b, out, accumulate, sorted_a=False):
        (ay, akl, akh), (by, bkl, bkh) = a, b
        check(lib.spl_count_less(self.eng._h, words, int(inclusive), ay.data_ptr(),
                                 akl.data_ptr() if words == 3 else None, akh.data_ptr() if words == 3 else None,
                                 ay.shape[0], by.data_ptr(), bkl.data_ptr() if words == 3 else None,
                                 bkh.data_ptr() if words == 3 else None, by.shape[0], out.data_ptr(), int(accumulate),
                                 int(sorted_a), self.eng._stream()), self.eng._h)


class CudaBackend(_Backend):
    """Compute primitives of one rank, all through the C ABI of libsplendor_b200.so: rows are the 32-byte speedrun records
    {lo, hi, aux, link} as int64 [n, 4], keys the 128-bit (cards, gems) as int64 [n, 2]."""

    ROW_COLS, KEY_COLS = 4, 2
    ROUTE, DEDUP, COMPACT, MOVE = lib.spl_route_keys, lib.spl_dedup_flags, lib.spl_compact_winners, lib.spl_move_rows

    def reset_visited(self):
        self.eng.reset_visited()

    def visited_count(self):
        return self.eng.visited_count()

    def first_goal(self, front, goal):
        pts = (front[:, 2] >> 16) & 0xff
        hit = torch.nonzero(pts >= goal)
        return int(hit[0]) if hit.numel() else -1

    def expand_rows(self, front, rank_base):
        """successors of the local queue slice as rows [m, 4]; link = (rank_base + parent) << 8 | ordinal"""
        n = front.shape[0]
        cap = max(64, n * 36)
        while True:
            out = torch.empty((cap, 4), dtype=torch.int64, device=self.device)
            m = C.c_int64()
            rc = lib.spl_expand_rows(self.eng._h, front.data_ptr(), n, rank_base, out.data_ptr(), cap, C.byref(m), self.eng._stream())
            if rc == SPL_E_CAPACITY:
                cap = m.value
                continue
            check(rc, self.eng._h)
            return out[:m.value]

    def ident_rows(self, cand):
        """identity='pyhash': rows whose key is (hash((cards, gems)), 0) -- the reference's own State.hash
        (src/solver.py:316, :335-336) -- so that routing and the owner's visited set work on that value"""
        m = cand.shape[0]
        out = torch.zeros((max(m, 1), 4), dtype=torch.int64, device=self.device)
        if m:
            out[:m, 0] = self.eng.pyhash(cand[:, :2].contiguous())
        return out[:m]

    def owner_partition(self, keys, world):
        n = keys.shape[0]
        perm = torch.empty(max(n, 1), dtype=torch.int64, device=self.device)
        counts = (C.c_int64 * world)()
        check(lib.spl_owner_partition(self.eng._h, keys.data_ptr(), n, world, perm.data_ptr(), counts, self.eng._stream()),
              self.eng._h)
        return perm[:n], np.array(counts[:], dtype=np.int64)

    def score(self, heuristic, noise, rows, draws=None):
        n = rows.shape[0]
        out = torch.empty(n, dtype=torch.float64, device=self.device)
        check(lib.spl_score_rows(self.eng._h, heuristic_id(heuristic), NOISE_IDS[noise], rows.data_ptr(), n, out.data_ptr(),
                                 draws.data_ptr() if draws is not None else None, self.eng._stream()), self.eng._h)
        return out


class ShardedSolver(Stepper):
    """State.solve (src/solver.py:390-464) over a frontier sharded across `comm.world` ranks.

    Queue layout: global rank space [0, N) cut into blocks of `block_parents` ranks; block b lives on rank
    b % G (block-cyclic), so that ROUND r = blocks r*G .. r*G+G-1 covers a contiguous range of global ranks,
    rank 0's block first.  Rounds are processed in order, each bounded in memory; within a round the
    receive buffers are concatenated by source rank -- hence every owner sees candidates in global arrival
    order, and anything inserted by an earlier round is simply "visited" (it arrived earlier).

    Rows are int64 tensors [n, ROW_COLS] with the parent link in column LINK_COL: here the 32-byte speedrun
    records {lo, hi, aux, link}; RShardedSolver runs the same levels on realistic mode's 96-byte records."""

    ROW_COLS, LINK_COL = 4, 3
    TURN_LIMIT = None  # level after which the search stops with the queue it has (realistic mode: 1000)

    def __init__(self, backend, comm: Comm, root_key: int, root_aux: int, goal_pts: int, use_heuristic: bool,
                 heuristic: str, beam_width: int, tie: str = 'stable', noise: str = 'const',
                 block_parents: int = 1 << 22, keep_links: bool = True, identity: str = 'key'):
        if identity not in ('key', 'pyhash'):
            raise ValueError(f'unknown identity {identity!r}')
        self.b, self.comm = backend, comm
        self.identity = identity
        self.goal, self.use_h, self.h, self.beam, self.tie, self.noise = goal_pts, use_heuristic, heuristic, beam_width, tie, noise
        self.C = int(block_parents)
        self.keep_links = keep_links
        root = self._root_row(root_key, root_aux)
        backend.reset_visited()  # trail = {}
        # the root is block 0 (rank 0); its key is registered in the visited set of its owner
        self.front = root if comm.rank == 0 else root[:0]
        self.N = 1
        send, counts = backend.route_keys(self._ident(root), comm.world)
        if counts[comm.rank]:
            backend.dedup_flags(send)
        self.level = 0
        self.ended = False
        self.goal_rank = -1
        self.infos = []
        self._growth = 1.0   # unique / frontier of the previous level (sizes the next queue buffer)
        self.noise_source = None
        if noise == 'mt':
            from .engine import MTNoise
            self.noise_source = MTNoise()
        self.links = []  # per level: local link column (block-cyclic local order)
        self._save_links()

    def _root_row(self, root_key, root_aux):
        m64 = (1 << 64) - 1

        def s64(x):
            x &= m64
            return x - (1 << 64) if x >> 63 else x
        return torch.tensor([[s64(root_key), s64(root_key >> 64), s64(root_aux), -1]], dtype=torch.int64, device=self.b.device)

    def _ident(self, rows):
        """what the visited set compares: the exact (cards, gems) key, or (identity='pyhash') the reference's 64-bit
        State.hash of it -- colliding states then share an owner and merge there, first arrival wins, as in its dict"""
        return rows if self.identity == 'key' else self.b.ident_rows(rows)

    # ------------------------------------------------------------------ block-cyclic layout
    def _local_count(self, n_total, g):
        C, G = self.C, self.comm.world
        nb = -(-n_total // C)                       # number of blocks
        mine = len(range(g, nb, G))                 # blocks owned by g
        if mine == 0:
            return 0
        last_owned = g + (mine - 1) * G
        return (mine - 1) * C + (min(C, n_total - last_owned * C))

    def _global_of_local(self, li, g):
        """global rank of local index li (tensor or int) on rank g"""
        C, G = self.C, self.comm.world
        return ((li // C) * G + g) * C + li % C

    def _locate(self, x):
        C, G = self.C, self.comm.world
        b = x // C
        return b % G, (b // G) * C + x % C

    def _save_links(self):
        self.links.append(self.front[:, self.LINK_COL].clone() if self.keep_links else None)

    def _redistribute(self, rows, x, dst, n_total_after):
        """send rows with global ranks x (tensor) to their block-cyclic owners; scatter into dst (grown as needed)"""
        comm, b, dev = self.comm, self.b, self.b.device
        G, me, C = comm.world, comm.rank, self.C
        blk = x // C
        dest = blk % G
        pos = (blk // G) * C + x % C
        if G > 1:
            send_counts = torch.bincount(dest, minlength=G).cpu().numpy() if x.numel() else np.zeros(G, np.int64)
            # x is ascending, so the rows are already grouped by destination unless they span more than one cycle of G blocks
            if x.numel() and int(blk[-1]) // G != int(blk[0]) // G:
                order = torch.argsort(dest, stable=True)
                rows, pos = b.move_rows(rows, order, order.shape[0], False), pos[order]
            all_counts = comm.gather_ints(*send_counts.tolist())
            recv_counts = all_counts[:, me]
            rows = comm.all_to_all_rows(rows, send_counts, recv_counts)
            pos = comm.all_to_all_rows(pos.contiguous(), send_counts, recv_counts)
        need = self._local_count(n_total_after, me)
        if dst is None or dst.shape[0] < need:
            # first allocation of a level: size it for the growth seen in the previous level (no regrow copies)
            guess = self._local_count(int(self.N * self._growth * 1.08) + 1024, me) if dst is None else 0
            cap = max(need, guess, int(1.5 * (dst.shape[0] if dst is not None else 0)), 1024)
            nd = torch.empty((cap, self.ROW_COLS), dtype=torch.int64, device=dev)
            if dst is not None and self._dst_used:
                nd[:self._dst_used] = dst[:self._dst_used]
            dst = nd
        if rows.shape[0]:
            b.scatter_into(dst, rows, pos)
        self._dst_used = need
        return dst

    # ------------------------------------------------------------------ one `while queue` iteration
    def step(self) -> dict:
        b, comm, dev = self.b, self.comm, self.b.device
        G, me, C = comm.world, comm.rank, self.C
        front, N = self.front, self.N
        n_local = front.shape[0]
        info = dict(level=self.level, ended=0, frontier=N, expanded=0, generated=0, unique=0, kept=0, goal_rank=-1)
        # 1. goal test (src/solver.py:443-445): first state in global queue order with pts >= goal
        g = b.first_goal(front, self.goal) if n_local else -1
        gt = torch.tensor([int(self._global_of_local(g, me)) if g >= 0 else I64_MAX], dtype=torch.int64, device=dev)
        comm.all_reduce(gt, dist.ReduceOp.MIN)
        if int(gt) != I64_MAX:
            self.ended, self.goal_rank = True, int(gt)
            info.update(ended=1, goal_rank=self.goal_rank)
            self.infos.append(info)
            return info
        t0 = _tick('goal', time.perf_counter() if TIMING else 0.0)
        rounds = -(-(-(-N // C)) // G)
        generated = u_total = 0
        pieces, arrivals = [], []
        nxt = None
        self._dst_used = 0
        for r in range(rounds):
            blk = r * G + me
            size = max(0, min(C, N - blk * C))
            parents = front[r * C: r * C + size]
            # 2. expand this rank's block of the round
            cand = b.expand_rows(parents, blk * C) if size else torch.empty((0, self.ROW_COLS), dtype=torch.int64, device=dev)
            m = cand.shape[0]
            t0 = _tick('expand', t0)
            # 3. route keys to their owners
            send_keys, counts = b.route_keys(self._ident(cand), G)
            all_counts = comm.gather_ints(*counts.tolist())  # [src, dst]
            recv_counts = all_counts[:, me]
            t0 = _tick('partition', t0)
            recv_keys = comm.all_to_all_rows(send_keys, counts, recv_counts)
            t0 = _tick('a2a_keys', t0)
            # 4. first-arrival dedup at the owner (receive order == global arrival order inside the round)
            flags_recv = b.dedup_flags(recv_keys)
            t0 = _tick('dedup', t0)
            # 5. winner bytes back to the source; compaction in arrival order
            flags_back = comm.all_to_all_rows(flags_recv, recv_counts, counts)
            winners = b.compact_winners(cand, flags_back)
            t0 = _tick('flags_compact', t0)
            w_all = comm.gather_ints(m, winners.shape[0])
            generated += int(w_all[:, 0].sum())
            abase = u_total + int(w_all[:me, 1].sum())     # global arrival index of my first winner of this round
            u_total += int(w_all[:, 1].sum())
            arr = abase + torch.arange(winners.shape[0], dtype=torch.int64, device=dev)
            if self.use_h:
                pieces.append(winners)
                arrivals.append(arr)
            else:  # pure BFS: the winners ARE the next queue, in arrival order -> place them right away
                nxt = self._redistribute(winners, arr, nxt, u_total)
                t0 = _tick('redistribute', t0)
        info.update(expanded=N, generated=generated, unique=u_total)
        if self.use_h and u_total:
            winners = torch.cat(pieces) if len(pieces) != 1 else pieces[0]
            arr = torch.cat(arrivals) if len(arrivals) != 1 else arrivals[0]
            del pieces, arrivals
            rows, grank, k_total = self._beam_cut(winners, arr, u_total)
            nxt = self._redistribute(rows, grank, None, k_total)
            t0 = _tick('beam_cut', t0)
            n_next = k_total
        else:
            n_next = u_total
        vis = self.comm.gather_ints(b.visited_count())
        info['kept'] = n_next
        info['visited'] = int(vis[:, 0].sum())
        self.infos.append(info)
        if n_next == 0 or (self.TURN_LIMIT is not None and self.level >= self.TURN_LIMIT):
            # frontier exhausted (or the turn limit): `puzzle` stays the last dequeued state
            self.ended, self.goal_rank = True, N - 1
            info['ended'] = 1
            return info
        self._growth = max(1.0, n_next / max(1, N)) if not self.use_h else 1.0
        self.front = nxt[:self._local_count(n_next, me)]
        self.N = n_next
        self.level += 1
        self._save_links()
        return info

    # ------------------------------------------------------------------ global beam cut + global ranks
    def _beam_cut(self, winners, arr, u_total):
        """-> (surviving local rows in local rank order, their global ranks, global survivor count).
        Tie policy `stable` (arrival order) runs through the same key machinery as `det` with the synthetic
        key (u_total - global arrival index): larger key == earlier arrival."""
        b, comm, dev = self.b, self.comm, self.b.device
        G, me = comm.world, comm.rank
        K = self.beam
        u_local = winners.shape[0]
        draws = None
        if self.noise == 'mt':
            # every rank replays the same seeded stream (src/solver.py:215 etc.): the state with global arrival
            # index a is the a-th one the reference's sorted(..., key=heuristic) would have scored in this level
            level_draws = torch.from_numpy(self.noise_source.draw(u_total)).to(dev)
            draws = level_draws[arr].contiguous()
        scores = b.score(self.h, self.noise, winners, draws) if u_local else torch.empty(0, dtype=torch.float64, device=dev)
        if self.tie == 'det':
            keys = winners[:, :2].contiguous()
        else:
            keys = torch.stack([u_total - arr, torch.zeros_like(arr)], dim=1).contiguous()
        t0 = _tick('bc_score_keys', time.perf_counter() if TIMING else 0.0)
        smin, smax = b.dtopk_begin(scores, keys)
        t0 = _tick('bc_begin', t0)
        allr = comm.gather_ints(smin >> 32, smin & 0xffffffff, smax >> 32, smax & 0xffffffff, u_local)
        mins = [(int(r[0]) << 32) | int(r[1]) for r in allr if r[4]]
        maxs = [(int(r[2]) << 32) | int(r[3]) for r in allr if r[4]]
        smin, smax = min(mins), max(maxs)
        keep_all = u_total <= K
        all_ties = True
        if not keep_all:
            nbits = _bitlen(smax - smin)
            b.dtopk_set([0, K, 0, u_total, 0, 0])
            _radix_select(comm, nbits, lambda shift, bits, first: b.dtopk_hist(0, shift, bits, first, smin),
                          lambda shift, first: b.dtopk_pick(0, shift, first, first, K))
            state = b.dtopk_get()
            quota, tie_count = state[1], state[3]
            if quota < tie_count:  # split the score ties by key (det) / by arrival (stable, synthetic key)
                all_ties = False
                # synthetic arrival keys are < 2^bitlen(u_total) with a zero high word: skip the constant digits
                for word, wbits in (((1, 41), (2, 64)) if self.tie == 'det' else ((2, _bitlen(u_total)),)):
                    _radix_select(comm, wbits, lambda shift, bits, first: b.dtopk_hist(word, shift, bits, first, smin),
                                  lambda shift, first: b.dtopk_pick(word, shift, first, False, K))
        t0 = _tick('bc_select', t0)
        # stable: the synthetic arrival keys fall with the local index, so the local sort only needs the score
        idx, y, kl, kh = b.dtopk_cut('det' if self.tie == 'det' else 'det_ordered', keep_all, all_ties, smin, smax, u_local)
        t0 = _tick('bc_cut_sort', t0)
        # global rank of every local survivor: local index + #smaller composites on the other ranks
        k_local = idx.shape[0]
        k_all = comm.gather_ints(k_local)[:, 0]
        k_total = int(k_all.sum())
        grank = torch.arange(k_local, dtype=torch.int64, device=dev)
        if G > 1:
            # one all-gather of the three sort words (rows of a [3, k] block), then one ranked search per peer
            packed = comm.all_gather_v(torch.stack([y, kl, kh]).t().contiguous().reshape(-1), k_all * 3)
            for g in range(G):
                if g == me or k_all[g] == 0 or k_local == 0:
                    continue
                other = packed[g].reshape(-1, 3).t().contiguous()
                b.count_less(3, False, (y, kl, kh), (other[0], other[1], other[2]), grank, True, True)
        t0 = _tick('bc_ranks', t0)
        out = b.move_rows(winners, idx, k_local, False)
        _tick('bc_gather', t0)
        return out, grank, k_total

    # ------------------------------------------------------------------ driver helpers
    def path(self):
        """(ranks, ordinals) of the winning line, walking the distributed link columns (src/solver.py:459-464)."""
        dev = self.b.device
        L = self.level
        r = self.goal_rank
        ranks, ords = [0] * (L + 1), [0] * L
        for lv in range(L, -1, -1):
            ranks[lv] = r
            if lv > 0:
                owner, li = self._locate(r)
                t = torch.zeros(1, dtype=torch.int64, device=dev)
                if owner == self.comm.rank:
                    t[0] = self.links[lv][li]
                self.comm.all_reduce(t, dist.ReduceOp.SUM)
                link = int(t)
                ords[lv - 1] = link & 0xff
                r = link >> 8
        return ranks, ords

    def gather_frontier(self):
        """the whole current queue on every rank, in global rank order (tests / small cases only)"""
        G, dev = self.comm.world, self.b.device
        sizes = [self._local_count(self.N, g) for g in range(G)]
        out = torch.empty((self.N, self.ROW_COLS), dtype=torch.int64, device=dev)
        cols = [self.comm.all_gather_v(self.front[:, c].contiguous(), sizes) for c in range(self.ROW_COLS)]
        for g in range(G):
            if sizes[g]:
                x = self._global_of_local(torch.arange(sizes[g], dtype=torch.int64, device=dev), g)
                out[x] = torch.stack([cols[c][g] for c in range(self.ROW_COLS)], dim=1)
        return out


class RCudaBackend(_Backend):
    """Compute primitives of one rank for realistic mode (MultiPlayerState, csrc/spl_realistic.cuh), with the method
    names of CudaBackend.  Rows are 96-byte records as int64 [n, 12]: players in columns 0-7, vis/cur in 8-9, link in
    10, spare in 11; keys are the 384-bit exact identity (spl_rpack) as int64 [n, 6].  Scores come from spl_rscore
    with the config's noise (`const` or `hash`); `root` is the record the search starts from (default: the config's
    new game)."""

    ROW_COLS, KEY_COLS = 12, 6
    ROUTE, DEDUP, COMPACT, MOVE = lib.spl_rroute_keys, lib.spl_rdedup_flags, lib.spl_rcompact_winners, lib.spl_rmove_rows

    def __init__(self, eng: Engine, rcfg, root=None):
        super().__init__(eng)
        self.rcfg = rcfg
        self._route_cfg = (C.byref(rcfg),)
        self.noise = {v: k for k, v in NOISE_IDS.items()}[rcfg.noise]
        self.goal = rcfg.target_points
        self._fanout = 27.0  # successors per parent the next expand_rows allocates for
        if root is None:
            from .realistic import RREC_DTYPE
            root = np.zeros(1, RREC_DTYPE)
            root['vis'][0] = [rcfg.deck[t][k] if k < rcfg.deck_len[t] else 255 for t in range(3) for k in range(4)]
            root['link'] = (1 << 64) - 1
        self.root = np.ascontiguousarray(root).reshape(-1)[:1].copy()

    def root_row(self):
        return torch.from_numpy(self.root.view(np.int64).reshape(1, 12).copy()).to(self.device)

    def reset_visited(self):
        check(lib.spl_rreset_visited(self.eng._h, self.eng._stream()), self.eng._h)

    def visited_count(self):
        n = C.c_int64()
        check(lib.spl_rvisited_count(self.eng._h, C.byref(n)), self.eng._h)
        return n.value

    def first_goal(self, front, goal):
        """first queue index whose game is over (players[cur].pts >= the config's target), -1 if none"""
        r = C.c_int64()
        check(lib.spl_rfirst_goal(self.eng._h, C.byref(self.rcfg), front.data_ptr(), front.shape[0], C.byref(r),
                                  self.eng._stream()), self.eng._h)
        return r.value

    def expand_rows(self, front, rank_base):
        """successors of the local queue slice as rows [m, 12]; link = (rank_base + parent) << 8 | ordinal.  The buffer is
        sized from the successors per parent of the previous call (at most 27: 12 buys, 10 colour triples, 5 double
        takes) rather than the worst case, so that device memory stays free for the visited table; when it is too small
        the call reports the exact count and runs again."""
        n = front.shape[0]
        cap = max(64, int(n * self._fanout) + 1024)
        while True:
            out = torch.empty((cap, 12), dtype=torch.int64, device=self.device)
            m = C.c_int64()
            rc = lib.spl_rexpand_rows(self.eng._h, C.byref(self.rcfg), front.data_ptr(), n, rank_base, out.data_ptr(), cap,
                                      C.byref(m), self.eng._stream())
            if rc == SPL_E_CAPACITY:
                cap = m.value
                continue
            check(rc, self.eng._h)
            if n:
                self._fanout = min(27.0, 1.1 * m.value / n)
            return out[:m.value]

    def score(self, heuristic, noise, rows, draws=None):
        """multi_competitive_heuristic of every row (the config's noise; `heuristic` is the reference's ignored name)"""
        n = rows.shape[0]
        out = torch.empty(n, dtype=torch.float64, device=self.device)
        check(lib.spl_rscore(self.eng._h, C.byref(self.rcfg), rows.data_ptr(), n, out.data_ptr(), self.eng._stream()), self.eng._h)
        return out


class RShardedSolver(ShardedSolver):
    """MultiPlayerState.solve (src/solver.py:750-860) on the key-sharded choreography of ShardedSolver: 96-byte records,
    the exact 384-bit identity as the routing and visited key, the beam always applied, score ties by arrival order (the
    reference's stable sort; it has no key tie-break), noise `const` or `hash` from the backend's config.  Every level
    holds the same records, in the same order, with the same links, as the single-GPU realistic solver (spl_rsolver).
    `backend` is an RCudaBackend (or a stand-in with its methods and `root_row`, `noise`, `goal`)."""

    ROW_COLS, LINK_COL = 12, 10
    TURN_LIMIT = 1000  # the reference leaves its loop after the iteration with turn == 1000 (src/solver.py:846-852)

    def __init__(self, backend, comm: Comm, beam_width: int, tie: str = 'stable', block_parents: int = 1 << 20,
                 keep_links: bool = True, identity: str = 'key'):
        if tie != 'stable':
            raise ValueError(f"realistic mode breaks score ties by arrival order only (tie='stable'), not {tie!r}")
        if identity != 'key':
            raise ValueError(f"realistic mode dedups on its exact identity key only (identity='key'), not {identity!r}")
        if backend.noise not in ('const', 'hash'):
            raise ValueError(f"the sharded realistic search supports noise 'const' and 'hash', not {backend.noise!r}")
        super().__init__(backend, comm, 0, 0, backend.goal, True, 'competitive', beam_width, tie, backend.noise,
                         block_parents=block_parents, keep_links=keep_links, identity=identity)

    def _root_row(self, root_key, root_aux):
        return self.b.root_row()


class DictionaryOverflow(RuntimeError):
    """A level holds more distinct scores than the score dictionary of the card-set-sharded beam cut (2048; `balanced`
    and `efficiency` at wide beams): the caller reruns the search on ShardedSolver, whose cut is a radix select.  The
    merged dictionary is the same on every rank, so every rank raises at the same level."""


class PeerRecv:
    """This rank's receive buffer for routed buy records, mapped into every other rank of the node (CUDA IPC through
    spl_ipc_*): the routing kernel of rank r stores the records owned by rank d straight into d's buffer over NVLink
    (spl_gs_round_buys_peer), so a round has no send buffer and no all-to-all.  One buffer per Engine, grown
    collectively (every rank sees the same gathered counts, hence takes the same decision)."""

    def __init__(self, eng: Engine, comm: Comm):
        self.eng, self.comm = eng, comm
        self.cap = 0            # records (32 B)
        self.local = None       # this rank's buffer
        self.ptrs = None        # ptrs[d]: rank d's buffer as mapped here

    def _fence(self):
        torch.cuda.synchronize(self.eng.tdev)
        self.comm.all_reduce(torch.zeros(1, dtype=torch.int64, device=self.eng.tdev), dist.ReduceOp.SUM)
        torch.cuda.synchronize(self.eng.tdev)

    def release(self):
        if self.local is None:
            return
        for g, p in enumerate(self.ptrs):
            if g != self.comm.rank:
                check(lib.spl_ipc_close(self.eng._h, C.c_void_p(p)), self.eng._h)
        self._fence()  # nobody maps the buffer any more
        check(lib.spl_ipc_free(self.eng._h, C.c_void_p(self.local)), self.eng._h)
        self.local, self.ptrs, self.cap = None, None, 0

    def ensure(self, records: int):
        """collective: every rank passes the same number"""
        if self.local is not None and records <= self.cap:
            return
        self.release()
        cap = max(int(records * 1.25), 1 << 20)
        ptr, handle = C.c_void_p(), (C.c_uint8 * 64)()
        check(lib.spl_ipc_alloc(self.eng._h, cap * 32, C.byref(ptr), handle), self.eng._h)
        words = np.frombuffer(bytes(handle), dtype=np.int64)
        allh = self.comm.gather_ints(*[int(x) for x in words])  # [rank, 8]
        ptrs = []
        for g in range(self.comm.world):
            if g == self.comm.rank:
                ptrs.append(ptr.value)
                continue
            hb = (C.c_uint8 * 64).from_buffer_copy(np.ascontiguousarray(allh[g], dtype=np.int64).tobytes())
            pp = C.c_void_p()
            check(lib.spl_ipc_open(self.eng._h, hb, C.byref(pp)), self.eng._h)
            ptrs.append(pp.value)
        self.local, self.ptrs, self.cap = ptr.value, ptrs, cap
        self._fence()  # every mapping exists before anyone stores through one


class GroupedShardedSolver(Stepper):
    """Beam search of State.solve (src/solver.py:390-464) over a queue sharded BY CARD SET (spl_gs_* entry points,
    csrc/spl_shard.cuh): a queue state lives on the rank that owns its cards, so its gem-take successors are
    deduplicated on the generating GPU by the fused on-chip walk and only card buys travel (32-byte records, one
    all-to-all per round).  The beam cut is global: the ranks' score dictionaries are all-gathered and merged into one
    threshold, score ties at the threshold are split by arrival order with all-reduced radix histograms, and the
    survivors get their dense global ranks -- the queue order of the next level -- from a sample sort of their sort
    words (score rank, arrival index).  Every level is the same set of states, in the same order, as on one GPU.

    Policy: ties by arrival order (`stable`), noise `const` (the score dictionary needs few distinct scores);
    anything else runs on ShardedSolver."""

    SAMPLES = 256

    def __init__(self, eng: Engine, comm: Comm, root_key: int, root_aux: int, goal_pts: int, heuristic: str, beam_width: int,
                 noise: str = 'const', round_parents: int = 1 << 27, keep_links: bool = True):
        self.eng, self.comm = eng, comm
        self.goal, self.h, self.beam, self.noise = goal_pts, heuristic, beam_width, noise
        self.C = int(round_parents)   # global ranks per round (all ranks walk the same window of the queue)
        k = _Key(root_key & ((1 << 64) - 1), root_key >> 64)
        h = C.c_void_p()
        check(lib.spl_gs_create(eng._h, comm.rank, comm.world, C.byref(k), root_aux, goal_pts, heuristic_id(heuristic), beam_width,
                                NOISE_IDS[noise], int(keep_links), C.byref(h)), eng._h)
        self._h = h
        self.N = 1
        self.level = 0
        self.ended = False
        self.goal_rank = -1
        self.infos = []
        self.noise_source = None
        # buy records go to their owners by peer stores from the routing kernel (SPL_NO_P2P=1: send buffer + NCCL all-to-all)
        self.peer = None
        if comm.on and not os.environ.get('SPL_NO_P2P'):
            if getattr(eng, '_peer_recv', None) is None:
                eng._peer_recv = PeerRecv(eng, comm)
            self.peer = eng._peer_recv

    def close(self):
        if getattr(self, '_h', None):
            lib.spl_gs_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---------------------------------------------------------------- helpers
    def _st(self):
        return self.eng._stream()

    def _sum_ints(self, *vals):
        a = self.comm.gather_ints(*vals)
        return [int(x) for x in a.sum(axis=0)]

    def _dev(self, ptr, shape, typestr='<i8'):
        return torch.as_tensor(_DevArray(ptr, shape, typestr), device=self.eng.tdev)

    def _tie_hist(self, shift, bits, first):
        hp = C.c_void_p()
        check(lib.spl_gs_tie_hist(self._h, shift, bits, int(first), C.byref(hp), self._st()), self.eng._h)
        return self._dev(hp.value, (1 << SEL_BITS,), '<i4')

    # ---------------------------------------------------------------- one `while queue` iteration
    def step(self) -> dict:
        eng, comm, dev = self.eng, self.comm, self.eng.tdev
        G, me = comm.world, comm.rank
        N = self.N
        info = dict(level=self.level, ended=0, frontier=N, expanded=0, generated=0, unique=0, kept=0, goal_rank=-1)
        # 1. goal test (src/solver.py:443-445): first state in global queue order with pts >= goal
        t0 = _tick('', time.perf_counter() if TIMING else 0.0)
        gr, nl = C.c_int64(), C.c_int64()
        check(lib.spl_gs_goal(self._h, C.byref(gr), C.byref(nl), self._st()), eng._h)
        gt = torch.tensor([gr.value], dtype=torch.int64, device=dev)
        comm.all_reduce(gt, dist.ReduceOp.MIN)
        if int(gt) != I64_MAX:
            self.ended, self.goal_rank = True, int(gt)
            info.update(ended=1, goal_rank=self.goal_rank)
            self.infos.append(info)
            return info
        t0 = _tick('goal', t0)
        # 2. rounds over windows of the global queue
        for lo in range(0, N, self.C):
            counts = (C.c_int64 * G)()
            npar = C.c_int64()
            check(lib.spl_gs_round_begin(self._h, lo, min(lo + self.C, N), counts, C.byref(npar), self._st()), eng._h)
            counts = np.array(counts[:], dtype=np.int64)
            t0 = _tick('count', t0)
            allc = comm.gather_ints(*counts.tolist())          # [src, dst]
            n_new = C.c_int64()
            if self.peer is not None:
                # every rank has finished reading the previous round's records (its counts above came after a stream
                # sync); the routing kernel stores each record into its owner's buffer, rank-major as an all-to-all would
                self.peer.ensure(int(allc.sum(axis=0).max()))
                n_recv = int(allc[:, me].sum())
                offs = (C.c_int64 * G)(*[int(x) for x in allc[:me].sum(axis=0)])
                ptrs = (C.c_void_p * G)(*self.peer.ptrs)
                check(lib.spl_gs_round_buys_peer(self._h, ptrs, offs, self._st()), eng._h)
                t0 = _tick('buys', t0)
                comm.all_reduce(torch.zeros(1, dtype=torch.int64, device=dev), dist.ReduceOp.SUM)  # all stores have landed
                t0 = _tick('a2a', t0)
                check(lib.spl_gs_round_group(self._h, C.c_void_p(self.peer.local) if n_recv else None, n_recv, C.byref(n_new), self._st()), eng._h)
            else:
                send = torch.empty((max(int(counts.sum()), 1), 4), dtype=torch.int64, device=dev)
                check(lib.spl_gs_round_buys(self._h, send.data_ptr(), self._st()), eng._h)
                t0 = _tick('buys', t0)
                recv = comm.all_to_all_rows(send[:int(counts.sum())], counts, allc[:, me])
                t0 = _tick('a2a', t0)
                check(lib.spl_gs_round_group(self._h, recv.data_ptr() if recv.shape[0] else None, recv.shape[0], C.byref(n_new), self._st()), eng._h)
                del send, recv
            t0 = _tick('group', t0)
        nu, gen, vis = C.c_int64(), C.c_int64(), C.c_int64()
        check(lib.spl_gs_counters(self._h, C.byref(nu), C.byref(gen), C.byref(vis)), eng._h)
        u_total, g_total, v_total = self._sum_ints(nu.value, gen.value, vis.value)
        ms = (C.c_float * 4)()
        check(lib.spl_gs_stage_ms(self._h, ms), eng._h)
        info.update(expanded=N, generated=g_total, unique=u_total, visited=v_total, local_unique=nu.value,
                    ms_sort=ms[0], ms_thread=ms[1], ms_warp=ms[2], ms_cta=ms[3])
        if u_total == 0:  # frontier exhausted: `puzzle` stays the last dequeued state
            self.ended, self.goal_rank = True, N - 1
            info['ended'] = 1
            self.infos.append(info)
            return info
        # 3. global beam threshold from the merged score dictionaries
        dp, nbytes = C.c_void_p(), C.c_int64()
        check(lib.spl_gs_dict(self._h, C.byref(dp), C.byref(nbytes), self._st()), eng._h)
        local = self._dev(dp.value, (nbytes.value,), '|u1')
        if comm.on:
            alld = torch.empty((G, nbytes.value), dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(alld, local.reshape(1, -1))
        else:
            alld = local.reshape(1, -1)
        need = C.c_int32()
        rc = lib.spl_gs_threshold(self._h, alld.data_ptr(), self.beam, u_total, C.byref(need), self._st())
        if rc == -6:  # SPL_E_CAPACITY
            raise DictionaryOverflow(f'level {self.level}: more than 2048 distinct scores')
        check(rc, eng._h)
        if need.value:  # split the ties of the threshold score by arrival order
            lt = C.c_int32()
            check(lib.spl_gs_tie_begin(self._h, C.byref(lt), self._st()), eng._h)
            _radix_select(comm, lt.value, self._tie_hist, lambda shift, first: check(lib.spl_gs_tie_pick(self._h, shift, int(first), self._st()), eng._h))
        kept, yp, ybits = C.c_int64(), C.c_void_p(), C.c_int32()
        t0 = _tick('threshold', t0)
        check(lib.spl_gs_cut(self._h, need.value, C.byref(kept), C.byref(yp), C.byref(ybits), self._st()), eng._h)
        t0 = _tick('cut', t0)
        k_local = kept.value
        k_all = comm.gather_ints(k_local)[:, 0]
        k_total = int(k_all.sum())
        assert k_total == min(u_total, self.beam), (k_total, u_total, self.beam)
        # 4. dense global ranks of the survivors: sample sort of the sort words
        granks = self._global_ranks(yp.value, k_local, ybits.value, k_total)
        t0 = _tick('ranks', t0)
        check(lib.spl_gs_adopt(self._h, granks.data_ptr() if k_local else None, k_total, self._st()), eng._h)
        t0 = _tick('adopt', t0)
        info['kept'] = k_total
        self.infos.append(info)
        self.N = k_total
        self.level += 1
        return info

    def _global_ranks(self, y_ptr, k_local, y_bits, k_total):
        eng, comm, dev = self.eng, self.comm, self.eng.tdev
        G, me = comm.world, comm.rank
        if G == 1:
            return torch.arange(k_local, dtype=torch.int64, device=dev)
        y = self._dev(y_ptr, (k_local,)) if k_local else torch.empty(0, dtype=torch.int64, device=dev)
        # splitters: regular samples of every rank's sorted words -> G - 1 quantiles of their union
        S = self.SAMPLES
        smp = torch.full((S,), I64_MAX, dtype=torch.int64, device=dev)
        if k_local:
            m = min(S, k_local)
            pick = (torch.arange(m, dtype=torch.int64, device=dev) * (k_local - 1)) // max(m - 1, 1)  # exact integer positions
            smp[:m] = y[pick]
        alls = torch.empty((G, S), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(alls, smp.reshape(1, -1))
        alls = np.sort(alls.cpu().numpy().reshape(-1))
        alls = alls[alls != I64_MAX]
        if len(alls):
            spl = [int(alls[min(len(alls) - 1, (g * len(alls)) // G)]) for g in range(1, G)]
        else:
            spl = [0] * (G - 1)
        bounds = (C.c_int64 * (G - 1))()
        check(lib.spl_gs_partition(self._h, (C.c_uint64 * (G - 1))(*spl), G - 1, bounds, self._st()), eng._h)
        b = [0] + [int(x) for x in bounds[:]] + [k_local]
        send_counts = np.diff(np.array(b, dtype=np.int64))
        allc = comm.gather_ints(*send_counts.tolist())            # [src, dst]
        recv_counts = allc[:, me]
        recv_y = comm.all_to_all_rows(y, send_counts, recv_counts)
        base = int(allc[:, :me].sum())                              # sort words held by the ranks below this one
        n_recv = int(recv_counts.sum())
        ranks_recv = torch.empty(max(n_recv, 1), dtype=torch.int64, device=dev)
        check(lib.spl_gs_rank_sort(self._h, recv_y.data_ptr() if n_recv else None, n_recv, y_bits, base, ranks_recv.data_ptr(), self._st()), eng._h)
        return comm.all_to_all_rows(ranks_recv[:n_recv], recv_counts, send_counts)

    def frontier_local(self):
        """(records [n, 4] int64, global ranks [n] int64) of this rank's share of the queue (device views)"""
        rp, gp, n = C.c_void_p(), C.c_void_p(), C.c_int64()
        check(lib.spl_gs_frontier(self._h, C.byref(rp), C.byref(gp), C.byref(n)), self.eng._h)
        if n.value == 0:
            z = torch.empty((0, 4), dtype=torch.int64, device=self.eng.tdev)
            return z, z[:, 0]
        return self._dev(rp.value, (n.value, 4)), self._dev(gp.value, (n.value,))

    def gather_frontier(self):
        """the whole queue in global rank order on every rank (tests / parity digests; small cases only)"""
        recs, gr = self.frontier_local()
        out = torch.zeros((self.N, 4), dtype=torch.int64, device=self.eng.tdev)
        if recs.shape[0]:
            out[gr] = recs
        self.comm.all_reduce(out, dist.ReduceOp.SUM)
        return out

    def path(self):
        """(ranks, ordinals) of the winning line: walk the per-level link columns, each held by the rank that owns
        the state's cards (src/solver.py:459-464)."""
        L, r = self.level, self.goal_rank
        ranks, ords = [0] * (L + 1), [0] * L
        for lv in range(L, -1, -1):
            ranks[lv] = r
            if lv > 0:
                found, link = C.c_int32(), C.c_uint64()
                check(lib.spl_gs_link_at(self._h, lv, r, C.byref(found), C.byref(link)), self.eng._h)
                t = torch.tensor([link.value if found.value else 0, found.value], dtype=torch.int64, device=self.eng.tdev)
                self.comm.all_reduce(t, dist.ReduceOp.SUM)
                assert int(t[1]) == 1, f'state of rank {r} in level {lv} is held by {int(t[1])} ranks'
                ords[lv - 1] = int(t[0]) & 0xff
                r = int(t[0]) >> 8
        return ranks, ords
