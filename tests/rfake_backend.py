"""CPU stand-in for sharded.RCudaBackend (realistic mode), used ONLY by the gloo tests of the multi-rank host logic.
Records are restated with the CPU oracle (oracle.r_expand / r_score / r_pts); the visited key is the oracle's identity
bytes (oracle.rident_bytes) padded to 80 bytes, and the owner of a key is a CRC -- deliberately unlike the device's
hash, since results must not depend on who owns which state.  The cut passes are FakeBackend's."""
import zlib

import numpy as np
import torch

import oracle
from fake_backend import FakeBackend

KEY_COLS = 10  # 80 bytes: the identity bytes of up to 4 players (16 B each) + vis (12 B) + cur (1 B), zero padded


def _recs(rows):
    return np.ascontiguousarray(rows.numpy()).view(oracle.RREC_DTYPE).reshape(-1)


def _rows(recs):
    return torch.from_numpy(np.ascontiguousarray(recs).view(np.int64).reshape(-1, 12).copy())


class RFakeBackend(FakeBackend):
    def __init__(self, cfg: oracle.RConfig):
        super().__init__()
        self.cfg = cfg
        self.P = cfg.num_players
        self.noise = {0: 'const', 1: 'hash'}[cfg.noise_mode]
        self.goal = cfg.target_points

    def root_row(self):
        return _rows(oracle.r_root(self.cfg))

    def first_goal(self, front, goal):
        for i, r in enumerate(_recs(front)):
            if oracle.r_pts(r, int(r['cur'])) >= self.goal:
                return i
        return -1

    def expand_rows(self, front, rank_base):
        out = []
        for r, rec in enumerate(_recs(front)):
            kids = oracle.r_expand(self.cfg, rec)
            kids['link'] = [(rank_base + r) << 8 | o for o in range(len(kids))]
            out.append(kids)
        return _rows(np.concatenate(out)) if out else torch.empty((0, 12), dtype=torch.int64)

    def _keys(self, rows):
        out = np.zeros((rows.shape[0], KEY_COLS * 8), np.uint8)
        for i, r in enumerate(_recs(rows)):
            b = oracle.rident_bytes(r, self.P)
            out[i, :len(b)] = np.frombuffer(b, np.uint8)
        return torch.from_numpy(out.view(np.int64).copy())

    def route_keys(self, cand, world):
        keys = self._keys(cand)
        own = np.array([zlib.crc32(k.tobytes()) % world for k in keys.numpy()], dtype=np.int64)
        perm = np.argsort(own, kind='stable')
        self._perm = torch.from_numpy(perm.astype(np.int64))
        return keys[self._perm].contiguous(), np.bincount(own, minlength=world).astype(np.int64)

    def dedup_flags(self, keys):
        flags = torch.zeros(keys.shape[0], dtype=torch.uint8)
        for i, k in enumerate(keys.numpy()):
            b = k.tobytes()
            if b not in self.visited:
                self.visited.add(b)
                flags[i] = 1
        return flags

    def score(self, heuristic, noise, rows, draws=None):
        return torch.from_numpy(oracle.r_score(self.cfg, _recs(rows)))

    def move_rows(self, rows, idx, n_out, scatter):
        if not scatter:
            return rows[idx]
        out = torch.empty((n_out, 12), dtype=torch.int64)
        out[idx] = rows
        return out
