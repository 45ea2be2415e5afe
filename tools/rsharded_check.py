"""Realistic mode on the key-sharded driver vs the CPU oracle, level by level, under torchrun:
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/rsharded_check.py --beam 20000
Cases: 2, 3 and 4 players with the market shuffled by seed 0, plus 2 players on the unshuffled market.  Rank 0 runs
oracle.RSolver beside the sharded search and compares frontier, generated, unique, kept, visited, goal_rank and the
sha256 of the queue's records in rank order (links included); it prints one line per level and exits non-zero on the
first mismatch."""
import argparse
import hashlib
import os
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch
import torch.distributed as dist

import oracle
import splendor_rl_gym_b200 as S
from splendor_rl_gym_b200.sharded import Comm, RCudaBackend, RShardedSolver

ap = argparse.ArgumentParser()
ap.add_argument('--beam', type=int, default=20_000)
ap.add_argument('--goal', type=int, default=15)
ap.add_argument('--players', default='2,3,4', help='player counts of the seed-0 cases')
ap.add_argument('--no-unshuffled', action='store_true', help='skip the 2-player case on the unshuffled market')
ap.add_argument('--noise', default='const', choices=['const', 'hash'])
ap.add_argument('--block-parents', type=int, default=0,
                help='parents per block (default: a quarter of the beam over the ranks, i.e. at least 3 rounds per level)')
ap.add_argument('--gloo', action='store_true',
                help='gloo process group with host-staged collectives, ranks sharing the visible GPUs round-robin '
                     '(checks N ranks on fewer than N GPUs; not a multi-GPU timing)')
a = ap.parse_args()

local = int(os.environ.get('LOCAL_RANK', '0')) % (torch.cuda.device_count() if a.gloo else 1 << 30)
torch.cuda.set_device(local)
if int(os.environ.get('WORLD_SIZE', '1')) > 1:
    if a.gloo:
        dist.init_process_group('gloo')
    else:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
eng = S.Engine(local)
comm = Comm(eng.tdev)
block = a.block_parents or max(64, a.beam // (4 * comm.world))
collectives = (f'gloo-host-staged,gpus={torch.cuda.device_count()}' if a.gloo else 'nccl') if comm.on else 'none'
cases = [(int(p), 0) for p in a.players.split(',')] + ([] if a.no_unshuffled else [(2, None)])
failed = False
for players, seed in cases:
    gpc = {2: 4, 3: 5, 4: 7}[players]
    root = S.MultiPlayerState.newgame(S.GameConfig(num_players=players, target_points=a.goal, gems_per_color=gpc,
                                                   infinite_resources=False), shuffle_market=seed is not None, seed=seed)
    rcfg = root.rconfig(a.noise)
    what = f'players={players} seed={seed} beam={a.beam} world={comm.world} block={block} noise={a.noise} collectives={collectives}'
    orc = oracle.RSolver(oracle.make_rconfig(players, a.goal, gpc, [list(x[:rcfg.deck_len[t]]) for t, x in enumerate(rcfg.deck)],
                                             a.noise), a.beam) if comm.rank == 0 else None
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sol = RShardedSolver(RCudaBackend(eng, rcfg, root.record()), comm, a.beam, block_parents=block)
    rounds = 0
    while True:
        gi = sol.step()
        rounds = max(rounds, -(-(-(-gi['frontier'] // block)) // comm.world))
        fr = sol.gather_frontier() if not gi['ended'] else None
        bad = 0
        if comm.rank == 0:
            oi = orc.step()
            fields = ('frontier', 'goal_rank') if gi['ended'] else ('frontier', 'generated', 'unique', 'kept', 'visited', 'goal_rank')
            diff = [f for f in fields if gi[f] != oi[f]]
            got = want = ''
            if not gi['ended']:
                got = hashlib.sha256(fr.cpu().numpy().tobytes()).hexdigest()
                want = hashlib.sha256(orc.level(oi['level'] + 1).tobytes()).hexdigest()
                if got != want:
                    diff.append('sha256')
            print(f"{what} level {gi['level']}: " + ' '.join(f'{f}={gi.get(f)}' for f in fields)
                  + (f' sha={got[:16]}' if got else '') + (' OK' if not diff else f' MISMATCH {diff} oracle={oi} oracle_sha={want[:16]}'),
                  flush=True)
            bad = int(bool(diff))
        t = torch.tensor([bad], device=eng.tdev)
        comm.all_reduce(t, dist.ReduceOp.MAX)
        if int(t):
            failed = True
            break
        if gi['ended']:
            break
    if failed:
        break
    ranks, ords = sol.path()
    dt = time.perf_counter() - t0
    if comm.rank == 0:
        print(f'{what}: {len(ords)} plies, at most {rounds} rounds per level, every level equal to oracle.RSolver '
              f'({dt:.1f} s with the oracle and the checks)', flush=True)
        orc.close()
if comm.on:
    dist.destroy_process_group()
sys.exit(1 if failed else 0)
