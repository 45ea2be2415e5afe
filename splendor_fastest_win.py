#!/usr/bin/env python
"""Fastest-win search for Splendor on a B200: the reference CLI's speedrun flags, GPU path only.

    python splendor_fastest_win.py 15 -u -H aggressive -w 30000000
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 splendor_fastest_win.py 15 -u

Mirrors the flags of the reference's splendor_fastest_win.py:18-83 that concern the solver
(`goal_pts -u -H -w -q`); `--gpu` is accepted for symmetry with the patched reference CLI
(INTEGRATION.md) and is always on here -- this repository has no CPU search.
"""
import argparse
import os
import sys


def cli():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('goal_pts', nargs='?', type=int, help='target amount of points')
    ap.add_argument('-u', '--use_heuristic', action='store_true', help='beam search guided by a heuristic')
    ap.add_argument('-H', '--heuristic', default='simple',
                    choices=['simple', 'balanced', 'aggressive', 'efficiency', 'competitive'])
    ap.add_argument('-w', '--beam_width', type=int, default=300_000)
    ap.add_argument('-q', '--quiet', action='store_true')
    ap.add_argument('--gpu', action='store_true', help='(always on) run the search on the GPU')
    ap.add_argument('--tie', default='stable', choices=['stable', 'det'], help='score tie-break: arrival order | key')
    ap.add_argument('--noise', default='const', choices=['const', 'hash', 'mt'],
                    help="randint noise: deterministic stand-ins, or 'mt' = Python's own seeded stream")
    ap.add_argument('--identity', default='key', choices=['key', 'pyhash'],
                    help="visited-set identity: exact (cards, gems) key | the reference's 64-bit hash((cards, gems))")
    ap.add_argument('--device', type=int, default=None)
    ap.add_argument('--realistic', action='store_true', help='realistic multi-player mode (gem pool, 12 visible cards)')
    ap.add_argument('--players', type=int, default=2, help='number of players for realistic mode')
    ap.add_argument('--shuffle', action='store_true', help='shuffle the card market in realistic mode')
    ap.add_argument('--seed', type=int, default=None, help='market shuffle seed (the reference passes none)')
    ap.add_argument('--shard', action='store_true',
                    help='realistic mode under torchrun: spread one search over the ranks (queue and visited set) '
                         'instead of solving the whole game on every rank')
    if len(sys.argv) == 1:
        ap.print_help()
        ap.exit()
    a = ap.parse_args()
    if not a.goal_pts:
        ap.error('goal_pts is required')
    import torch
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    from splendor_rl_gym_b200 import Color, GameConfig, MultiPlayerState, State
    rank0 = int(os.environ.get('RANK', '0')) == 0
    if a.realistic:  # reference CLI lines 95-129 (under torchrun every rank solves the same game on its own GPU and
        try:          # rank 0 reports; with --shard the ranks share one search)
            cfg = GameConfig(num_players=a.players, target_points=a.goal_pts,
                             gems_per_color={2: 4, 3: 5, 4: 7}.get(a.players, 4), infinite_resources=False)
            solution = MultiPlayerState.newgame(config=cfg, shuffle_market=a.shuffle, seed=a.seed).solve(
                use_heuristic=True, heuristic_name='competitive',
                beam_width=a.beam_width if a.beam_width != 300_000 else 20_000, verbose=not a.quiet and rank0,
                device=local if world > 1 else a.device, shard=a.shard)
            last = solution[-1]
            if rank0:
                print(f'\n{"=" * 60}')
                print(f'Game Over! Winner: Player {last.get_winner()}')
                print('Final Scores:')
                for p in last.players:
                    print(f'  Player {p.player_id}: {p.pts} points, {len(p.cards)} cards')
                print(f'Total moves: {last.turn_number}')
                print(f'{"=" * 60}\n')
        except KeyboardInterrupt:
            print('Execution stopped by the user.')
        finally:
            if world > 1:
                dist.destroy_process_group()
        return
    try:
        solution = State.newgame().solve(goal_pts=a.goal_pts, use_heuristic=a.use_heuristic, heuristic_name=a.heuristic,
                                         beam_width=a.beam_width, verbose=not a.quiet and rank0, tie_policy=a.tie,
                                         noise=a.noise, device=local if world > 1 else a.device, identity=a.identity)
        if rank0:
            print('\nSolution:')
            print(f'({", ".join(c.name.title() for c in Color)}) Cards')
            for state in solution:
                print(state)
    except KeyboardInterrupt:
        print('Execution stopped by the user.')
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == '__main__':
    cli()
