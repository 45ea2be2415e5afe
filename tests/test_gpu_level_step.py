"""Visited tables of the single-GPU solver (-m gpu): each one counts its own entries."""
import pytest

import splendor_rl_gym_b200 as S

pytestmark = pytest.mark.gpu


def test_dedup_after_grouped_solve_sizes_the_key_table_by_its_own_entries():
    """A grouped beam search keeps its visited set in the card-set node table.  Engine.dedup after it, without a reset,
    sizes the key table by what the key table holds: it fits a small max_table_bytes although the search visited more
    states than that table has slots, and it still adds its new states to the visited count."""
    eng = S.Engine(0, max_table_bytes=1 << 20)  # key table: 16 384 buckets = 49 152 slots, and no room to grow
    try:
        k, a = S.State.newgame().record()
        sol = eng.solver(k, a, 15, True, 'aggressive', 20_000, 'stable', 'const')
        infos = sol.run()
        assert infos[-1]['ended']
        fr = sol.frontier()[:300].clone()
        sol.close()
        visited = eng.visited_count()
        assert visited > 49_152 and fr.shape[0] == 300
        uk, ua, _ = eng.dedup(fr[:, :2].contiguous(), fr[:, 2].contiguous())
        assert uk.shape[0] == 300  # the queue's states were never in the key table
        assert eng.visited_count() == visited + 300
        assert eng.dedup(fr[:, :2].contiguous(), fr[:, 2].contiguous())[0].shape[0] == 0
    finally:
        eng.close()
