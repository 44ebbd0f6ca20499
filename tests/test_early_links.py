"""hotloop.early_links: which K4 links of a waved step may read their batch-side inputs before griddepcontrol.wait
(host logic, no GPU).  Only a link whose sole predecessor is the previous K4 may: never one that joins a gather wave or
the write-back plan, and none when the step gathers with a single launch."""
from agent0_b200.hotloop import early_links, wave_plan

F = 84 * 84


def test_the_auto_plan_at_batch_32_leaves_out_the_wave_joins_and_the_plan_join():
    waves = wave_plan(20, 32, F)                                     # waves of 1, 1, 2, 4, 12 batches
    assert [w[0] for w in waves] == [0, 1, 2, 4, 8]
    assert early_links(20, waves) == frozenset({3, 5, 6, 7} | set(range(9, 20)))
    assert early_links(20, waves, 16) == frozenset({3, 5, 6, 7} | set(range(9, 20))) - {16}


def test_one_wave_per_batch_leaves_no_link():
    assert early_links(20, wave_plan(20, 512, F)) == frozenset()
    assert early_links(5, wave_plan(5, 3, F, [1, 1, 1, 1, 1]), 4) == frozenset()


def test_the_single_gather_launch_leaves_no_link():
    assert early_links(20, wave_plan(20, 32, F, None)) == frozenset()
    assert early_links(20, None, 16) == frozenset()


def test_the_first_link_always_joins():
    for L, B, spec in ((20, 32, "auto"), (7, 12, [2, 5]), (6, 32, "auto"), (16, 32, [1, 1, 2, 12])):
        waves = wave_plan(L, B, F, spec)
        e = early_links(L, waves, L - 1)
        assert 0 not in e and L - 1 not in e
        assert all(0 < k < L for k in e)
        assert all(k not in e for k, _, _, _ in waves)
        assert len(e) == L - len(waves) - 1 + (1 if any(w[0] == L - 1 for w in waves) else 0)
