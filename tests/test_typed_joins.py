"""hotloop.captured_early_links: the K4 links of a captured waved step that read their batch-side inputs before
griddepcontrol.wait (host logic, no GPU).  Captured, a link that joins a wave takes it through a full graph edge and the
write-back plan joins the apply, so every link but the first is early -- except under one wave per batch, where the
ordinary joins of ``early_links`` stay."""
from agent0_b200.hotloop import captured_early_links, early_links, wave_plan

F = 84 * 84


def test_the_auto_plan_at_batch_32_runs_every_link_but_the_first_early():
    waves = wave_plan(20, 32, F)                                     # waves of 1, 1, 2, 4, 12 batches
    assert captured_early_links(20, waves) == frozenset(range(1, 20))
    for L, B, spec in ((7, 12, [2, 5]), (6, 32, "auto"), (16, 32, [1, 1, 2, 12]), (20, 32, [1, 1, 1, 2, 3, 12])):
        assert captured_early_links(L, wave_plan(L, B, F, spec)) == frozenset(range(1, L))


def test_one_wave_per_batch_keeps_the_ordinary_joins():
    for L, B, spec in ((20, 512, "auto"), (5, 3, [1, 1, 1, 1, 1]), (2, 32, [1, 1])):
        waves = wave_plan(L, B, F, spec)
        assert captured_early_links(L, waves) == early_links(L, waves) == frozenset()


def test_the_single_gather_launch_leaves_no_link():
    assert captured_early_links(20, wave_plan(20, 32, F, None)) == frozenset()
    assert captured_early_links(20, None) == frozenset()
