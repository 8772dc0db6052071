"""Host side of bidirectional point tracking (CPU only): the shared K1 lists of several groups are split by direction,
so that every shared list has a floor frame next to its query frame."""
from fgvc_b200 import _lib, engine


def _bidirectional_table(T, precede, t0s):
    tb = engine.JobTable()
    for t0 in t0s:
        for t in range(t0 + 1, T):
            mem = engine.memory_frames(t, precede, True, first=t0)
            tb.add(t, mem, mem, t, unmasked=1)
        for t in range(t0 - 1, -1, -1):
            mem = [T - 1 - r for r in engine.memory_frames(T - 1 - t, precede, True, first=T - 1 - t0)]
            tb.add(t, mem, mem, t, unmasked=1)
    return tb


def test_backward_memory_mirrors_the_forward_one():
    T, precede = 12, 3
    tb = _bidirectional_table(T, precede, [7])
    back = [(j[0], [r & ~_lib.MEM_UNMASKED for r in tb.mem_feat[j[1]:j[2]]]) for j in tb.jobs if j[0] < 7]
    assert back[0] == (6, [7, 7]) and back[1] == (5, [7, 7, 6]) and back[-1] == (0, [7, 3, 2, 1])
    assert all(engine.pair_key(tb, j)[1] == (j[0] < 7) for j in tb.jobs)


def test_shared_lists_are_split_by_direction():
    T, precede = 12, 3
    tb = _bidirectional_table(T, precede, (0, 2, 5, 6, 11))
    ut, g, pr = engine.shared_pair_table(tb, None, T)
    keys = [engine.pair_key(ut, j) for j in ut.jobs]
    assert len(set(keys)) == len(keys) == len({engine.pair_key(tb, j) for j in tb.jobs})
    for job in tb.jobs:
        key = engine.pair_key(tb, job)
        for k in range(job[1], job[2]):
            u, i = divmod(pr[k], g)
            assert engine.pair_key(ut, ut.jobs[u]) == key and ut.mem_feat[ut.jobs[u][1] + i] == tb.mem_feat[k]
    # every shared list of a direction has the neighbouring frame in the memory of all of its jobs
    for (q, b, e, _), (_, back) in zip(ut.jobs, keys):
        common = None
        for job in tb.jobs:
            if engine.pair_key(tb, job) == (q, back):
                mem = {r & ~_lib.MEM_UNMASKED for r in tb.mem_feat[job[1]:job[2]]}
                common = mem if common is None else common & mem
        assert (q + 1 if back else q - 1) in common
