"""Host side of the cycle-consistency occlusion flags (test_cfg.cycle_occlusion, CPU only): the job table of the
checks, the K1 list sharing with them, and the key's validation."""
import pytest

from fgvc_b200 import _lib, engine


def _tables(T, precede, t0s, frames, bidirectional=True, with_first=True, unmasked=lambda mem: 0):
    table, spans = engine.query_job_table(t0s, T, precede, with_first, bidirectional, unmasked)
    n_track = len(table)
    checks = engine.cycle_job_table(table, spans, T, precede, with_first, bidirectional, frames, unmasked)
    return table, spans, n_track, checks


def _feat(table, j):
    return [r & ~_lib.MEM_UNMASKED for r in table.mem_feat[table.jobs[j][1]:table.jobs[j][2]]]


@pytest.mark.parametrize("frames", [1, 3, None])
@pytest.mark.parametrize("bidirectional", [True, False])
@pytest.mark.parametrize("with_first", [True, False])
def test_check_jobs_are_the_tracking_jobs_of_a_group_queried_at_t(frames, bidirectional, with_first):
    T, precede = 11, 3
    t0s = (0, 4, T - 1)
    unmasked = lambda mem: 1                                                   # noqa: E731
    table, spans, n_track, checks = _tables(T, precede, t0s, frames, bidirectional, with_first, unmasked)
    before, _ = engine.query_job_table(t0s, T, precede, with_first, bidirectional, unmasked)
    assert table.jobs[:n_track] == before.jobs and table.mem_feat[:len(before.mem_feat)] == before.mem_feat
    want = {(t0s.index(t0), t) for t0 in t0s for t in range(T) if t > t0 or (bidirectional and t < t0)}
    assert {(g, t) for g, t, *_ in checks} == want
    lengths = [je - jb for *_, jb, je in checks]
    assert lengths == sorted(lengths, reverse=True)
    for g, t, s, jb, je in checks:
        t0 = t0s[g]
        assert s == (t0 if frames is None else (max(t0, t - frames) if t > t0 else min(t0, t + frames)))
        assert je - jb == abs(t - s) >= 1
        ref, rspans = engine.query_job_table([t], T, precede, with_first, True, unmasked)
        step = 1 if s > t else -1
        for k, j in enumerate(range(jb, je)):
            q, b, e, out = table.jobs[j]
            assert q == t + step * (k + 1) and out == k + 1
            r = next(i for i, job in enumerate(ref.jobs) if job[0] == q)    # the one job of the group at t for frame q
            assert table.mem_feat[b:e] == ref.mem_feat[ref.jobs[r][1]:ref.jobs[r][2]]
            # label slots of the check's own bank: slot 0 = frame t, slot k = the frame of its k-th job
            assert table.mem_label[b:e] == [abs(f - t) for f in _feat(table, j)]
            assert all(0 <= x < k + 1 for x in table.mem_label[b:e])


def test_short_checks_add_no_list_to_a_query_frame_the_tracks_already_score():
    """frames <= precede_frames: a check's memory lies in the window of the tracking jobs of its query frame and
    direction, except after the last query frame minus precede_frames, where no backward tracking window reaches the
    frames the checks start from"""
    T, precede = 50, 5
    t0s = tuple(range(0, T, 5))
    for frames in (1, 3, 5):
        table, spans, n_track, checks = _tables(T, precede, t0s, frames)
        track_pairs, pairs = set(), set()
        for j, job in enumerate(table.jobs):
            key = engine.pair_key(table, job)
            for r in table.mem_feat[job[1]:job[2]]:
                (track_pairs if j < n_track else pairs).add((key, r))
        extra = {p for p in pairs if p not in track_pairs}
        assert extra and all(back and q > t0s[-1] - precede for ((q, back), _) in extra), (frames, extra)


@pytest.mark.parametrize("frames", [1, 5, None])
def test_sharing_is_decided_by_the_tracking_jobs(frames):
    T, precede = 50, 5
    t0s = tuple(range(0, T, 5))
    table, spans, n_track, checks = _tables(T, precede, t0s, frames)
    track, _ = engine.query_job_table(t0s, T, precede, True, True, lambda mem: 0)
    ut0, g0, pr0 = engine.shared_pair_table(track, spans, T)
    ut, g, pr = engine.shared_pair_table(table, spans, T, decide_jobs=n_track, max_entries=64)
    assert g <= 64 and len(pr) == len(table.mem_feat)
    # every memory entry of every job reads a list of its own (query frame, direction) and frame
    for job in table.jobs:
        key = engine.pair_key(table, job)
        for k in range(job[1], job[2]):
            u, i = divmod(pr[k], g)
            assert engine.pair_key(ut, ut.jobs[u]) == key and ut.mem_feat[ut.jobs[u][1] + i] == table.mem_feat[k]
    # the lists the tracks use are the same (query frame, frame) pairs as without the checks
    old = {(engine.pair_key(ut0, ut0.jobs[p // g0]), ut0.mem_feat[ut0.jobs[p // g0][1] + p % g0]) for p in pr0}
    new = {(engine.pair_key(ut, ut.jobs[p // g]), ut.mem_feat[ut.jobs[p // g][1] + p % g]) for p in pr[:len(pr0)]}
    assert old == new
    # one group: no sharing, with or without the checks
    one, sp1 = engine.query_job_table([7], T, precede, True, True, lambda mem: 0)
    n1 = len(one)
    engine.cycle_job_table(one, sp1, T, precede, True, True, frames, lambda mem: 0)
    assert engine.shared_pair_table(one, sp1, T, decide_jobs=n1, max_entries=64) is None


def test_long_clips_split_a_union_over_several_lists_jobs():
    """frames=None on a clip longer than 64 frames: a backward query frame sees more than 64 distinct first frames;
    its union is split over utable jobs of at most 64 entries instead of giving up sharing"""
    T, precede = 90, 5
    t0s = tuple(range(0, T, 5))
    table, spans, n_track, _ = _tables(T, precede, t0s, None)
    ut, g, pr = engine.shared_pair_table(table, spans, T, decide_jobs=n_track, max_entries=64)
    assert g == 64 and max(j[2] - j[1] for j in ut.jobs) <= 64
    assert len({engine.pair_key(ut, j) for j in ut.jobs}) < len(ut.jobs)


def test_cycle_key_is_validated():
    import torch
    import fgvc_b200
    base = dict(precede_frames=3, topk=10, temperature=0.07, neighbor_range=10)
    for bad, err in ((dict(frames=0, threshold=4), ValueError), (dict(frames=1.5, threshold=4), ValueError),
                     (dict(frames=2), TypeError), (dict(frames=2, threshold=4, extra=1), TypeError),
                     (dict(frames=2, threshold=-1), ValueError)):
        with pytest.raises(err):
            fgvc_b200.VanillaTracker(backbone=torch.nn.Identity(), test_cfg=dict(base, cycle_occlusion=bad))
    trk = fgvc_b200.VanillaTracker(backbone=torch.nn.Identity(), test_cfg=dict(base, cycle_occlusion=dict(
        frames=None, threshold=4)))
    assert trk.cycle_cfg() == dict(frames=None, threshold=4.0, max_bytes=None)
    assert fgvc_b200.VanillaTracker(backbone=torch.nn.Identity(), test_cfg=base).cycle_cfg() is None
    from fgvc_b200.c2f_tracker import C2FPointTracker
    with pytest.raises(NotImplementedError):
        C2FPointTracker(dict(base, radius_fine=5, cycle_occlusion=dict(frames=1, threshold=4)))


def test_packed_cuts_keep_the_tracking_tiles():
    """K1 over tracking and check jobs in one launch packs query tiles within each range only: the tile groups of the
    tracking jobs are those of a launch over them alone"""
    T, precede = 20, 5
    table, spans, n_track, _ = _tables(T, precede, (3,), 4)
    for J in (2, 4):
        g0, u0, p0 = table.packed(0, n_track, J, "cpu")
        g1, u1, p1 = table.packed(n_track, len(table), J, "cpu")
        g, u, p = table.packed_cuts([(0, n_track), (n_track, len(table))], J, "cpu")
        assert g.shape[0] == g0.shape[0] + g1.shape[0]
        assert g[:g0.shape[0]].tolist() == g0.tolist() and u[:u0.numel()].tolist() == u0.tolist()
        assert p[:p0.shape[0]].tolist() == p0.tolist()
        rest = g[g0.shape[0]:].clone()
        rest[:, 5:7] -= u0.numel()
        assert rest.tolist() == g1.tolist() and u[u0.numel():].tolist() == u1.tolist()
        assert p[p0.shape[0]:].tolist() == p1.tolist()
