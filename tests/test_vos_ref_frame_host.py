"""Host side of mask propagation from an annotated frame anywhere in the clip (CPU only): argument checks and the job
table of MaskClipPropagator(ref_frame=...)."""
import pytest
import torch

from fgvc_b200 import _lib, engine


@pytest.mark.parametrize("ref_frame", [-1, 8, 2.0, "1", None, True])
def test_bad_ref_frame_raises_value_error(ref_frame):
    with pytest.raises(ValueError):
        engine.MaskClipPropagator(8, 64, 16, 24, 3, (32, 48), dict(precede_frames=3, topk=10, temperature=0.07),
                                  torch.device("cpu"), ref_frame=ref_frame)


def test_ref_frame_checks():
    assert engine.check_ref_frame(0, 1) == 0
    assert engine.check_ref_frame(7, 8) == 7
    for bad, T in ((1, 1), (-1, 5), (5, 5)):
        with pytest.raises(ValueError):
            engine.check_ref_frame(bad, T)


def test_tracker_rejects_a_bad_ref_frame():
    import fgvc_b200
    trk = fgvc_b200.VanillaTracker(backbone=torch.nn.Identity(), test_cfg=dict(precede_frames=3, topk=10,
                                                                                temperature=0.07))
    with pytest.raises(ValueError):
        trk.propagate_masks(torch.zeros(4, 8, 6, 6), torch.zeros(6, 6, dtype=torch.long), (12, 12), 2, ref_frame=4)


def test_run_host_takes_frame_zero_only():
    clip = object.__new__(engine.MaskClipPropagator)       # (the constructor needs a device; run_host checks first)
    clip.ref_frame = 3
    with pytest.raises(NotImplementedError):
        clip.run_host(None, None, None)


@pytest.mark.parametrize("with_first", [True, False])
@pytest.mark.parametrize("nr", [12, None])
def test_frame_zero_table_is_the_forward_loop(with_first, nr):
    """query_job_table([0], ..., bidirectional=True) is the table MaskClipPropagator always built for frame 0."""
    T, precede = 15, 4
    unmasked_first = 1
    want = engine.JobTable()
    for t in range(1, T):
        mem = engine.memory_frames(t, precede, with_first)
        want.add(t, mem, mem, t, unmasked=len(mem) if nr is None else unmasked_first)
    got, _ = engine.query_job_table([0], T, precede, with_first, True,
                                    lambda mem: len(mem) if nr is None else unmasked_first)
    assert (got.jobs, got.mem_feat, got.mem_label) == (want.jobs, want.mem_feat, want.mem_label)


def test_both_directions_of_a_middle_frame():
    T, precede, t0 = 12, 3, 5
    tb, _ = engine.query_job_table([t0], T, precede, True, True, lambda mem: 1)
    q = [j[0] for j in tb.jobs]
    assert q == list(range(t0 + 1, T)) + list(range(t0 - 1, -1, -1))
    assert [j[3] for j in tb.jobs] == q
    back = [[r & ~_lib.MEM_UNMASKED for r in tb.mem_feat[j[1]:j[2]]] for j in tb.jobs[T - 1 - t0:]]
    # the forward memory rule on the time-reversed clip, mapped back
    assert back[0] == [t0, t0] and back[1] == [t0, t0, t0 - 1] and back[-1] == [t0, 3, 2, 1]
