"""CPU: host side of sliding-window tagging of long recordings -- the window plan, its execution batches, and the argument
checks of the _windows C entry points (all return before touching a device)."""
import pytest
import torch

from audioset_convnext_inf_b200 import _native
from audioset_convnext_inf_b200.engine import MIN_RAGGED_LEN
from audioset_convnext_inf_b200.windows import plan_windows, window_batches


def _rows(plan):
    return list(zip(plan.recording.tolist(), plan.start.tolist(), plan.length.tolist()))


def test_plan_adds_an_end_aligned_tail_only_when_needed():
    W = 320000
    # 30 s at 10 s hop ends exactly on the last sample: no tail
    assert _rows(plan_windows([960000], W, W)) == [(0, 0, W), (0, W, W), (0, 2 * W, W)]
    # 30 s + 17 samples: the hop-grid windows end 17 samples early, one end-aligned window is added
    assert _rows(plan_windows([960017], W, W)) == [(0, 0, W), (0, W, W), (0, 2 * W, W), (0, 960017 - W, W)]
    # 1 s hop over 95.3 s: every sample covered by a full window
    n = 3049600
    p = plan_windows([n], W, 32000)
    starts = p.start.tolist()
    assert starts[:-1] == list(range(0, n - W + 1, 32000)) and starts[-1] == n - W
    assert (p.length == W).all()


def test_plan_short_and_exact_recordings():
    W = 320000
    assert _rows(plan_windows([W], W, 32000)) == [(0, 0, W)]                       # exactly one window: an ordinary one
    assert _rows(plan_windows([240000], W, 32000)) == [(0, 0, 240000)]             # shorter: one window at its own length
    assert _rows(plan_windows([MIN_RAGGED_LEN], W, 1)) == [(0, 0, MIN_RAGGED_LEN)]


def test_plan_gaps_when_hop_exceeds_the_window():
    W, hop = 320000, 400000
    p = plan_windows([1500000], W, hop)
    assert _rows(p) == [(0, 0, W), (0, 400000, W), (0, 800000, W), (0, 1500000 - W, W)]
    assert _rows(plan_windows([1120000], W, hop)) == [(0, 0, W), (0, 400000, W), (0, 800000, W)]   # last ends at n


def test_plan_order_and_offsets_across_recordings():
    W = 320000
    lens = [960017, 240000, W, 3049600]
    p = plan_windows(lens, W, 100001)
    rec, start = p.recording.tolist(), p.start.tolist()
    assert rec == sorted(rec) and set(rec) == {0, 1, 2, 3}
    for r in range(4):
        s = [st for rr, st in zip(rec, start) if rr == r]
        assert s == sorted(s)
    base = [0, 960017, 960017 + 240000, 960017 + 240000 + W]
    assert p.offset.tolist() == [base[r] + s for r, s in zip(rec, start)]
    assert all((p.offset + p.length <= sum(lens)).tolist())


def test_plan_tables_are_int64():
    p = plan_windows([2 ** 31 + 10 ** 6], 320000, 2 ** 30)
    for t in (p.recording, p.start, p.length, p.offset):
        assert t.dtype == torch.int64 and t.device.type == "cpu"
    assert p.offset.max().item() + 320000 == 2 ** 31 + 10 ** 6                    # offsets past 2^31 are exact


@pytest.mark.parametrize("args, match", [(([MIN_RAGGED_LEN - 1], 320000, 32000), "recording 0 has 7359 samples"),
                                         (([400000, 100], 320000, 32000), "recording 1 has 100 samples"),
                                         (([400000], MIN_RAGGED_LEN - 1, 32000), "window_samples=7359"),
                                         (([400000], 320000, 0), "hop_samples"),
                                         (([400000], 320000, -5), "hop_samples")])
def test_plan_errors(args, match):
    with pytest.raises(ValueError, match=match):
        plan_windows(*args)


def test_plan_of_no_recordings_is_empty():
    p = plan_windows([], 320000, 32000)
    assert p.recording.numel() == p.start.numel() == p.length.numel() == p.offset.numel() == 0
    assert p.offset.dtype == torch.int64
    assert window_batches(p, 64) == []


def test_window_batches_full_chunks_non_ragged_and_short_windows_ragged():
    W = 320000
    lens = [W * 20, 240000, 100000, W, 7360]
    p = plan_windows(lens, W, 32000)
    batches = window_batches(p, 16)
    seen = sorted(i for _, _, idx in batches for i in idx)
    assert seen == list(range(p.length.numel()))
    length = p.length.tolist()
    full = [b for b in batches if b[1] is None]
    assert all(canvas == W and len(idx) <= 16 and all(length[i] == W for i in idx) for canvas, _, idx in full)
    assert [len(idx) for _, _, idx in full[:-1]] == [16] * (len(full) - 1)       # whole chunks first, as forward_all cuts them
    rag = [b for b in batches if b[1] is not None]
    assert sorted(i for _, _, idx in rag for i in idx) == [i for i, n in enumerate(length) if n != W]
    for canvas, ls, idx in rag:
        assert ls == [length[i] for i in idx] and canvas >= max(ls)


# ---- C ABI: every _windows entry point checks its arguments before it touches a device ---------------------------------
_P = 4096        # a non-null, 16-byte aligned dummy address: the calls below must fail before dereferencing anything
_NEW = {
    "acx_wave_prep_windows": lambda rec, n, off, B: (rec, n, off, 0, _P, _P, B, 32000, 1024, 33024, _native.ACX_BF16, 0),
    "acx_wave_prep_pcm16_windows": lambda rec, n, off, B: (rec, n, off, 0, _P, _P, B, 32000, 1024, 33024, _native.ACX_BF16, 0),
    "acx_frame_fold_windows": lambda rec, n, off, B: (rec, n, off, 0, _P, _P, B, 32000, 101, 1024, 320, 0),
    "acx_frame_fold_pcm16_windows": lambda rec, n, off, B: (rec, n, off, 0, _P, _P, B, 32000, 101, 1024, 320, 0),
}


def test_new_entry_points_are_the_windows_set():
    assert {n for n in _native.SIGNATURES if n.endswith("_windows")} == set(_NEW)


@pytest.mark.parametrize("name", sorted(_NEW))
def test_windows_entry_points_reject_bad_arguments(name):
    fn = getattr(_native.load(), name)
    assert len(_native.SIGNATURES[name]) == len(_NEW[name](_P, 10 ** 6, _P, 2))
    assert fn(*_NEW[name](0, 10 ** 6, _P, 2)) == 1 and "null" in _native.last_error()          # ACX_ERR_ARG: no recording
    assert fn(*_NEW[name](_P, 10 ** 6, 0, 2)) == 1 and "null" in _native.last_error()          # no offsets
    assert fn(*_NEW[name](_P, 512, _P, 2)) == 1 and "rec_len" in _native.last_error()          # too short to reflect
    assert fn(*_NEW[name](_P, -1, _P, 2)) == 1 and "rec_len" in _native.last_error()
    assert fn(*_NEW[name](_P, 10 ** 6, _P, 0)) == 1 and "B=0" in _native.last_error()          # empty batch
    assert fn(*_NEW[name](_P, 2 ** 40, _P, -3)) == 1 and "B=-3" in _native.last_error()        # 64-bit rec_len passes through
    assert fn(*([0] * len(_native.SIGNATURES[name]))) == 1                                       # everything null
