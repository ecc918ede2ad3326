"""CPU: host side of ragged batches (clips of different lengths in one forward) -- batch planner, per-clip bound table,
length validation and the argument checks of the _ragged C entry points (all return before touching a device)."""
import numpy as np
import pytest
import torch

from audioset_convnext_inf_b200 import _native
from audioset_convnext_inf_b200.engine import MIN_RAGGED_LEN, check_lengths, out_time_dims, ragged_table
from audioset_convnext_inf_b200.extract import CANVAS_STEP, extract_clipwise, ragged_batches


def test_min_ragged_len_is_the_shortest_clip_with_a_last_stage_row():
    assert out_time_dims(MIN_RAGGED_LEN)[1][3] == 1
    assert out_time_dims(MIN_RAGGED_LEN - 1)[1][3] == 0
    assert MIN_RAGGED_LEN > 1024 // 2                  # reflect padding needs L > n_fft / 2


def test_ragged_batches_sorted_bounded_and_rounded_up():
    rng = np.random.default_rng(0)
    lengths = rng.integers(7360, 30 * 32000, size=203).tolist() + [32000, 32000, 64001]
    plan = ragged_batches(lengths, max_batch=16)
    flat = [i for _, idx in plan for i in idx]
    assert sorted(flat) == list(range(len(lengths)))                  # every clip exactly once
    assert [lengths[i] for i in flat] == sorted(lengths)              # length-sorted
    assert all(len(idx) <= 16 for _, idx in plan) and len(plan) == -(-len(lengths) // 16)
    for canvas, idx in plan:
        longest = max(lengths[i] for i in idx)
        assert canvas % CANVAS_STEP == 0 and longest <= canvas < longest + CANVAS_STEP
    assert ragged_batches([32000], 4) == [(32000, [0])]               # an exact multiple is not rounded further
    assert ragged_batches([], 4) == []


def test_ragged_table_matches_out_time_dims():
    lengths = [7360, 7679, 7680, 96123, 320000, 480001]
    tab = ragged_table(lengths)
    assert tab.dtype == torch.int32 and tab.shape == (6, len(lengths)) and tab.is_contiguous()
    for b, n in enumerate(lengths):
        T, hs = out_time_dims(n)
        assert tab[:, b].tolist() == [n, T] + hs


@pytest.mark.parametrize("bad, match", [([7359, 9000], r"\[7360, 32000\]"), ([9000, 32001], r"\[7360, 32000\]"),
                                        ([9000], "1 entries for a batch of 2"), ([9000, 9000, 9000], "3 entries"),
                                        ([9000, "x"], "integers")])
def test_check_lengths_rejects(bad, match):
    with pytest.raises(ValueError, match=match):
        check_lengths(bad, 2, 32000)


def test_check_lengths_accepts_sequences_and_cpu_tensors():
    assert check_lengths([7360, 32000], 2, 32000) == [7360, 32000]
    assert check_lengths(torch.tensor([9000, 10000]), 2, 32000) == [9000, 10000]
    assert check_lengths(np.array([9000, 10000]), 2, 32000) == [9000, 10000]


class _FakeModel(torch.nn.Module):
    """forward_all over a ragged batch on the host: each output is a function of the clip's own samples only."""

    def __init__(self):
        super().__init__()
        self.p = torch.nn.Parameter(torch.zeros(1))
        self.calls = []

    def forward_all(self, x, lengths=None):
        self.calls.append((tuple(x.shape), list(lengths)))
        s = torch.stack([x[b, :n].double().sum() for b, n in enumerate(lengths)]).float()
        h3 = torch.tensor([out_time_dims(n)[1][3] for n in lengths])
        frame = torch.zeros(x.shape[0], 2, out_time_dims(x.shape[1])[1][3], 7)
        for b, h in enumerate(h3.tolist()):
            frame[b, :, :h] = s[b]
        return {"clipwise_logits": s[:, None].repeat(1, 3), "frame_embeddings": frame, "frame_lengths": h3}


def test_extract_clipwise_restores_input_order_and_ignores_the_canvas_tail():
    rng = np.random.default_rng(1)
    lengths = rng.integers(7360, 100000, size=37).tolist()
    waves = [rng.standard_normal(n).astype(np.float32) for n in lengths]
    m = _FakeModel()
    res = extract_clipwise(m, waves, max_batch=8, want=("clipwise_logits", "frame_embeddings", "frame_lengths"))
    assert len(m.calls) == 5
    for shape, ls in m.calls:
        assert shape[1] % CANVAS_STEP == 0 and shape[1] >= max(ls) and len(ls) <= 8
    for i, w in enumerate(waves):
        s = torch.tensor(w, dtype=torch.float64).sum().float()
        assert torch.equal(res["clipwise_logits"][i], s.repeat(3))
        h3 = out_time_dims(lengths[i])[1][3]
        assert res["frame_lengths"][i].item() == h3
        assert res["frame_embeddings"][i].shape == (2, h3, 7) and (res["frame_embeddings"][i] == s).all()


# ---- C ABI: every _ragged entry point checks its arguments before it touches a device ---------------------------------
_P = 4096        # a non-null, 16-byte aligned dummy address: the calls below must fail before dereferencing anything
_NEW = {
    "acx_wave_prep_ragged": lambda v: (_P, _P, _P, 2, 32000, 1024, 33024, _native.ACX_BF16, 32000, v, 0),
    "acx_frame_fold_ragged": lambda v: (_P, _P, _P, 2, 32000, 101, 1024, 320, 32000, v, 0),
    "acx_stem_ragged": lambda v: (_P, _P, _P, _P, _P, _P, 2, 101, 224, _native.ACX_BF16, v, 0),
    "acx_stem_gp_ragged": lambda v: (_P, _P, _P, _P, _P, _P, 2, 101, 224, v, 0),
    "acx_dwconv_tc_ragged": lambda v: (_P, _P, _P, 2 * _P, 2, 27, 56, 96, v, 0),
    "acx_dwconv_tc_gp_ragged": lambda v: (_P, _P, _P, 2 * _P, 2, 27, 56, 96, v, 0),
    "acx_dwconv_ln_ragged": lambda v: (_P, _P, _P, _P, _P, _P, 2, 3, 7, 768, _native.ACX_BF16, v, 0),
    "acx_head_ragged": lambda v: (_P, _P, _P, _P, _P, _P, _P, _P, _P, 2, 3, 7, 768, 527, _native.ACX_BF16, v, 0),
    "acx_nhwc_to_nchw_f32_ragged": lambda v: (_P, _P, 2, 3, 7, 768, _native.ACX_BF16, v, 0),
}


def test_new_entry_points_are_the_ragged_set():
    assert {n for n in _native.SIGNATURES if n.endswith("_ragged")} == set(_NEW)


@pytest.mark.parametrize("name", sorted(_NEW))
def test_ragged_entry_points_reject_null_pointers(name):
    fn = getattr(_native.load(), name)
    assert len(_native.SIGNATURES[name]) == len(_NEW[name](0))
    assert fn(*_NEW[name](0)) == 1 and "valid" in _native.last_error()          # ACX_ERR_ARG: no bound array
    zeros = [0] * len(_native.SIGNATURES[name])
    assert fn(*zeros) == 1                                                        # everything null


def test_ragged_prep_checks_the_row_pitch():
    lib = _native.load()
    assert lib.acx_wave_prep_ragged(_P, _P, _P, 2, 32000, 1024, 33024, _native.ACX_BF16, 31999, _P, 0) == 1
    assert "pitch" in _native.last_error()
    assert lib.acx_frame_fold_ragged(_P, _P, _P, 2, 32000, 101, 1024, 320, 31999, _P, 0) == 1
    assert "pitch" in _native.last_error()
