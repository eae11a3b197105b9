"""The argument handling of policy_step without a GPU (policy._step_mode): the mode names, and the narrowing of caller-given
actions of any integer dtype to the int8 the head kernel reads.  An action outside 0..A-1 must stay outside it -- it gets
logp NaN -- however wide or unsigned its dtype; none may wrap onto a valid action."""
import pytest
import torch

A = 8
CPU = torch.device("cpu")


def _policy():
    from sequential_social_dilemma_games_b200 import policy
    return policy


@pytest.mark.parametrize("dtype", [torch.uint8, torch.uint16, torch.uint32, torch.uint64, torch.int16, torch.int32, torch.int64])
def test_given_actions_of_every_integer_dtype_keep_their_validity(dtype):
    values = [0, 3, 7, 8, 9, 200, 255]
    if dtype.is_signed:
        values += [-1, -2, -128, 135, 2 ** 15 - 1]
    actions = torch.tensor(values, dtype=dtype)
    code, a = _policy()._step_mode("given", actions, len(values), A, CPU)
    assert a.dtype == torch.int8 and a.is_contiguous()
    want = [v if 0 <= v < A else (A if v >= A else -1) for v in values]
    assert a.tolist() == want


def test_unsigned_values_above_the_signed_range_stay_invalid():
    big = torch.tensor([2 ** 64 - 1, 2 ** 63, 2 ** 63 + 3, 5], dtype=torch.uint64)
    _, a = _policy()._step_mode("given", big, 4, A, CPU)
    assert a.tolist() == [-1, -1, -1, 5]


def test_int8_actions_are_passed_as_they_are():
    actions = torch.tensor([-1, 0, 7, 8, 127, -128], dtype=torch.int8)
    _, a = _policy()._step_mode("given", actions, 6, A, CPU)
    assert a.data_ptr() == actions.data_ptr()


def test_modes_and_their_actions_argument():
    from sequential_social_dilemma_games_b200 import _lib
    policy = _policy()
    assert policy._step_mode("sample", None, 4, A, CPU) == (_lib.ACT_SAMPLE, None)
    assert policy._step_mode("greedy", None, 4, A, CPU) == (_lib.ACT_GREEDY, None)
    ok = torch.zeros(4, dtype=torch.int8)
    for mode, actions in (("Sample", None), ("argmax", None), (0, None), (None, None), ("sample", ok), ("greedy", ok),
                          ("given", None), ("given", ok[:3]), ("given", ok.float()), ("given", ok.bool()), ("given", ok.tolist())):
        with pytest.raises(ValueError):
            policy._step_mode(mode, actions, 4, A, CPU)
