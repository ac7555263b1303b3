"""CPU tests of the engine's decode-row setup (engine.init_rows): the tokens, teacher-forcing table, row state
(tw_row_state) and grammar begin index that greedy decode and beam search start from, with and without a prefilled text
prompt, against literal tensors.  Small constants keep the tables readable: pad 9, <|0.00|> 100,
max_initial_timestamp_index 50, [<|startoftranscript|>, language, task] = [1, 2, 3], <|notimestamps|> 4, prompt_ids
[7, 8]; a language of -1 asks for language detection."""
from types import SimpleNamespace

import pytest
import torch

from turbo_whisper_workspace_b200 import _lib
from turbo_whisper_workspace_b200.engine import WhisperEngine, init_rows

MAX_LEN = 8
_ = -1      # free position of the teacher-forcing table

# (rows, timestamps, prefilled, flat) -> (tokens, forced, state {pos, finished, last_ts, text_lo, ts_lo, ts_hi, begin,
# mode}, begin_index)
CASES = {
    "greedy_ts": (
        [[1, 2, 3], [1, -1, 3]], True, False, False,
        [[1, 9, 9, 9, 9, 9, 9, 9], [1, 9, 9, 9, 9, 9, 9, 9]],
        [[_, 2, 3, _, _, _, _, _], [_, _, 3, _, _, _, _, _]],
        [[0, 0, -1, 0, 0, 0, 0, 0], [0, 0, -1, 0, 0, 0, 0, 1]], 3),
    "greedy_nots": (
        [[1, 2, 3, 4], [1, -1, 3, 4]], False, False, False,
        [[1, 9, 9, 9, 9, 9, 9, 9], [1, 9, 9, 9, 9, 9, 9, 9]],
        [[_, 2, 3, 4, _, _, _, _], [_, _, 3, 4, _, _, _, _]],
        [[0, 0, -1, 0, 0, 0, 0, 2], [0, 0, -1, 0, 0, 0, 0, 3]], 4),
    "greedy_prompt_ts": (
        [[7, 8, 1, 2, 3], [7, 8, 1, 5, 3]], True, True, False,
        [[7, 8, 1, 2, 3, 9, 9, 9], [7, 8, 1, 5, 3, 9, 9, 9]],
        [[_] * 8, [_] * 8],
        [[4, 0, -1, 100, 100, 150, 1, 0], [4, 0, -1, 100, 100, 150, 1, 0]], 5),
    "greedy_prompt_nots": (
        [[7, 8, 1, 2, 3, 4]], False, True, False,
        [[7, 8, 1, 2, 3, 4, 9, 9]],
        [[_] * 8],
        [[5, 0, -1, 100, 100, 150, 1, 2]], 6),
    "beam_ts": (
        [[1, 2, 3], [1, 5, 3]], True, False, True,
        [[1, 2, 3, 9, 9, 9, 9, 9], [1, 5, 3, 9, 9, 9, 9, 9]],
        [[_, 2, 3, _, _, _, _, _], [_, 5, 3, _, _, _, _, _]],
        [[0, 0, -1, 0, 0, 0, 0, 2], [0, 0, -1, 0, 0, 0, 0, 2]], 3),
    "beam_nots": (
        [[1, 2, 3, 4]], False, False, True,
        [[1, 2, 3, 4, 9, 9, 9, 9]],
        [[_, 2, 3, 4, _, _, _, _]],
        [[0, 0, -1, 0, 0, 0, 0, 2]], 4),
    "beam_prompt_ts": (
        [[7, 8, 1, 2, 3]], True, True, True,
        [[7, 8, 1, 2, 3, 9, 9, 9]],
        [[_, 8, 1, 2, 3, _, _, _]],
        [[4, 0, -1, 100, 100, 150, 1, 2]], 5),
    "beam_prompt_nots": (
        [[7, 8, 1, 2, 3, 4], [7, 8, 1, 5, 3, 4]], False, True, True,
        [[7, 8, 1, 2, 3, 4, 9, 9], [7, 8, 1, 5, 3, 4, 9, 9]],
        [[_, 8, 1, 2, 3, 4, _, _], [_, 8, 1, 5, 3, 4, _, _]],
        [[5, 0, -1, 100, 100, 150, 1, 2], [5, 0, -1, 100, 100, 150, 1, 2]], 6),
}


def _grammar():
    g = _lib.Grammar()
    g.pad, g.ts_begin, g.max_initial_ts = 9, 100, 50
    return g


@pytest.mark.parametrize("case", list(CASES))
def test_init_rows(case):
    rows, timestamps, prefilled, flat, tokens, forced, state, begin = CASES[case]
    got = init_rows(torch.tensor(rows), MAX_LEN, _grammar(), timestamps, prefilled=prefilled, flat=flat)
    for name, g, want in zip(("tokens", "forced", "state"), got[:3], (tokens, forced, state)):
        assert g.dtype == torch.int32 and g.tolist() == want, name
    assert got[3] == begin


@pytest.mark.parametrize("prompt_ids, timestamps, want", [
    (None, True, [1, 2, 3]), (None, False, [1, 2, 3, 4]), ([7, 8], True, [7, 8, 1, 2, 3]),
    ([7, 8], False, [7, 8, 1, 2, 3, 4])])
def test_prompt_row(prompt_ids, timestamps, want):
    eng = SimpleNamespace(gen=SimpleNamespace(no_timestamps_token_id=4))
    assert WhisperEngine.prompt_row(eng, prompt_ids, torch.tensor([1, 2, 3], dtype=torch.int32), timestamps) == want
