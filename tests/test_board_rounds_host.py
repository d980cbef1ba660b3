"""Later rounds of the board search (max_num_of_boards > 2) in the host build of the board core
(csrc/ag_board_core.h through tests/host_board_test.cpp) against the oracle, on frames holding
several boards whose tag ids overlap: a later board overwrites the ids an earlier one decoded."""
import numpy as np
import pytest

import synth
from test_board_core_host import hb, host_detect  # noqa: F401  (hb is a fixture)


@pytest.fixture(scope="module")
def composites():
    return {"four_boards": synth.composite_boards(*synth.FOUR_BOARDS),
            "small_boards": synth.composite_boards(*synth.SMALL_BOARDS, canvas=(960, 1280))}


@pytest.mark.parametrize("max_boards", [3, 4, 255])
@pytest.mark.parametrize("name", ["four_boards", "small_boards"])
def test_later_rounds_identical_to_oracle(hb, pkg, oracle, composites, name, max_boards):  # noqa: F811
    img = composites[name]
    got, _, status, _ = host_detect(hb, pkg, oracle, img, max_boards=max_boards)
    want = oracle.detect(img, max_boards=max_boards)
    assert status == 0 and len(want) >= 12
    # the input has to exercise the rounds: a third round changes the second round's answer
    two = oracle.detect(img, max_boards=2)
    assert sorted(two) != sorted(want) or any(not np.array_equal(two[k], want[k]) for k in want)
    assert sorted(got) == sorted(want)
    for k in want:
        assert np.array_equal(got[k], want[k]), k
