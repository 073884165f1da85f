"""CPU tests of the content-mode input builders: argument errors that wire.aggregation_inputs raises before any engine
call (the reference's ValueError for non-bitstring messages, malformed group offsets)."""
import numpy as np
import pytest


def test_aggregation_inputs_rejects_non_bitstrings_before_the_engine():
    from lattice_cryptography_b200 import wire
    with pytest.raises(ValueError, match='Input messages must be bitstrings.'):
        wire.aggregation_inputs(None, np.array([0, 2], np.int64), None, ['0101', 'hello'])
    with pytest.raises(ValueError, match='Input messages must be bitstrings.'):
        wire.aggregation_inputs(None, np.array([0, 1], np.int64), None, [7])


@pytest.mark.parametrize('agg_off', [[1, 2], [0, 3], [0, 2, 1, 2], [[0, 2]]])
def test_aggregation_inputs_rejects_bad_group_offsets(agg_off):
    from lattice_cryptography_b200 import wire
    with pytest.raises(ValueError, match='agg_off'):
        wire.aggregation_inputs(None, np.array(agg_off, np.int64), None, ['01', '1'])
