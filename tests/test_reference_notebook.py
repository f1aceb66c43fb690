""" Drop-in check of the public API against the reference's own behaviour: `Solver.reshape_and_concat` on random
argument mixes, compared with outputs of the unmodified reference stored in tests/golden/reshape_and_concat.npz
(written by oracle/make_golden.py). """
import pytest
import torch

import problems as P
from helpers import load_golden


def test_reshape_and_concat_equals_the_reference_on_random_inputs():
    """ `Solver.reshape_and_concat` (reference model_torch.py:328-362) decides how `predict` and constraints read
    numbers / arrays / lists / tensors: same output as the reference's own classmethod on random argument mixes. """
    from pydens_b200 import Solver
    g = load_golden('reshape_and_concat')
    cases = P.reshape_and_concat_cases()
    assert len(cases) == g['rejected'].size
    off = 0
    for case, args in enumerate(cases):
        if g['rejected'][case]:                            # the reference rejects the mix: so must we
            with pytest.raises(Exception):
                Solver.reshape_and_concat(list(args))
            continue
        shape = tuple(int(s) for s in g['shapes'][case])
        want = torch.from_numpy(g['values'][off:off + shape[0] * shape[1]].reshape(shape))
        off += shape[0] * shape[1]
        got = Solver.reshape_and_concat(list(args))
        assert tuple(got.shape) == shape, (case, [type(a).__name__ for a in args])
        assert torch.allclose(got.to(torch.float64), want, rtol=1e-6, atol=1e-7), case
    assert off == g['values'].size
