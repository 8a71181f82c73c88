"""Pin the oracle on the reference: the port must be bit-identical to the reference's own outputs on the golden cases
(tests/golden/*.npz, made by running the reference with tests/golden/make_golden.py)."""
import numpy as np
import pytest
import torch

from tests.golden import cases as G
from tests import util


@pytest.mark.parametrize("name", ["sins_b2_f24_h128", "sins_b1_f7_h33", "sins_b1_f12_h40_m65_initphase",
                                  "combsub_b2_f24", "superfast_b2_f24", "superfast_b1_f2_constpad",
                                  "sinegen_b2_f12", "csfast_b2_f24", "csfast_b1_f9_initphase", "srcmod_b2_f10"])
def test_port_bit_identical_to_live_reference(name):
    inp = G.build_inputs(name)
    gold = util.load_golden(name)
    util.check_inputs_match_golden(name, inp, gold)
    out = util.port_outputs(name, inp)
    for key in inp["case"]["store"]:
        ref = torch.from_numpy(gold[key])
        assert torch.equal(out[key], ref), (name, key, np.abs(out[key].numpy() - gold[key]).max())
