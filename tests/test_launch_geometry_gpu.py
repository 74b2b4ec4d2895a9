"""Launch geometry of the inference chain (set_option "geometry" / "geo_front" / "geo_proj" / "geo_head"): the grids of
front_tc, proj_h and head change, the bytes they compute do not.  Every kernel strides its windows, tiles or rows by
gridDim.x, so full-chip grids (geometry 0), work-sized grids (geometry 1) and a single CTA per kernel must agree exactly."""
import numpy as np
import pytest
import torch

from roko_b200._cabi import RokoB200Error
from roko_b200.synth import structured_windows, uniform_windows

pytestmark = pytest.mark.gpu

ONE_CTA = 1 << 20          # more units per CTA than any batch has: one CTA (block) per launch
WORK_SIZED = dict(geometry=1)
FULL_CHIP = dict(geometry=0)
SINGLE = dict(geometry=1, geo_front=ONE_CTA, geo_proj=ONE_CTA, geo_head=ONE_CTA)
# the default first, then every change of setting followed by a capture and a replay; the last step leaves one CTA per kernel
SEQUENCE = [("work-sized", WORK_SIZED), ("full-chip", FULL_CHIP), ("one-cta", SINGLE), ("full-chip again", FULL_CHIP)]


def _windows(n):
    half = n // 2
    return np.concatenate([structured_windows(n - half, seed=4000 + n), uniform_windows(half, seed=5000 + n)])


def _predict_twice(m, x, stream):
    with torch.cuda.stream(stream):                 # graphs need a real (capturable) stream
        first = m.predict(x, return_logits=True)
        again = m.predict(x, return_logits=True)    # with graphs on: the replay of the instance the first call captured
    stream.synchronize()
    return first, again


@pytest.mark.parametrize("batch", [1, 5, 63, 64, 128, 129, 300, 1000, 2368])
def test_geometry_is_bit_identical(make_model, batch):
    """Logits and labels under every setting, with graphs on and off; 63 / 64 straddle the tensor-core recurrence's
    rec_tc_min, 129 / 300 / 1000 leave ragged projection tiles, 2368 is a whole predict_host pass."""
    x = torch.from_numpy(_windows(batch)).to("cuda:0")
    ref_labels, ref_logits = make_model(graphs=0, **FULL_CHIP).predict(x, return_logits=True)
    s = torch.cuda.Stream()
    for graphs in (1, 0):
        m = make_model(graphs=graphs)
        for name, setting in SEQUENCE:
            for k, v in setting.items():
                m.set_option(k, v)
            for labels, logits in _predict_twice(m, x, s):
                assert torch.equal(labels, ref_labels), (graphs, name)
                assert torch.equal(logits, ref_logits), (graphs, name)


@pytest.mark.parametrize("setting", [WORK_SIZED, SINGLE], ids=["work-sized", "one-cta"])
def test_batch_128_matches_reference_class(make_model, golden_b128, setting):
    """The batch bench.py times: labels equal the reference class's (tests/golden/golden_b128_seed1.npz)."""
    m = make_model(**setting)
    labels, logits = _predict_twice(m, torch.from_numpy(golden_b128["x"]).to("cuda:0"), torch.cuda.Stream())[1]
    assert np.array_equal(labels.cpu().numpy(), golden_b128["labels"])
    assert np.abs(logits.cpu().numpy() - golden_b128["logits"]).max() <= 5e-6
    m.check_codes()


@pytest.mark.parametrize("setting", [WORK_SIZED, SINGLE], ids=["work-sized", "one-cta"])
def test_range_guard_under_geometry(make_model, golden, seed1_state, setting):
    """A GRU weight beyond the fp16-split range is still reported by check_codes() when the projection runs on fewer CTAs."""
    sd = {k: v.clone() for k, v in seed1_state.items()}
    sd["gru.weight_hh_l1"][5, 7] = 300.0
    m = make_model(**setting)
    m.load_state_dict(sd)
    m.predict(torch.from_numpy(golden["x"][:1]).to("cuda:0"))
    with pytest.raises(RokoB200Error):
        m.check_codes()


def test_geometry_options_reject_bad_values(make_model):
    m = make_model()
    for name, value in (("geometry", 2), ("geometry", -1), ("geo_front", 0), ("geo_proj", -3), ("geo_head", ONE_CTA + 1)):
        with pytest.raises(RokoB200Error):
            m.set_option(name, value)
