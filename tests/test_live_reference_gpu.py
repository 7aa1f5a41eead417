"""SURVEY.md 8c-i at full width: 64 seeds x 1000 steps per environment, recorded from the reference AT TEST TIME (one
process per lane, from the reference tree oracle/ref_shim finds) and replayed through the CUDA engine -- one-step mode
within 1e-12 with exact flags and time, free-running within the per-family tolerance with exact flags on every lane that
is still reproducible by the reference itself.  Without a reference tree the same checks run on every recording of the
same adapter committed under tests/golden/ (made from the unmodified reference by the same recorder, fewer seeds:
cartpole 40, uav_att_rand 3, uav_pos_dis 27)."""
import glob
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from helpers import ENGINE_TOL, EngineBackend, replay  # noqa: E402

pytestmark = pytest.mark.gpu

# fixture family (helpers.env_specs / ENGINE_TOL key) for each recorded adapter, and the share of (step, lane) samples that
# must stay comparable in free-running mode (the rest are lanes past the chaos cut-off: their self-drift exceeds 1e-11)
CASES = {"cartpole": ("cartpole", 0.5), "uav_att_rand": ("uav_att_rand", 0.99), "uav_pos_dis": ("uav_pos_dis", 0.9)}
# free-running ceilings over 64 fresh seeds, ~10x the values measured on B200 (cartpole 5.9e-14, uav_att_rand 2.4e-14,
# uav_pos_dis 7.4e-10 .. 4.0e-9 depending on the seed: the worst of 64 lanes is a lane whose redrawn gains amplify a
# last-bit difference ~1e7-fold, profiles/r2/drift.md -- the reference's own one-ulp twin drifts 1e-8 there)
LIVE_TOL = {"cartpole": 2e-12, "uav_att_rand": 2e-13, "uav_pos_dis": 5e-8}


def _have_reference():
    from oracle import ref_shim
    return ref_shim.available()


def _recordings(adapter):
    """64 lanes x 1000 steps recorded now from the reference tree, else the committed recordings of `adapter`."""
    if _have_reference():
        from oracle.live_record import record_parallel
        g = record_parallel(adapter, lanes=64, steps=1000, seed=77)
        assert g["reward"].shape == (1000, 64)
        return [g]
    out = []
    for path in sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "*.npz"))):
        with np.load(path) as z:
            if "meta" in z.files and json.loads(str(z["meta"]))["adapter"] == adapter:
                out.append({k: z[k] for k in z.files})
    assert out, f"no committed recording of {adapter} under tests/golden"
    return out


@pytest.mark.parametrize("adapter", sorted(CASES))
def test_64_seeds_1000_steps_against_the_live_reference(adapter):
    family, live_min = CASES[adapter]
    for g in _recordings(adapter):
        L = g["reward"].shape[1]
        assert int(g["done"].sum()) >= L   # as many episode ends as lanes
        res = replay(g, EngineBackend(family, L), resync=True, name=family)
        assert res["flag_mismatch"] == 0 and res["done_mismatch"] == 0 and res["worst"]["time"] == 0.0, res
        for k, v in res["worst"].items():
            assert v <= 1e-12, (adapter, k, v)
        res = replay(g, EngineBackend(family, L), resync=False, name=family)
        assert res["flag_mismatch"] == 0 and res["done_mismatch"] == 0 and res["worst"]["time"] == 0.0, res
        assert res["live_fraction"] >= live_min, (adapter, res["live_fraction"])
        assert res["worst_ratio"] <= 1.0, res
        for k, v in res["worst"].items():
            assert v <= LIVE_TOL[adapter], (adapter, k, v)
        print(f"{adapter}: {L} x {g['reward'].shape[0]} reference lanes, one-step <= 1e-12, free-running worst state "
              f"{res['worst']['state']:.1e} (median lane {np.median(res['lane_state']):.1e}), live {res['live_fraction']:.2f}")
