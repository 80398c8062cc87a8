"""Table builder (fleetrl_b200/tables.py) vs the `db` the unmodified reference DataLoader built, as stored in the golden
fixtures whose fleet comes from the product's own seeded generator (oracle/gen_golden.py, `generated`).

The fleet is regenerated from that seed and written in the reference's CSV dialects; the builder reading those files must
give every constant and every table column the reference held, bit for bit, over the fixture's window of the year.
"""
import numpy as np
import pytest

from golden_util import Golden, golden_names

GENERATED = [n for n in golden_names() if Golden(n).meta.get("generated") is not None]
WINDOW_KEYS = ("table_len", "auto_reset", "start_lo", "start_hi", "seed", "carry_degradation_state")


def test_generated_fixtures_present():
    assert len(GENERATED) >= 4


@pytest.mark.parametrize("name", GENERATED)
def test_builder_matches_stored_reference_db(name, tmp_path):
    from fleetrl_b200.schedule import generate_schedule, synthetic_series, write_reference_csvs
    from fleetrl_b200.tables import build_fleet

    g = Golden(name)
    seed, (w0, w1) = g.meta["generated"], g.meta["window"]
    n_evs = g.consts_dict["num_evs"]
    cfg = dict(g.meta["cfg"])
    sched = generate_schedule(cfg["use_case"], n_evs, seed=seed)
    price, tariff, load, pv = synthetic_series(seed=seed + 1)
    cfg.update(write_reference_csvs(str(tmp_path), f"{n_evs}_{name}.csv", sched, price, tariff, load, pv))

    built = build_fleet(cfg, auto_reset=False)
    mine = built.consts.to_dict()
    for k, v in g.consts_dict.items():
        if k not in WINDOW_KEYS:
            assert mine[k] == v, f"const {k}: {mine[k]!r} != {v!r}"
    for k, v in g.tables.items():
        b = np.asarray(built.tables[k])
        b = b[:, w0:w1] if k in ("there", "time_left", "soc_on_return") else b[w0:w1]
        np.testing.assert_array_equal(b, v, err_msg=f"table {k}")
    for start, t in zip(g.meta["starts"], g.start_idx):
        assert int(np.searchsorted(built.dates, np.datetime64(start))) == w0 + int(t), start
