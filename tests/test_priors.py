"""priors.py against the reference's own load_sp_flex / lookup_sp_flex (golden priors.json)."""
import json
import os

import pytest

from conftest import GOLDEN, NO_REFERENCE, REFERENCE, has_reference
from fast_monte_carlo_b200 import priors


@pytest.fixture(scope="module")
def golden():
    return json.load(open(os.path.join(GOLDEN, "priors.json")))


def test_packaged_table_matches_reference_loader(golden):
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    rows = [dict(team=r.team, RATING=r.RATING, OFFENSE=r.OFFENSE, DEFENSE=r.DEFENSE, norm_team=r.norm_team)
            for r in sp.itertuples()]
    assert rows == golden["table"]


def test_lookups_and_errors(golden):
    sp = priors.load_sp_flex(priors.packaged_priors_path())
    for q, want in golden["lookups"].items():
        if isinstance(want, dict):
            with pytest.raises(ValueError) as e:
                priors.lookup_sp_flex(q, sp)
            assert str(e.value) == want["error"]
        else:
            assert list(priors.lookup_sp_flex(q, sp)) == want


def test_csv_base(golden):
    for k, want in golden["csv_base"].items():
        a, b, w = k.split("|")
        assert priors.csv_base_from(a, b, int(w)) == want


def test_schema_b_with_bom_and_aliases(tmp_path):
    p = tmp_path / "sp.csv"
    p.write_bytes("﻿Current SP+,Past SP+,Rating,Offense Rating,Defense Rating\r\n"
                  "App State,Appalachian State,-8.8,24.1,32.9\r\nAlabama,Alabama,27.9,40.4,12.6\r\n"
                  " UTSA ,UT San Antonio,0,28.0,27.5\r\n".encode("utf-8"))
    sp = priors.load_sp_flex(str(p))
    assert list(sp["team"]) == ["App State", "Alabama", "UTSA", "Appalachian State", "UT San Antonio"]
    assert priors.lookup_sp_flex("appalachian state", sp) == (-8.8, 24.1, 32.9)
    assert priors.lookup_sp_flex("utsa", sp) == (0.0, 28.0, 27.5)
    ctx = priors.build_team_context_from_sp_flex("Alabama", 2025, 1, sp)
    assert (ctx.sp_rating, ctx.sp_offense, ctx.sp_defense) == (27.9, 40.4, 12.6)
    assert list(ctx.qb_share["passer_name"]) == ["Unknown"] and ctx.track_pass == set()


def test_bad_schema(tmp_path):
    p = tmp_path / "bad.csv"
    p.write_text("a,b\n1,2\n")
    with pytest.raises(ValueError, match="Unrecognized SP\\+ schema"):
        priors.load_sp_flex(str(p))


@pytest.mark.skipif(not has_reference("PregameSPPlus2025_1.csv"), reason=NO_REFERENCE)
def test_real_csv(golden):
    sp = priors.load_sp_flex(os.path.join(REFERENCE, "PregameSPPlus2025_1.csv"))
    assert [r.team for r in sp.itertuples()] == [r["team"] for r in golden["table"]]
    assert priors.lookup_sp_flex("Kansas State", sp) == (15.6, 35.7, 20.0)
