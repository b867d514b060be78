"""Known-answer vectors for InterpolatedIdentity::interpolate_identities (linnaean_ranks.rs:220-383),
SURVEY.md section 3.3, checked on BOTH oracle restatements (Python mirror and C++)."""
import pytest

import pyoracle as po
from helpers import CUTOFFS_16S, KAT, same
from oracle_ffi import interpolate as c_interpolate

@pytest.mark.parametrize("ranks,bact,cust", KAT)
def test_interpolation_kat(ranks, bact, cust):
    names = ranks.split()
    pr = [po.rank_from_str(x) for x in names]
    assert same(po.interpolate(pr, po.backbone_for("bacteria")), [float(x) for x in bact])
    assert same(po.interpolate(pr, po.backbone_for("custom", CUTOFFS_16S)), [float(x) for x in cust])
    assert same(c_interpolate(names, "bacteria"), [float(x) for x in bact])
    assert same(c_interpolate(names, "custom", CUTOFFS_16S), [float(x) for x in cust])


def test_fungi_equals_eukaryotes():
    names = "d clade p c o f g s strain".split()
    assert c_interpolate(names, "fungi") == c_interpolate(names, "eukaryotes") == [60.0, 67.5, 75.0, 80.0, 85.0, 90.0, 95.0, 97.0, 100.0]


def test_rank_parsing():
    assert po.rank_from_str(" Phylum ") == ("D", "phylum")
    assert po.rank_from_str("S") == ("D", "species")
    assert po.rank_from_str("species group") == ("O", "species-group")
    assert po.rank_from_str("Sub_Order!") == ("O", "sub-order")
    assert po.rank_display(("D", "undefined")) == "u"
    with pytest.raises(po.DataError):
        po.rank_from_str("--")


def test_ryu_format():
    f = po.ryu_f64
    assert f(845.0) == "845.0" and f(99.356) == "99.356" and f(0.001) == "0.001" and f(1e-5) == "0.00001"
    assert f(1e-6) == "1e-6" and f(1.5e-7) == "1.5e-7" and f(1e16) == "1e16" and f(1.2345e20) == "1.2345e20"
    assert f(1e15) == "1000000000000000.0" and f(123456789012345680.0) == "1.2345678901234568e17" and f(-2.5) == "-2.5"
