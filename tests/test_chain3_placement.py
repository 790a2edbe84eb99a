"""k_chain3's warp placement (kernel_chain3.cu placeChain3Warps, DESIGN.md 4.2a): C2's unit-gain saving has to reach its busiest
sub-partition, and a CTA that a per-stream coefficient row sends back to the general form must run no worse than a program
without unit-gain parts.  Host-only, through the placement line of avdsp_b200_describe."""
import re

import numpy as np
import pytest

from conftest import load_program
import avdsp_b200

C2, FS = "c2_testrpi_xover_f2_192k", 192000


def _placement(trace):
    ln = [ln for ln in trace.splitlines() if ln.startswith("chain kernel v3 placement")][0]
    macs = re.search(r"IMAD.WIDE per frame on sub-partitions 0-3: (\d+) (\d+) (\d+) (\d+), every part general: (\d+) (\d+) (\d+) (\d+)", ln)
    bins = [int(b) for b in re.search(r"sub-partition of each item ([0-9,]+)", ln).group(1).split(",")]
    return [int(v) for v in macs.groups()[:4]], [int(v) for v in macs.groups()[4:]], bins


def _general(words):
    """b2 of every unit-gain section one LSB up: the same program shape with no part in the unit-gain form"""
    w = np.array(words, dtype=np.int32)
    for c in avdsp_b200.coef_words(w, 2).reshape(-1, 5):
        b0, b1, b2, a1, a2 = (int(w[i]) for i in c)
        if b0 == 1 << 28 and b1 + a1 == -(1 << 28) and b2 + a2 == 0:
            w[c[2]] += 1
    return w


def test_c2_gets_the_fastest_measured_placement():
    """(4uT,3u,4,helper) x 2 + (3,4u,3,3) x 2: 1.920 ms per call in the sweep against 2.058 for the placement that priced a unit
    section at 4 (31 31 56 56) and 2.00-2.03 for the four placements whose busiest sub-partition executes 44"""
    t = avdsp_b200.describe(load_program(C2), FS, 2, n_streams=4096, num_sms=148)
    macs, general, bins = _placement(t)
    assert sum(macs) == 174 and sum(general) == 240
    assert sorted(macs) == [34, 34, 53, 53], macs
    ln = [ln for ln in t.splitlines() if ln.startswith("chain kernel v3 placement")][0]
    items = re.findall(r" ([0-9]+[uTg]*|d|s):\d+\+\d+", ln)
    shape = sorted(tuple(sorted(items[k] for k in range(len(items)) if bins[k] == q)) for q in range(4))
    assert shape == sorted([("3u", "4", "4uT", "d"), ("3u", "4", "4uT", "s"), ("3", "3", "3", "4u"), ("3", "3", "3", "4u")]), shape


def test_c2_all_general_fallback_is_no_worse_than_a_program_without_unit_parts():
    """every part voted back to the general form: the busiest sub-partition stays at 65 IMAD.WIDE, what the program with the
    identity broken in every section gets as its own placement"""
    _, general, _ = _placement(avdsp_b200.describe(load_program(C2), FS, 2, n_streams=4096, num_sms=148))
    own, own_general, _ = _placement(avdsp_b200.describe(_general(load_program(C2)), FS, 2, n_streams=4096, num_sms=148))
    assert own == own_general
    assert max(general) <= 65, general
    assert max(general) <= max(own), (general, own)


@pytest.mark.parametrize("prog,fmt,fs,bins", [("c3_peq16_f2_48k", 2, 48000, [0, 2, 3, 2, 1, 3, 0, 1, 2, 3, 0, 1]),
                                              ("c3_peq16_f3_48k", 3, 48000, [2, 0, 3, 2, 1, 3, 0, 1, 2, 3, 0, 1, 0])])
def test_programs_without_unit_gain_parts_keep_their_placement(prog, fmt, fs, bins):
    """C3 and C3-float: the section-cost placement, which ran faster on both than what the exact search on the prices picks"""
    macs, general, got = _placement(avdsp_b200.describe(load_program(prog), fs, fmt, n_streams=65536, num_sms=148))
    assert macs == general == [40, 40, 40, 40]
    assert got == bins


def test_placement_line_matches_the_geometry_line():
    """the placement line's sub-partition of each item is the one the v3 geometry line prints by sections"""
    t = avdsp_b200.describe(load_program(C2), FS, 2, n_streams=4096, num_sms=148)
    geo = [ln for ln in t.splitlines() if ln.startswith("chain kernel v3 geometry")][0]
    nsec = [int(n) for n in re.findall(r" \d+:\d+\+(\d+)@\d+", geo.split("parts (chain:first+n@base):")[1].split(";")[0])]
    _, _, bins = _placement(t)
    tokens = nsec + ["d", "s"]
    want = [sorted(str(tokens[k]) for k in range(len(bins)) if bins[k] == q) for q in range(4)]
    got = [sorted(b.split()) for b in geo.split("s = store warp):")[1].split("|")]
    assert got == want
