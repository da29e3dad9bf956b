"""Every device-learned capacity of the default path grows through the repeat.  With option tiny_caps every capacity starts at its
minimum; each overflow shows in a TFBS_DEBUG repeat line as need > cap, and the block's rows, attribution, sites and record sites
equal those of a run with the usual capacities.  The block is chosen so that every capacity that can overflow does: many reference
hits per region (capr), several groups per region (groups), terms, and several sites per record (rsites).  The work list (items)
cannot: it is sized for the reference pieces plus one item per diff-list entry of the virtual sequences (vd), its bound while vd
fits, and its gate only checks that bound.

On the GPU through the product library; on the CPU the same run goes through the emulated kernels (tests/cuda_emu) in a subprocess."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from find_tfbs_b200 import binding, synth
from find_tfbs_b200.binding import PatternSet
import test_attribution as ta
import test_record_sites as tr
import test_sites as ts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "cuda_emu")
MODES = (binding.ROWS_VARYING, binding.ROWS_ALL_KEYS)
# the capacity table of the default path (Cap in find_tfbs_b200/csrc/k2c_configs.cuh), in the order of the repeat line
CAPS = ("seq", "d", "cfg", "vd", "items", "units", "dwords", "rows", "rowwords", "capr", "groups", "terms", "sites_raw", "sites", "rsites")
GROWN = set(CAPS) - {"items"}
REPEAT = re.compile(r"tfbs: block repeated \(attempt \d+\): collided \d+, need(.*) \| caps(.*)")


def case():
    """12 samples, 6 regions, loose thresholds (dozens of reference hits per region), a record every 10 bp, a fifth of them indels."""
    pats = synth.make_pwms(4, seed=7, lmin=6, lmax=12, pvalue=2e-2)
    lmax = max(p["weights"].shape[0] for p in pats)
    blk = synth.make_cohort(12, 6, seed=7, lmax_pattern=lmax, region_len=(150, 400), variant_rate=1 / 10.0, frac_ins=0.1, frac_del=0.1,
                            two_beds=True)
    return PatternSet(pats), blk


def run(ps, blk, mode, tiny):
    ctx = binding.Context(0)
    try:
        for k, v in (("rows_mode", mode), ("tiny_caps", tiny), ("attribution", 1), ("sites", 1), ("record_sites", 1)):
            ctx.set_option(k, v)
        ctx.set_patterns(ps)
        ctx.submit_block(blk)
        g = ta.own(ctx.collect_grouped(expand=True))
        return g, ctx.attribution(), ctx.sites(), ctx.record_sites()
    finally:
        ctx.close()


def check_block(mode):
    """tiny_caps against the usual capacities: the same rows, attribution, sites and record sites."""
    ps, blk = case()
    (g0, a0, s0, r0), (g1, a1, s1, r1) = run(ps, blk, mode, 0), run(ps, blk, mode, 1)
    for k in g0:
        if isinstance(g0[k], np.ndarray) and k not in ("offset", "packed"):
            assert np.array_equal(g0[k], g1[k]), k
    assert np.array_equal(ta.rows_packed(g0), ta.rows_packed(g1))
    assert len(g0["region"]) > 0 and a0["term_cfg"].size > 0 and s0["change"].size > 0 and r0["change"].size > 0
    ta.assert_same_attribution(a0, a1)
    ts.assert_same_sites(s0, s1)
    tr.assert_same_records(r0, r1)


def overflowed(stderr):
    """Capacities with need > cap in some repeat line; every line lists the whole table."""
    over = set()
    for need, caps in REPEAT.findall(stderr):
        need, caps = need.split(), caps.split()
        assert need[0::2] == list(CAPS) and caps[0::2] == list(CAPS), (need, caps)
        over |= {c for c, n, k in zip(CAPS, need[1::2], caps[1::2]) if int(n) > int(k)}
    return over


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_every_capacity_grows(mode, capfd, monkeypatch):
    monkeypatch.setenv("TFBS_DEBUG", "1")
    check_block(mode)
    assert overflowed(capfd.readouterr().err) == GROWN


@pytest.mark.parametrize("mode", MODES)
def test_every_capacity_grows_emulated(mode):
    subprocess.check_call(["make", "-C", EMU, "-j2", "libtfbs_emu.so"], stdout=subprocess.DEVNULL)
    env = dict(os.environ, TFBS_B200_LIB=os.path.join(EMU, "libtfbs_emu.so"), TFBS_DEBUG="1",
               PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests")]))
    code = "import test_capacities as t\nt.check_block(%d)\n" % mode
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert overflowed(r.stderr) == GROWN
