"""Host-side launch planning (b200dn_igemm_plan: no GPU touched): every layer shape of the three network widths, at the
BASELINE batch sizes and at batch 1-2, plus a sweep of odd shapes, must get a configuration that fits the kernels'
shared-memory and TMEM budgets.  The dispatch rules DESIGN.md states are pinned for the headline layers."""
import itertools
import json
import os
import subprocess
import sys
from pathlib import Path

import pytest

import dispatch_configs
from helpers import SMS, dispatch_rows, network_layers, plan, render_dispatch_configs
from vub_image_denoising_b200 import _lib

TESTS = Path(__file__).resolve().parent


def check_budgets(i, what):
    assert i.data_bytes_used <= i.data_bytes_budget, f"{what}: {i.data_bytes_used} B of rings > {i.data_bytes_budget}"
    assert 32 <= i.tmem_cols <= 512 and i.tmem_cols & (i.tmem_cols - 1) == 0, f"{what}: tmem_cols {i.tmem_cols}"
    assert i.tmem_cols >= 2 * i.mt * i.block_n, f"{what}: two accumulator stages do not fit {i.tmem_cols} columns"
    assert i.block_n % 16 == 0 and 16 <= i.block_n <= 256, what
    assert i.mt in (1, 2) and i.num_tiles >= 1 and 1 <= i.grid <= SMS, f"{what}: grid {i.grid}"
    if i.kernel == 2:
        assert i.grid % 2 == 0 and not i.wres and i.block_n >= 32, what
    if i.kernel in (1, 2):
        assert i.num_slabs >= 2 or (i.wres and i.num_slabs >= 1), f"{what}: {i.num_slabs} slab(s)"
        assert i.num_slabs <= 6 and i.slab_bytes % 1024 == 0, what
        if not i.wres:
            assert 2 <= i.num_stages <= 8 and i.stage_bytes % 1024 == 0, f"{what}: W ring {i.num_stages} x {i.stage_bytes}"
    else:
        assert 2 <= i.num_stages <= 8, f"{what}: ring of {i.num_stages}"


@pytest.mark.parametrize("F,B", [(128, 64), (128, 1), (128, 2), (64, 64), (64, 1), (32, 32), (32, 2), (32, 4), (16, 3), (48, 5)])
def test_every_network_layer_fits(F, B, built_lib):
    layers = network_layers(F, B)
    assert len(layers) == 68
    for prec in (_lib.PREC_BF16, _lib.PREC_FP16X2, _lib.PREC_BF16X3):
        for L in layers:
            i = plan(L.mode, L.B, L.H, L.W, L.cin, L.cout, prec=prec, in_ctot=L.in_ctot, out_ctot=L.out_ctot,
                     coff=L.coff, nchw=L.nchw)
            check_budgets(i, f"F={F} B={B} prec={prec} mode={L.mode} {L.H}x{L.W} {L.cin}->{L.cout}")


def test_shape_sweep_fits(built_lib):
    n = 0
    for cin, cout, hw, B, impl in itertools.product((8, 16, 24, 48, 80, 96, 160, 200, 320, 640, 1000, 2560),
                                                    (8, 16, 24, 40, 64, 72, 128, 200, 256, 512, 1024),
                                                    ((8, 8), (16, 24), (40, 56), (128, 128), (256, 256)), (1, 3, 64), (0, 1, 2, 3)):
        i = plan(0, B, hw[0], hw[1], cin, cout, impl=impl)
        check_budgets(i, f"conv3x3 impl={impl} B={B} {hw} {cin}->{cout}")
        n += 1
    for cin, hw, B in itertools.product((16, 64, 208, 512, 1024), ((8, 8), (24, 40), (128, 128)), (1, 5, 64)):
        check_budgets(plan(1, B, hw[0], hw[1], cin, 2 * cin), f"down {cin}")
        check_budgets(plan(2, B, hw[0], hw[1], cin, cin, out_ctot=cin // 2 + cin, coff=cin // 2), f"up {cin}")
        n += 2
    assert n > 7000


def test_dispatch_rules_of_the_headline_layers(built_lib):
    # BASELINE config 2 (F = 128, B = 64): growth convs (N = 64) and conv_3 (N = 128) at level 0 run on CTA pairs with
    # two sub-tiles per CTA and a filter row per W stage for N = 64; level-3 convs (N = 256 tiles) with one sub-tile
    i = plan(0, 64, 256, 256, 128, 64, in_ctot=320, out_ctot=320, coff=128)
    assert (i.kernel, i.mt, i.block_n, i.w_taps, i.grid) == (2, 2, 64, 3, 148)
    i = plan(0, 64, 256, 256, 320, 128, in_ctot=320, out_ctot=320)
    assert (i.kernel, i.mt, i.block_n, i.w_taps) == (2, 2, 128, 1)
    i = plan(0, 64, 32, 32, 2560, 1024, in_ctot=2560, out_ctot=2560)
    assert (i.kernel, i.mt, i.block_n, i.num_n_tiles) == (2, 1, 256, 4)
    # the F = 32 network's level-0 growth convs keep their weights resident; the output conv pads N 3 -> 16
    i = plan(0, 32, 256, 256, 32, 16, prec=_lib.PREC_FP16, in_ctot=80, out_ctot=80, coff=32)
    assert (i.kernel, i.wres, i.mt, i.block_n) == (1, 1, 2, 16) and i.num_slabs >= 3
    i = plan(0, 64, 256, 256, 128, 3, in_ctot=128, nchw=True)
    assert (i.kernel, i.wres, i.block_n) == (1, 1, 16)
    # batch 1: the level-3 conv splits N down to 64 and still uses CTA pairs (under-filled grid)
    i = plan(0, 1, 32, 32, 2560, 1024, in_ctot=2560, out_ctot=2560)
    assert (i.kernel, i.block_n, i.num_n_tiles) == (2, 64, 16) and i.grid == 2 * 4 * 16
    # explicit implementations are honoured; a layer with one pixel tile cannot pair
    assert plan(0, 2, 32, 32, 128, 64, impl=1).kernel == 0
    assert plan(0, 2, 32, 32, 128, 64, impl=2).kernel == 1
    assert plan(0, 2, 32, 32, 128, 64, impl=3).kernel == 2
    assert plan(0, 1, 16, 8, 128, 64).kernel == 1
    # down / up convs run on the per-tap kernel
    assert plan(1, 64, 256, 256, 128, 256, in_ctot=384).kernel == 0
    assert plan(2, 64, 128, 128, 256, 256, in_ctot=640, out_ctot=384, coff=128).kernel == 0


def test_plan_rejects_what_launch_rejects(built_lib):
    with pytest.raises(RuntimeError, match="in_ctot"):
        plan(0, 1, 8, 8, 16, 16, in_ctot=20)
    with pytest.raises(RuntimeError, match="even H, W"):
        plan(1, 1, 9, 8, 16, 32)
    with pytest.raises(RuntimeError, match="8-channel aligned"):
        plan(0, 1, 8, 8, 16, 12, out_ctot=16)
    with pytest.raises(RuntimeError, match="sm_count"):
        plan(0, 1, 8, 8, 16, 16, sms=0)


def _row_diff(want, have):
    added, removed = sorted(set(want) - set(have)), sorted(set(have) - set(want))
    lines = [f"+ {r!r}," for r in added] + [f"- {r!r}," for r in removed]
    return added, removed, "\n".join(lines)


def test_dispatch_table_matches_the_planner(built_lib):
    """tests/dispatch_configs.py lists every configuration the planner picks for the network, each with the layer that
    test_gpu_dispatch_parity.py checks it on.  A dispatch change that adds or drops a configuration fails here until the
    table is regenerated, so that every configuration the product runs keeps a parity row."""
    want = dispatch_rows()
    assert len(want) == len({r[:-4] for r in want})
    added, removed, diff = _row_diff(want, dispatch_configs.ROWS)
    assert not added and not removed, (
        f"the planner's configurations differ from tests/dispatch_configs.py ({len(added)} added, {len(removed)} "
        f"removed; regenerate with `python tests/dispatch_configs.py --write`):\n{diff}")
    assert (TESTS / "dispatch_configs.py").read_text() == render_dispatch_configs(want)


def test_dispatch_table_notices_a_dispatch_change(built_lib):
    """The same regeneration in a process where B200DN_SPLIT_N=256 turns off the under-filled-grid N split: the row set
    must change (the split-N rows of batch 1-2 disappear), i.e. the table test above fails on a dispatch change."""
    code = ("import json, sys; sys.path[:0] = [sys.argv[1], sys.argv[2]]; import helpers; "
            "print(json.dumps(helpers.dispatch_rows()))")
    env = dict(os.environ, B200DN_SPLIT_N="256")
    out = subprocess.run([sys.executable, "-c", code, str(TESTS), str(TESTS.parent)], env=env, check=True,
                         capture_output=True, text=True).stdout
    rows = [tuple(r) for r in json.loads(out.strip().splitlines()[-1])]
    added, removed, diff = _row_diff(rows, dispatch_configs.ROWS)
    assert added or removed, "B200DN_SPLIT_N=256 left the configuration table unchanged"
