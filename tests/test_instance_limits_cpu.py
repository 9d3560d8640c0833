"""The instance limits on the CPU: what the scene generators of tools/instance_scenes.py reach (nesting depth 4,
65536 instances, traversal stacks of 28 / 32 entries and one past the cap), and the flattened layouts walked with the
reference's semantics (tests/flat_interp.py) against the oracle on every one of them."""
import numpy as np
import pytest

from nr_ray_tracer_b200 import api
from oracle import oracle as O
from tests import flat_interp, kat
from tools import instance_scenes as S


@pytest.mark.parametrize("depth,opt", [(d, o) for d in range(5) for o in ("plain", "spec", "pool", "textured", "motion")
                                       if o != "motion" or d >= 3])
def test_nested_scenes_reach_the_promised_depth_and_sizes(depth, opt):
    kw = {"spec": {"mesh": "spec"}, "pool": {"mesh": "pool"}, "textured": {"textured": True},
          "motion": {"motion": True}}.get(opt, {})
    g, levels = S.nested(depth, **kw)
    hs = api.HostScene(g)
    d = hs.desc
    lv = S.instance_levels(hs)
    want_inst = 3 * depth + max(0, depth - 2) + (opt == "pool")
    assert d.n_instances == want_inst and len(lv) == want_inst
    reached = max((max(v) + 1 for v in lv.values()), default=0)
    assert reached == max(depth, opt == "pool")
    # each level-k group is a space of its own: its instances are entered at exactly one level
    assert all(len(v) == 1 for v in lv.values())
    assert d.max_stack <= 32
    if opt == "spec":
        assert 64 <= d.n_nodes < 1024
    elif opt == "pool":
        assert d.n_nodes >= 1024
    else:
        assert d.n_nodes < 64 and S.binary_stack(hs) <= 32
    assert bool(d.sphere_speed) == (opt == "motion")
    # the innermost group is shared: its primitives occur at several levels from depth 3 on
    shared = [o for o, ls in levels.items() if len(ls) > 1]
    assert bool(shared) == (depth >= 3)
    if depth == 4:
        assert {l for o in shared for l in levels[o]} == {2, 3, 4}
    print(f"nested({depth}, {opt}): {d.n_nodes} nodes, {d.n_wnodes} four-slot nodes, {d.n_instances} instances, "
          f"max_stack {d.max_stack}")


def test_full_stack_scenes_reach_their_targets_exactly():
    for target in (28, 32):
        hs = api.HostScene(S.full_stack(target))
        assert hs.desc.max_stack == target
        assert max(max(v) for v in S.instance_levels(hs).values()) == 3       # four levels of instances
    lite = api.HostScene(S.lite_full_stack())
    assert lite.desc.n_nodes < 64
    bs = S.binary_stack(lite)
    assert bs == 24 and ((bs + 3) & ~3) == bs                               # no rounding slack in the LITE cap
    assert max(max(v) for v in S.instance_levels(lite).values()) == 3
    # one past the cap: the host builds it and reports the need; nrrt_scene_upload refuses it (GPU test)
    over = api.HostScene(S.full_stack(33))
    assert over.desc.max_stack == 33


@pytest.mark.parametrize("n_inner,level", [(65535, 1), (65534, 2), (65536, 1)])
def test_many_instances_ids_and_levels(n_inner, level):
    hs = api.HostScene(S.many_instances(n_inner, level))
    d = hs.desc
    assert d.n_instances == n_inner + level and d.max_stack <= 32
    lv = S.instance_levels(hs)
    assert len(lv) == d.n_instances
    fan = sorted(i for i, v in lv.items() if v == {level})
    assert fan == list(range(n_inner))                  # the fan takes ids 0 .. n_inner - 1, all at `level`
    assert lv[d.n_instances - 1] == {0}                 # the outermost wrapper is numbered last
    assert max(fan) >= 32768


def _check_layout_against_oracle(g, n_rand=120, n_aim=200, n_special=120, seed=0):
    rng = np.random.default_rng(seed)
    sp = kat.special_rays(g)
    rays = np.concatenate([kat.random_rays(g, n_rand, seed=seed + 3), kat.aimed_rays(g, n_aim, seed=seed + 4),
                           sp[rng.permutation(len(sp))[:n_special]]])
    ref, _ = O.OracleScene(g).trace_rays(rays)
    assert (ref["object"] != 0xFFFFFFFF).sum() >= 0.1 * len(rays)
    for bvh in ("reference", "sah"):
        hs = api.HostScene(g, bvh=bvh)   # FlatScene views its instance records: keep the scene alive
        assert hs.desc.max_stack <= 32, bvh   # both builds must upload (NRRT_STACK_CAP)
        fs = flat_interp.FlatScene(hs)
        for wide in (False, True):
            for i, r in enumerate(rays):
                h = flat_interp.trace(fs, r[:3], r[3:], tie_by_order=(bvh == "sah"), wide=wide)
                if ref["object"][i] == 0xFFFFFFFF:
                    assert h is None, (bvh, wide, i, r, h)
                else:
                    assert h is not None and h[1] == ref["object"][i] and h[0] == ref["t"][i], (bvh, wide, i, r, h, ref[i])


@pytest.mark.parametrize("name", list(S.all_scenes()))
def test_flat_layouts_give_the_oracle_hits_on_generated_scenes(name):
    """Binary and four-slot layouts, reference and SAH trees: zero mismatches against the oracle's hits, ties included
    (the coincident scenes tie on every ray that hits their pairs)."""
    _check_layout_against_oracle(S.all_scenes()[name]())


def test_flat_layouts_give_the_oracle_hits_with_65536_instances():
    _check_layout_against_oracle(S.many_instances(65534, 2), n_rand=40, n_aim=120, n_special=40)


@pytest.mark.parametrize("split", [2, 3])
def test_coincident_pairs_tie_and_the_later_one_wins(split):
    g, pairs = S.coincident_across_levels(split)
    hs = api.HostScene(g)
    lv = S.instance_levels(hs)
    assert max(max(v) for v in lv.values()) == split        # the two chains part at level `split`
    osc = O.OracleScene(g)
    rays = kat.aimed_rays(g, 20000, seed=8)
    ref, _ = osc.trace_rays(rays)
    won = np.isin(ref["object"], pairs["later"])
    assert won.sum() > 100 and not np.isin(ref["object"], pairs["first"]).any()
    g0, _ = S.coincident_across_levels(split, with_later=False)
    alone, _ = O.OracleScene(g0).trace_rays(rays[won])
    assert np.isin(alone["object"], pairs["first"]).all() and np.array_equal(alone["t"], ref["t"][won])
