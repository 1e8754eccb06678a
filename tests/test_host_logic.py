"""Host-side logic that needs no GPU: the mmcv import shim, operator surface, anti-noise sampling
protocol and the parameters evaluated on the host."""
import importlib
import inspect
import sys

import numpy as np
import pytest
import torch

from cim_b200 import heads, integration, ops, synth
from oracle import heads_oracle


def test_mmcv_shim_resolves_reference_import_line():
    integration.install_mmcv_shim()
    for m in [k for k in sys.modules if k == "mmcv" or k.startswith("mmcv.")]:
        del sys.modules[m]
    mod = importlib.import_module("mmcv.ops")
    # lib/ops/__init__.py:6 of the reference
    from mmcv.ops import RoIPool, RoIAlign, roi_pool, roi_align, nms, soft_nms  # noqa: F401
    assert mod.RoIAlign is ops.RoIAlign and mod.RoIPool is ops.RoIPool


def test_roi_module_signatures_match_mmcv():
    sig = inspect.signature(ops.RoIAlign.__init__)
    assert list(sig.parameters)[1:] == ["output_size", "spatial_scale", "sampling_ratio", "pool_mode", "aligned",
                                        "use_torchvision"]
    assert sig.parameters["aligned"].default is True and sig.parameters["sampling_ratio"].default == 0
    m = ops.RoIAlign(7, 1.0 / 16, 0)          # the positional call of model_builder.py:230-231
    assert m.output_size == (7, 7) and m.aligned is True and not list(m.parameters())
    p = ops.RoIPool(7, 1.0 / 16)              # model_builder.py:228
    assert p.output_size == (7, 7)


def test_heads_surface_matches_reference_names():
    m = heads.cls_iou_model(32, 21, 3)
    names = sorted(n for n, _ in m.named_parameters())
    want = sorted([f"{p}.{s}" for p in ["classifier", "detector"] + [f"refine_cls.{k}" for k in range(3)] +
                   [f"refine_iou.{k}" for k in range(3)] for s in ("weight", "bias")])
    assert names == want
    mapping, orphans = m.detectron_weight_mapping()
    assert sorted(mapping) == want and orphans == []
    layer = heads.CIM_layer(p_seed=0.1, cls_thr=0.35, iou_thr=0.6, Anti_noise_sampling=False)
    assert layer.nms_thr == layer.cls_thr == 0.35 and layer.con_thr == 0.85
    assert list(inspect.signature(layer.forward).parameters) == [
        "predict_cls", "predict_det", "rois", "labels", "iou_map", "asy_iou_map", "using_CIM"]


def test_anti_noise_sampling_consumes_rng_like_the_oracle():
    rng = np.random.RandomState(5)
    gt_cls = rng.randint(0, 4, 40)
    gt_w = rng.rand(40).astype(np.float32)
    labels = np.zeros(20, np.float32)
    labels[[0, 2, 3, 7]] = 1                      # class 1 is mined but "absent": must be left alone
    np.random.seed(3)
    a = heads._anti_noise_keep(gt_cls, gt_w, np.nonzero(labels)[0])
    after_a = np.random.rand()
    np.random.seed(3)
    b = heads_oracle.anti_noise_keep(gt_cls, gt_w, labels)
    after_b = np.random.rand()
    assert a.astype(bool).tolist() == b.tolist() and after_a == after_b
    assert a[gt_cls == 1].all()


def test_anti_noise_draw_equals_numpy_choice_on_many_cases():
    """The spelled-out draw of heads._anti_noise_keep against np.random.choice itself (what the reference calls,
    heads.py:459, and what the oracle calls): same survivors, same RNG state afterwards, over sizes from one
    pseudo GT to several hundred, skewed and near-degenerate weights included."""
    rng = np.random.RandomState(17)
    for case in range(300):
        g = int(rng.choice([1, 2, 3, 7, 40, 200, 800]))
        n_cls = int(rng.randint(1, 6))
        gt_cls = rng.randint(0, n_cls, g)
        gt_w = rng.rand(g).astype(np.float32) ** int(rng.choice([1, 4, 12]))
        gt_w = np.maximum(gt_w, np.float32(1e-30))
        labels = np.zeros(20, np.float32)
        labels[:n_cls] = 1
        np.random.seed(case)
        a = heads._anti_noise_keep(gt_cls, gt_w, np.nonzero(labels)[0])
        state_a = np.random.get_state()[1].copy(), np.random.get_state()[2]
        np.random.seed(case)
        b = heads_oracle.anti_noise_keep(gt_cls, gt_w, labels)
        state_b = np.random.get_state()[1].copy(), np.random.get_state()[2]
        assert a.astype(bool).tolist() == b.tolist(), case
        assert state_a[1] == state_b[1] and np.array_equal(state_a[0], state_b[0]), case


def _zero_weight_groups(rng, n_cases):
    """Pseudo-GT lists whose class groups hold exact zeros (det underflowed), all-equal weights and a single non-zero
    weight among zeros; no group is all zero."""
    cases = []
    for _ in range(n_cases):
        g = int(rng.choice([2, 3, 9, 40, 130, 600]))
        gt_cls = rng.randint(0, 3, g)
        kind = int(rng.randint(3))
        if kind == 0:                                              # some zeros, anywhere (first and last included)
            gt_w = rng.rand(g).astype(np.float32) * (rng.rand(g) < 0.5)
        elif kind == 1:                                            # all equal
            gt_w = np.full(g, np.float32(rng.choice([1.0, 0.0625, 1e-30])), np.float32)
        else:                                                      # one non-zero weight per class
            gt_w = np.zeros(g, np.float32)
        for c in range(3):
            idx = np.nonzero(gt_cls == c)[0]
            if len(idx) and gt_w[idx].sum() == 0:
                gt_w[idx[rng.randint(len(idx))]] = np.float32(rng.rand() + 1e-3)
        cases.append((gt_cls, gt_w.astype(np.float32)))
    return cases


def test_anti_noise_draw_equals_numpy_choice_with_zero_weights():
    """Zero weights are legal input for np.random.choice (heads.py:459) as long as a class's weights do not all
    vanish: the host draw must pick what choice picks and consume what it consumes."""
    rng = np.random.RandomState(31)
    cases = _zero_weight_groups(rng, 200)
    assert sum(int((w == 0).sum()) for _, w in cases) > 1000
    assert any(len(np.unique(w)) == 1 and len(w) > 1 for _, w in cases)
    assert any(np.count_nonzero(w[c == 0]) == 1 and (c == 0).sum() > 3 for c, w in cases)
    labels = np.zeros(20, np.float32)
    labels[:3] = 1
    for case, (gt_cls, gt_w) in enumerate(cases):
        np.random.seed(case)
        a = heads._anti_noise_keep(gt_cls, gt_w, np.nonzero(labels)[0])
        state_a = np.random.get_state()
        np.random.seed(case)
        b = heads_oracle.anti_noise_keep(gt_cls, gt_w, labels)
        state_b = np.random.get_state()
        assert a.astype(bool).tolist() == b.tolist(), case
        assert state_a[2] == state_b[2] and np.array_equal(state_a[1], state_b[1]), case
        assert not a[gt_w == 0].any(), case                          # a zero-weight pseudo GT is never drawn


def test_anti_noise_all_zero_group_keeps_first_gt_and_consumes_the_stream():
    """A class whose pseudo GTs all have weight 0: np.random.choice raises (the reference stops), the host keeps the
    class's first pseudo GT, consumes the class's n doubles, and draws the other classes as choice does."""
    gt_cls = np.array([0, 1, 1, 2, 1, 0, 1, 2, 2], np.int64)
    gt_w = np.array([0.5, 0, 0, 0.25, 0, 0.125, 0, 0, 0.75], np.float32)
    present = np.array([0, 1, 2])
    with np.errstate(invalid="ignore"):
        with pytest.raises(ValueError):
            np.random.choice(np.nonzero(gt_cls == 1)[0], 4, replace=True, p=gt_w[gt_cls == 1] / gt_w[gt_cls == 1].sum())
        np.random.seed(7)
        keep = heads._anti_noise_keep(gt_cls, gt_w, present)
    state = np.random.get_state()
    assert keep[gt_cls == 1].tolist() == [1, 0, 0, 0] and keep[1] == 1
    np.random.seed(7)
    want = np.ones(len(gt_cls), np.uint8)
    for c in present:
        idx = np.nonzero(gt_cls == c)[0]
        if c == 1:
            np.random.random_sample(len(idx))
            want[idx] = 0
            want[idx[0]] = 1
            continue
        drawn = np.random.choice(idx, len(idx), replace=True, p=gt_w[idx] / gt_w[idx].sum())
        want[idx] = 0
        want[drawn] = 1
    assert keep.tolist() == want.tolist()
    want_state = np.random.get_state()
    assert state[2] == want_state[2] and np.array_equal(state[1], want_state[1])
    np.random.seed(7)
    np.random.random_sample(len(gt_cls))
    assert np.array_equal(np.random.get_state()[1], state[1])      # exactly n doubles per class, n summed


def test_one_random_sample_call_is_the_stream_of_the_per_class_choice_calls():
    """heads.draw_uniforms: ONE random_sample(T) call hands out the doubles the reference's per-(image, layer, class)
    np.random.choice calls consume, in the same order, and leaves the global RNG in the same state; with those doubles
    the device algorithm (restated here: float32 p, float64 cumsum / last, searchsorted right) picks what choice picks."""
    rng = np.random.RandomState(23)
    lists = []
    for _ in range(12):                                        # (image, layer) lists in the reference's order
        g = int(rng.choice([0, 1, 5, 60, 300]))
        lists.append((rng.randint(0, 3, g), np.maximum(rng.rand(g).astype(np.float32) ** 3, np.float32(1e-20))))
    present = np.array([0, 1, 2])
    np.random.seed(11)
    want = [heads._anti_noise_keep(c, w, present) for c, w in lists]
    state_want = np.random.get_state()
    np.random.seed(11)
    u = heads.draw_uniforms(np.array([len(c) for c, _ in lists]))
    state_got = np.random.get_state()
    assert state_want[2] == state_got[2] and np.array_equal(state_want[1], state_got[1])
    off = 0
    for (cls, w), keep_want in zip(lists, want):
        keep = np.ones(len(cls), np.uint8)
        for c in present:
            idx = np.nonzero(cls == c)[0]
            if len(idx) == 0:
                continue
            p = w[idx] / w[idx].sum()
            cdf = p.astype(np.float64).cumsum()
            cdf /= cdf[-1]
            drawn = idx[np.searchsorted(cdf, u[off:off + len(idx)], side="right")]
            off += len(idx)
            keep[idx] = 0
            keep[drawn] = 1
        assert keep.tolist() == keep_want.tolist()
    assert off == len(u)


def test_host_evaluated_parameters():
    for r in (64, 300, 2000, 4000, 257):
        assert int(np.ceil(0.1 * r)) == {64: 7, 300: 30, 2000: 200, 4000: 400, 257: 26}[r]
    assert float(np.float32(0.9 * 300)) == 270.0


def test_synth_is_deterministic_and_nested():
    p = synth.proposal_params(130, size=64, seed=9)
    m1, m2 = synth.rasterize(p), synth.rasterize(p, chunk=7)
    assert torch.equal(m1, m2) and m1.dtype == torch.uint8 and m1.sum((1, 2)).min() > 0
    rois = synth.rois_from_params(p)
    ys, xs = torch.nonzero(m1[3], as_tuple=True)
    assert rois[3].tolist() == [0, xs.min(), ys.min(), xs.max() + 1, ys.max() + 1]
    # proposals 5 and 5+64 share a seed ellipse: one contains the other
    a, b = m1[5].bool(), m1[69].bool()
    inter = (a & b).sum()
    assert inter == min(a.sum(), b.sum())
    down = synth.rasterize(p, out_size=16)
    assert torch.equal(down, m1[:, ::4, ::4])


def test_uniform_stream_hands_out_numpys_global_stream_and_commits_it():
    """heads.UniformStream (the host half of the sync-free sampling mode): the doubles drawn ahead are numpy's global
    stream in order, consumption is learned with a lag, commit() leaves np.random where per-step draws would have,
    and foreign draws between commit() and the next step keep their place in the stream."""
    from cim_b200.heads import UniformStream
    M = 50
    rng = np.random.RandomState(7)
    counts = rng.randint(0, M + 1, size=40)
    # reference: every step draws its own count from the global generator; a foreign draw after step 24
    np.random.seed(11)
    want = []
    for i, c in enumerate(counts):
        want.append(np.random.random_sample(c))
        if i == 24:
            foreign_want = np.random.random_sample(3)
    state_want = np.random.get_state()[1].copy()

    np.random.seed(11)
    us = UniformStream(16 * M, M)
    ring = np.full(us.ring_len, np.nan)
    inflight, got, cursor = [], [], 0
    for i, c in enumerate(counts):
        while len(inflight) > 1:                               # lagged read-back: at most 2 steps unknown
            us.note_consumed(inflight.pop(0))
        if not us.attached:
            us.attach()
        inflight.append(int(c))
        n = us.need(len(inflight))
        if n:
            pos, u = us.draw(n)
            assert pos + n - us.ring_len <= us.consumed        # only consumed slots are overwritten
            ring[(pos + np.arange(n)) % us.ring_len] = u
        assert cursor + c <= us.drawn
        got.append(ring[(cursor + np.arange(c)) % us.ring_len].copy())   # what the device kernel reads
        cursor += c
        if i == 24:
            while inflight:
                us.note_consumed(inflight.pop(0))
            us.commit()
            assert not us.attached
            foreign = np.random.random_sample(3)
            np.testing.assert_array_equal(foreign, foreign_want)
        if i == 10:                                            # a commit nobody draws after: the reserve is kept
            while inflight:
                us.note_consumed(inflight.pop(0))
            drawn_before = us.drawn
            us.commit()
            assert not us.attached
            us.attach()
            assert us.attached and us.drawn == drawn_before
    while inflight:
        us.note_consumed(inflight.pop(0))
    us.commit()
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g, w)
    assert np.array_equal(np.random.get_state()[1], state_want)
    assert us.consumed == us.committed == cursor


def test_rank_core_plan_follows_the_gpus_numa_node():
    """dist.plan_rank_cores: ranks take slices of the cores of THEIR GPU's NUMA node when it is known and usable,
    else equal slices of all usable cores (containers whose cpuset does not reach the other socket)."""
    from cim_b200 import dist as cdist
    assert cdist._parse_cpulist("0-3,8,10-11\n") == [0, 1, 2, 3, 8, 10, 11]
    nodes = [0, 0, 0, 0, 1, 1, 1, 1]
    cpus = {0: list(range(0, 32)), 1: list(range(32, 64))}
    plan = [cdist.plan_rank_cores(r, 8, range(64), nodes, cpus) for r in range(8)]
    assert plan[0] == list(range(0, 8)) and plan[3] == list(range(24, 32)) and plan[4] == list(range(32, 40))
    assert sorted(sum(plan, [])) == list(range(64))                       # disjoint, complete
    # the cpuset only holds node 0's cores: every rank falls back to disjoint slices of what is usable
    plan = [cdist.plan_rank_cores(r, 8, range(16), nodes, cpus) for r in range(8)]
    assert plan[1] == [2, 3] and plan[5] == [10, 11] and sorted(sum(plan, [])) == list(range(16))
    # unknown nodes, fewer cores than ranks
    assert cdist.plan_rank_cores(2, 4, range(8), [-1] * 4, {}) == [4, 5]
    assert cdist.plan_rank_cores(0, 8, range(4), [-1] * 8, {}) is None


def test_bench_dump_outputs_writes_whole_or_fixed_sample(tmp_path):
    """bench.py --dump-outputs: small results whole, larger ones as the same seeded sample every run, all float32,
    numpy's global generator (the step's anti-noise sampling) untouched."""
    import types
    import bench
    n = bench.DUMP_ELEMS
    g = torch.Generator().manual_seed(0)
    step = types.SimpleNamespace(head_grads=False, **{name: torch.randn(3, 7, generator=g)
                                                      for name in bench.STEP_OUTPUTS})
    step.roi_out = torch.arange(2 * n + 6, dtype=torch.float32).view(-1, 2)     # value = flat index
    step.iou = torch.rand(4, 5, generator=g).half()
    step.valid = torch.tensor([[1, 0]], dtype=torch.uint8)
    np.random.seed(5)
    state = np.random.get_state()[1].copy()
    bench.dump_outputs(step, str(tmp_path / "a"))
    bench.dump_outputs(step, str(tmp_path / "b"))
    assert np.array_equal(np.random.get_state()[1], state)
    assert sorted(p.name for p in (tmp_path / "a").iterdir()) == sorted(f"{s}.npy" for s in bench.STEP_OUTPUTS)
    for name in bench.STEP_OUTPUTS:
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, b)
        full = getattr(step, name).float().reshape(-1).numpy()
        if name == "roi_out":
            np.testing.assert_array_equal(a, bench.dump_indices(full.size))
        else:
            np.testing.assert_array_equal(a, full)
