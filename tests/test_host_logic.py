"""CPU: host-side logic of the product that needs no GPU -- the conditioner-output contract (`_parse_params`), the
data-parallel batch schedule, the weight-cache epoch, argument validation, the drop-in import names."""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_split_params_follows_parse_params():
    """`MaskedAffineCoupling._parse_params` (`/root/reference/src/nf4ad/transforms.py:40-64`): (s, t) pair; tensor of x's
    shape = additive (s absent); 2C channels along dim 1; anything else is the reference's ValueError (same text)."""
    from nf4ad_b200.transforms import split_params
    x = torch.randn(4, 6)
    s, t = split_params((torch.ones(4, 6), torch.zeros(4, 6)), x)
    assert torch.equal(s, torch.ones(4, 6)) and torch.equal(t, torch.zeros(4, 6))
    s, t = split_params([torch.ones(4, 6).double(), torch.zeros(4, 6).double()], x)
    assert s.dtype == torch.float32 and t.dtype == torch.float32          # cast to x.dtype (:62-63)
    p = torch.randn(4, 6)
    s, t = split_params(p, x)
    assert s is None and torch.equal(t, p)                                # additive-only form (:46-49)
    p = torch.randn(4, 12)
    s, t = split_params(p, x)
    assert torch.equal(s, p[:, :6]) and torch.equal(t, p[:, 6:])          # 2C split (:52-55)
    xi, pi = torch.randn(2, 3, 5, 5), torch.randn(2, 6, 5, 5)             # image-shaped: channels are dim 1
    s, t = split_params(pi, xi)
    assert torch.equal(s, pi[:, :3]) and torch.equal(t, pi[:, 3:])
    for bad in (torch.randn(4, 7), torch.randn(4, 18), torch.randn(24)):
        with pytest.raises(ValueError, match="Conditioner output shape not compatible"):
            split_params(bad, x)


def test_unsupported_scale_activation_is_the_reference_error():
    from nf4ad_b200 import ops
    assert ops.scale_activation_id("exp") == 0 and ops.scale_activation_id("softplus") == 1
    with pytest.raises(ValueError, match="Unsupported scale_activation"):       # transforms.py:86-87
        ops.scale_activation_id("sigmoid")


def test_rank_batches_partition_the_reference_schedule():
    """Data parallel `fit`: the ranks' shards of every global batch are disjoint, cover it in order, differ by at most one
    row, and an epoch sees every sample once (`adbench_wrapper.py:364-377` is the single-process schedule)."""
    from nf4ad_b200.parallel import rank_batches, shard_bounds
    for n, bs, world in ((200, 32, 1), (200, 32, 2), (203, 32, 4), (64, 64, 8), (10, 4, 3), (5, 4, 8)):
        perm = torch.randperm(n, generator=torch.Generator().manual_seed(n))
        per_rank = [list(rank_batches(perm, bs, r, world)) for r in range(world)]
        steps = {len(b) for b in per_rank}
        assert len(steps) == 1                                   # every rank takes the same number of steps
        seen = []
        for step in range(steps.pop()):
            shards = [per_rank[r][step] for r in range(world)]
            sizes = [s.numel() for s in shards]
            assert max(sizes) - min(sizes) <= 1 and min(sizes) >= 1
            glob = torch.cat(shards)
            assert torch.equal(glob, perm[step * bs: step * bs + glob.numel()])
            seen.append(glob)
        seen = torch.cat(seen) if seen else torch.empty(0, dtype=torch.long)
        # only batches with fewer rows than ranks (un-shardable: normally just a short tail) are dropped
        kept = sum(min(bs, n - i) for i in range(0, n, bs) if min(bs, n - i) >= world or world == 1)
        assert seen.numel() == kept
        assert seen.unique().numel() == seen.numel()
    assert shard_bounds(10, 0, 3) == (0, 4) and shard_bounds(10, 2, 3) == (7, 10)


def test_weights_epoch_is_part_of_the_cache_key():
    """ADVICE r1 (high): optimizer steps that bypass torch's version counters (FusedAdam's raw-pointer kernel, a CUDA-graph
    replay) bump `_lib.weights_epoch()`, which is part of every flow's packed-weight key."""
    import nf4ad_b200
    from nf4ad_b200 import _lib
    from _cases import build_flow
    flow = build_flow(nf4ad_b200.namespace(), "NonUSFlow", 8, 2, ("mlp", [16]), affine_conjugation=True)
    k0 = flow._weights_key()
    assert flow._weights_key() == k0
    _lib.bump_weights_epoch()
    k1 = flow._weights_key()
    assert k1 != k0
    with torch.no_grad():
        flow.layers[-1].scale.mul_(2.0)          # eager in-place updates are seen through the version counter
    assert flow._weights_key() != k1


def test_optimizer_argument_validation():
    from nf4ad_b200.optim import FusedAdam, SophiaG
    p = [torch.nn.Parameter(torch.zeros(3))]
    for bad in (dict(lr=-1.0), dict(betas=(1.0, 0.9)), dict(weight_decay=-0.1)):
        with pytest.raises(ValueError):
            FusedAdam(p, **bad)
        with pytest.raises(ValueError):
            SophiaG(p, **bad)
    p[0].grad = torch.ones(3)
    for opt in (FusedAdam(p), SophiaG(p)):       # CPU parameters: no CPU path
        with pytest.raises(nf4ad_b200_error()):
            opt.step()


def nf4ad_b200_error():
    import nf4ad_b200
    return nf4ad_b200.USFError


def test_image_shaped_flow_builds_with_reference_layer_list():
    """`in_dims=[C, H, W]` (`nf4ad/flows.py:78-145`): same layer list and state_dict keys as the oracle, N-D masks."""
    import nf4ad_b200
    import oracle
    from _cases import build_flow
    P, O = nf4ad_b200.namespace(), oracle.load()
    for masktype in ("checkerboard", "channel"):
        a = build_flow(O, "NonUSFlow", [4, 6, 6], 2, ("conv", [8]), affine_conjugation=True, masktype=masktype)
        b = build_flow(P, "NonUSFlow", [4, 6, 6], 2, ("conv", [8]), affine_conjugation=True, masktype=masktype)
        assert list(a.state_dict().keys()) == list(b.state_dict().keys())
        b.load_state_dict(a.state_dict())
        assert [type(l).__name__ for l in a.layers] == [type(l).__name__ for l in b.layers]
        assert b.event_shape == (4, 6, 6) and b.event_dim == 144
        for la, lb in zip(a.layers, b.layers):
            if hasattr(la, "mask"):
                assert la.mask.shape == (1, 4, 6, 6) and torch.equal(la.mask, lb.mask)
    with pytest.raises(ValueError, match="Unknown mask type"):
        build_flow(P, "NonUSFlow", [4, 6, 6], 2, ("conv", [8]), masktype="stripes")
    with pytest.raises(ValueError, match="LU transforms must be non-negative"):
        build_flow(P, "NonUSFlow", 8, 2, ("mlp", [8]), lu_transform=-1)
    with pytest.raises(ValueError, match="Householder vectors transforms must be non-negative"):
        build_flow(P, "NonUSFlow", 8, 2, ("mlp", [8]), householder=-1)


def test_dropin_import_names_resolve_to_the_product():
    """The names nf4ad imports (`flows.py:3-17`, `transforms.py:5-6`, YAML `pyro.nn.DenseNN`, `src.usflows.sophia.SophiaG`,
    `src.usflows.networks.ConvNet`) resolve to this package once the drop-in is on the path (own interpreter: the oracle
    shim uses the same module names)."""
    code = (
        "import nf4ad_b200; nf4ad_b200.install_dropin(with_pyro=True)\n"
        "from src.usflows.flows import Flow, USFlow\n"
        "from src.usflows.transforms import (ScaleTransform, LUTransform, InverseTransform, BaseTransform,\n"
        "    BlockAffineTransform, HouseholderTransform, SequentialAffineTransform, MaskedCoupling)\n"
        "from src.usflows.distributions import Normal\n"
        "from src.usflows.networks import ConvNet\n"
        "from src.usflows.sophia import SophiaG\n"
        "from pyro import distributions as dist\n"
        "from pyro.nn import DenseNN, ConditionalDenseNN\n"
        "assert dist.constraints.real_vector is not None and dist.Normal and dist.Laplace and dist.TransformModule\n"
        "mods = {c.__module__.split('.')[0] for c in (Flow, USFlow, LUTransform, MaskedCoupling, Normal, ConvNet, SophiaG, DenseNN)}\n"
        "assert mods == {'nf4ad_b200'}, mods\n"
        "print('ok')\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=300,
                       env=dict(os.environ, PYTHONPATH=ROOT))
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_affine_run_plan_groups_the_layers_between_couplings():
    """`Flow._compose_affine_runs` (host logic, no CUDA): the layers of the data -> latent pass grouped into maximal runs
    of affine layers between couplings -- with affine conjugation K + 1 runs for K blocks, each run but the last the affine
    layer of one block followed by the inverse of the previous block's -- and on the CPU (or for a batch the tensor-core GEMMs do not take) nothing is
    composed.  `conditioner_weights` folds the coupling mask into the first layer only."""
    import nf4ad_b200
    from _cases import build_flow
    from nf4ad_b200 import stack
    from nf4ad_b200.transforms import InverseTransform, LUTransform, conditioner_weights
    ns = nf4ad_b200.namespace()
    K, D = 3, 16
    flow = build_flow(ns, "NonUSFlow", D, K, ("mlp", [32]), affine_conjugation=True, prior_scale=1.0)
    plan, composer = flow._compose_affine_runs(torch.zeros(8, D))
    assert composer is None                                           # CPU tensor: layer-wise
    runs = [item for item in plan if isinstance(item, list)]
    couplings = [item for item in plan if not isinstance(item, list)]
    assert len(couplings) == K and all(stack._is_coupling(c) for c in couplings)
    assert len(runs) == K + 1
    # reversed layer list: [scale, final affine, inverse of block K's], coupling K, [block K's affine, inverse of block
    # K-1's], ..., coupling 1, [block 1's affine]
    assert [len(r) for r in runs] == [3] + [2] * (K - 1) + [1]
    for r in runs[:-1]:                            # head of one block (its inverse direction) after the tail of the next
        assert isinstance(r[-1], InverseTransform) and not isinstance(r[-2], InverseTransform)
    assert all(any(isinstance(m, LUTransform) for layer in r for m in layer.modules()) for r in runs)
    flat = [layer for item in plan for layer in (item if isinstance(item, list) else [item])]
    assert flat == list(reversed(list(flow.layers)))                  # nothing lost, order kept
    # mask folding: (x * m) W^T == x (W * m)^T for the first layer, the others untouched
    cpl = couplings[0]
    ws = conditioner_weights(cpl.conditioner, cpl.mask)
    lin = [m for m in cpl.conditioner.modules() if isinstance(m, torch.nn.Linear)]
    assert len(ws) == len(lin) and ws[1][0] is lin[1].weight and ws[0][1] is lin[0].bias
    x = torch.randn(5, D)
    m = cpl.mask.reshape(-1)
    assert torch.allclose((x * m) @ lin[0].weight.t(), x @ ws[0][0].t(), atol=1e-6)
    assert conditioner_weights(torch.nn.Sequential(torch.nn.Tanh()), cpl.mask) is None      # opaque conditioner


def test_bench_dump_outputs_sample_past_the_limit(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: float32 files (float64 stays float64); past the byte limit every array keeps the same
    seeded sample of its rows, in order, so that two runs -- and the arrays of one run -- stay aligned entry for entry."""
    import numpy as np
    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4000)
    a = torch.arange(1000, dtype=torch.float64)
    b = torch.arange(2000, dtype=torch.float32).reshape(1000, 2)
    for run in ("r0", "r1"):
        bench.dump_outputs(str(tmp_path / run), {"a": a, "b": b})
    ra, rb = np.load(tmp_path / "r0" / "a.npy"), np.load(tmp_path / "r0" / "b.npy")
    assert ra.dtype == np.float64 and rb.dtype == np.float32 and 0 < ra.nbytes + rb.nbytes <= 4000
    assert np.all(np.diff(ra) > 0) and np.array_equal(rb[:, 0], 2 * ra)
    assert np.array_equal(ra, np.load(tmp_path / "r1" / "a.npy")) and np.array_equal(rb, np.load(tmp_path / "r1" / "b.npy"))
    bench.dump_outputs(str(tmp_path / "small"), {"c": torch.arange(10, dtype=torch.bfloat16)})
    c = np.load(tmp_path / "small" / "c.npy")
    assert c.dtype == np.float32 and np.array_equal(c, np.arange(10))


def test_bench_reference_arm_contract(tmp_path):
    """`bench.py --impl reference` (the CPU reference arm): rank 0 prints ONE JSON line with the contract's keys --
    `impl`, BASELINE.json's metric / unit, a `cpu_baseline` describing this very run (`kind` "reference" when the
    `oracle/_ref` snapshot exists, else "port"), an `e2e` that moves no bytes, and with `--dump-outputs` the log_prob of
    its last timed step on the seeded rows -- and every other rank exits 0 silently."""
    import json
    import numpy as np
    import bench
    import oracle
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "3",
           "--rows", "1024", "--config", "C4-adbench-D64", "--dump-outputs", str(tmp_path)]
    env = dict(os.environ, RANK="0", WORLD_SIZE="2", LOCAL_RANK="0", OMP_NUM_THREADS="4")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "log_prob samples/sec" and j["unit"] == "samples/s"
    assert j["higher_is_better"] is True and j["n_gpus"] == 2 and j["steps"] == 2 and j["warmup"] == 3
    assert j["value"] > 0 and abs(j["value"] - 1024 / (j["ms_per_step"] * 1e-3)) < 1e-6 * j["value"]
    cb = j["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == j["value"] and "1024 rows" in cb["sample"]
    assert j["e2e"] == {"value": j["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "C4-adbench-D64" in j["config"]["workload"] and "model" not in j["config"]
    lp = np.load(tmp_path / "log_prob.npy")
    assert lp.dtype == np.float32 and lp.shape == (1024,)
    ns = oracle.load_ref() if cb["kind"] == "reference" else oracle.load()
    with torch.no_grad():
        want = bench.build_config_flow(ns, "C4-adbench-D64", "cpu").log_prob(
            torch.randn(1024, 64, generator=torch.Generator().manual_seed(42)))
    np.testing.assert_allclose(lp, want.numpy(), rtol=1e-5, atol=1e-5)
    # the other ranks of a torchrun launch: no work, no output, exit 0
    r1 = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(env, RANK="1", LOCAL_RANK="1"), cwd=ROOT)
    assert r1.returncode == 0 and r1.stdout.strip() == ""
