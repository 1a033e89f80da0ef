"""BASELINE.json's full-size configurations on the GPU, checked through size-independent properties (the oracle
would take too long at these sizes): the 200 x 200 m map at 0.25 m cells, thousands of 1080-beam scans, 1M-scale
hypothesis sweeps. Properties: batch == single, permutation invariance, host API == device API, LaserScan input ==
point input, sweep score == evaluate score, incremental map == one-shot map, and recovery of the true poses."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def world():
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    B = 4096
    sc = synth.SCAN_1080
    ranges, poses = synth.scans(B, traj_len=B, **sc)
    init = poses + synth.uniform3(B) * np.array([0.03, 0.03, math.radians(0.3)])
    map_xy = synth.make_map(1024, traj_len=1024, **sc)
    cb, sb = synth.beam_table(sc["nbeams"], sc["angle_min"], sc["angle_inc"])
    xy = np.stack([ranges * cb, ranges * sb], -1).astype(np.float32).reshape(-1, 2)
    off = np.arange(B + 1, dtype=np.int64) * sc["nbeams"]
    m = g.NdtMatcher2D([0.25])
    m.set_grid(-100.0, -100.0, 200.0, 200.0)
    m.set_target(map_xy)
    return dict(g=g, synth=synth, m=m, B=B, ranges=ranges, poses=poses, init=init, map_xy=map_xy, xy=xy, off=off, sc=sc)


def test_config2_batch_recovers_truth_and_is_order_independent(world):
    m, B = world["m"], world["B"]
    assert m.geometry() == dict(res=np.float32(0.25), st=np.float32(0.25), inv_st=np.float32(4.0), ox=np.float32(-100.0),
                                oy=np.float32(-100.0), nhx=800, nhy=800, njx=800, njy=800)
    r = m.align_batch(world["xy"], world["off"], world["init"])
    assert (r["status"] == 0).mean() > 0.99 and r["iterations"].mean() < 16
    err = r["pose"] - world["poses"]
    err[:, 2] = (err[:, 2] + np.pi) % (2 * np.pi) - np.pi
    ok = r["status"] == 0
    e = np.hypot(err[ok, 0], err[ok, 1])   # single-level 0.25 m NDT: a few percent settle in a neighbouring optimum
    assert np.median(e) < 2e-3 and np.percentile(e, 95) < 0.02 and (e < 0.05).mean() > 0.97, (np.percentile(e, [50, 95, 99]), (e < 0.05).mean())
    pd = (np.linalg.eigvalsh(r["hessian"][ok]).min(1) > 0).mean()   # a usable information matrix at (nearly) every optimum
    assert pd > 0.99, pd
    # permutation of the batch permutes the results bit for bit
    perm = np.random.default_rng(1).permutation(B)
    xy3 = world["xy"].reshape(B, 1080, 2)[perm].reshape(-1, 2)
    r2 = m.align_batch(xy3, world["off"], world["init"][perm])
    assert r2.tobytes() == r[perm].tobytes()
    # single calls equal the batch
    for i in (0, 777, B - 1):
        assert m.align(world["xy"][i * 1080:(i + 1) * 1080], world["init"][i]).tobytes() == r[i].tobytes()
    world["res"] = r


def test_config2_laserscan_input_equals_point_input(world):
    m, sc = world["m"], world["sc"]
    r = world.get("res")
    if r is None:
        r = m.align_batch(world["xy"], world["off"], world["init"])
    rr = m.align_batch_ranges(world["ranges"], sc["angle_min"], sc["angle_inc"], world["init"], range_scale=1.0)
    assert rr.tobytes() == r.tobytes()


def test_config2_laserscan_pipeline_over_several_chunks(world):
    """The batch tiled four times (16 384 scans) crosses the host-buffer pipeline's ~18 MB chunk size: four chunks of f32
    ranges, two of u16. A result does not depend on its place in the batch, so the results tile too."""
    m, sc, init = world["m"], world["sc"], world["init"]
    r = world.get("res")
    if r is None:
        r = m.align_batch(world["xy"], world["off"], init)
    init4 = np.tile(init, (4, 1))
    rr = m.align_batch_ranges(np.tile(world["ranges"], (4, 1)), sc["angle_min"], sc["angle_inc"], init4, range_scale=1.0)
    assert rr.tobytes() == np.tile(r, 4).tobytes()
    u16 = np.round(world["ranges"] / 0.004).clip(0, 65535).astype(np.uint16)
    one = m.align_batch_ranges(u16, sc["angle_min"], sc["angle_inc"], init, range_scale=0.004)      # a single chunk
    r4 = m.align_batch_ranges(np.tile(u16, (4, 1)), sc["angle_min"], sc["angle_inc"], init4, range_scale=0.004)
    assert r4.tobytes() == np.tile(one, 4).tobytes()


def test_config2_device_api_equals_host_api(world):
    import torch
    m, B, g = world["m"], world["B"], world["g"]
    r = world.get("res")
    if r is None:
        r = m.align_batch(world["xy"], world["off"], world["init"])
    dev = torch.device("cuda", 0)
    d_xy = torch.from_numpy(world["xy"]).to(dev)
    d_off = torch.from_numpy(world["off"]).to(dev)
    d_init = torch.from_numpy(np.ascontiguousarray(world["init"])).to(dev)
    d_res = torch.zeros(B * 144, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    m.align_batch_device(d_xy, d_off, B, 1080, d_init, d_res)
    m.synchronize()
    got = np.frombuffer(d_res.cpu().numpy().tobytes(), dtype=g.RESULT_DTYPE)
    assert got.tobytes() == r.tobytes()


def test_config3_pyramid_batch(world):
    g, B = world["g"], 2048
    m = g.NdtMatcher2D([2.0, 1.0, 0.5])
    m.set_grid(-100.0, -100.0, 200.0, 200.0)
    m.set_target(world["map_xy"])
    init = world["poses"][:B] + world["synth"].uniform3(B, first=10 ** 6) * np.array([0.2, 0.2, math.radians(3.0)])
    r = m.align_batch(world["xy"][: B * 1080], world["off"][: B + 1], init)
    err = r["pose"] - world["poses"][:B]
    assert (r["status"] == 0).mean() > 0.98
    assert np.percentile(np.hypot(err[:, 0], err[:, 1]), 98) < 0.03


def test_config4_sweep_scores_are_evaluations_and_best_is_truth(world):
    m, synth = world["m"], world["synth"]
    scan = world["xy"][5 * 1080: 6 * 1080]
    truth = world["poses"][5]
    side, nth = 46, 120                                       # 46 * 46 * 120 = 253 920 hypotheses
    gx = (np.arange(side) - side // 2) * 0.2
    lat = np.stack(np.meshgrid(gx, gx, np.radians(np.arange(nth) * 3.0 - 180.0), indexing="ij"), -1).reshape(-1, 3)
    hyp = (truth + lat).astype(np.float32)
    s, bi, bs = m.sweep(scan, hyp, k=16)
    order = np.lexsort((np.arange(len(s)), -s))[:16]
    assert np.array_equal(bi, order) and np.array_equal(bs, s[order])
    assert np.abs(hyp[bi[0]].astype(np.float64) - truth).max() < 1e-3
    pick = np.random.default_rng(2).integers(0, len(hyp), 200)
    ev, _ = m.evaluate(scan, hyp[pick].astype(np.float64))
    assert np.array_equal(ev[:, 0], s[pick])                  # the sweep is the evaluation's score, bit for bit
    # sharding the hypotheses (as the multi-GPU path does) gives the same winner
    from gtsam_ndt_b200.distributed import shard_range
    best = []
    for rk in range(8):
        lo, hi = shard_range(len(hyp), rk, 8)
        _, i, v = m.sweep(scan, hyp[lo:hi], k=1, want_scores=False)
        best.append((-v[0], i[0] + lo))
    assert min(best)[1] == bi[0]


def test_incremental_map_equals_one_shot_at_full_size(world):
    g = world["g"]
    a = g.NdtMatcher2D([0.25]); a.set_grid(-100.0, -100.0, 200.0, 200.0)
    n = len(world["map_xy"])
    a.set_target(world["map_xy"][: n // 3])
    a.add_target(world["map_xy"][n // 3: n // 2])
    a.add_target(world["map_xy"][n // 2:])
    assert a.cells().tobytes() == world["m"].cells().tobytes()
