"""Multi-rank (SURVEY.md §8e): block-sharded scan points / patches + all-reduce of the packed normal
equations.  CPU tier: world_size-2 gloo, sharding + reduction logic against the unsharded oracle.
GPU tier (needs >= 2 GPUs): the NCCL path of libfastlivo_b200 against the unsharded oracle."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def shard(n, rank, world):
    per = (n + world - 1) // world
    lo = min(rank * per, n)
    return lo, min(lo + per, n)


def _cpu_worker(rank, world, port, out):
    import torch
    import torch.distributed as dist
    import fastlivo_loader
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    flb = fastlivo_loader.load()
    po = fastlivo_loader.oracle()
    f = flb.synth.make_frame("T1")
    s0, s1 = shard(len(f["scan_body"]), rank, world)
    lio = po.Lio(f["map_xyz"], f["scan_body"][s0:s1])
    o = lio.run_pass(po.lio_params(f, 3, nthreads=1), f["R_prop"], f["p_prop"], True)
    packed = np.concatenate([o["HTH6"].ravel(), o["HTz6"], [o["n"], o["total_residual"]]])
    p0, p1 = shard(len(f["patch_pos"]), rank, world)
    vio = po.Vio(f["image"], f["patch_pos"][p0:p1], f["patch_ref"][p0:p1], f["patch_level"][p0:p1], f["cam"])
    v = vio.run_pass(po.vio_params(f, 3), f["R_prop"], f["p_prop"], 1, rows=False)
    vpacked = np.concatenate([v["HTH6"].ravel(), v["HTz6"], [v["n_meas"], v["skipped"]]])
    t = torch.from_numpy(np.concatenate([packed, vpacked]))
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    # equal-size padded shards for the all-gather of the per-patch errors (padding = 0.0f)
    per = (len(f["patch_pos"]) + world - 1) // world
    e = np.zeros(per, np.float32)
    e[:p1 - p0] = v["errors"]
    parts = [torch.zeros(per) for _ in range(world)]
    dist.all_gather(parts, torch.from_numpy(e))
    if rank == 0:
        np.savez(out, reduced=t.numpy(), errors=torch.cat(parts).numpy())
    dist.destroy_process_group()


def test_sharded_normal_equations_gloo(flb, po, frames, tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "red.npz")
    world = 2
    mp.spawn(_cpu_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    r = np.load(out)
    f = frames("T1")
    lio = po.Lio(f["map_xyz"], f["scan_body"])
    o = lio.run_pass(po.lio_params(f, 3), f["R_prop"], f["p_prop"], True)
    full = np.concatenate([o["HTH6"].ravel(), o["HTz6"], [o["n"], o["total_residual"]]])
    np.testing.assert_allclose(r["reduced"][:44], full, rtol=1e-11, atol=1e-12)
    vio = po.Vio(f["image"], f["patch_pos"], f["patch_ref"], f["patch_level"], f["cam"])
    v = vio.run_pass(po.vio_params(f, 3), f["R_prop"], f["p_prop"], 1, rows=False)
    vfull = np.concatenate([v["HTH6"].ravel(), v["HTz6"], [v["n_meas"], v["skipped"]]])
    np.testing.assert_allclose(r["reduced"][44:], vfull, rtol=1e-11, atol=1e-9)
    # gathered errors, in patch order, reproduce the exact sequential float sum (zeros are exact no-ops)
    e_seq = np.float32(0)
    for x in r["errors"]:
        e_seq = np.float32(e_seq + np.float32(x))
    assert np.float32(e_seq / np.float32(v["n_meas"])) == v["error"]


def test_shard_partition_properties():
    for n in (0, 1, 7, 2000, 24000):
        for w in (1, 2, 3, 4, 8):
            cuts = [shard(n, r, w) for r in range(w)]
            assert cuts[0][0] == 0 and cuts[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(cuts, cuts[1:]))
            assert max(b - a for a, b in cuts) <= (n + w - 1) // w


def _trim(f, mode):
    """'p2p-ragged': a frame so small that rank 1's shards are EMPTY (1 scan point, 1 patch over 2 ranks)."""
    if mode != "p2p-ragged":
        return f
    g = dict(f)
    g["scan_body"] = f["scan_body"][:1]
    for k in ("patch_pos", "patch_ref", "patch_level"):
        g[k] = f[k][:1]
    return g


def _gpu_worker(rank, world, port, out, mode="nccl"):
    import torch
    import torch.distributed as dist
    import fastlivo_loader
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)      # only to hand the NCCL id around
    flb = fastlivo_loader.load()
    f = _trim(flb.synth.make_frame("T1"), mode)
    h = flb.Handle(device=rank)
    if mode == "nccl":
        uid = [flb.Handle.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        h.comm_init(uid[0], rank, world)
    else:   # fused NVLink exchange inside the persistent kernels
        handles = [None] * world
        dist.all_gather_object(handles, h.p2p_export())
        h.p2p_attach(rank, world, handles)
    s0, s1 = shard(len(f["scan_body"]), rank, world)
    p0, p1 = shard(len(f["patch_pos"]), rank, world)
    h.map_upload(f["map_xyz"])
    h.scan_upload(f["scan_body"][s0:s1])
    h.camera_set(f["cam"])
    h.image_upload(f["image"])
    h.patches_upload(f["patch_pos"][p0:p1], f["patch_ref"][p0:p1], f["patch_level"][p0:p1])
    x = flb.capi.State18.from_frame(f)
    lrep = h.lio_update(flb.capi.lio_params(f, 4), x, x.copy())
    vrep = h.vio_update(flb.capi.vio_params(f, 4), x, x.copy())
    states = [None] * world
    dist.all_gather_object(states, x.vector().tolist())
    if rank == 0:
        np.savez(out, states=np.array(states), P=x.P, lio=[lrep.passes, lrep.knn_passes, lrep.n_eff_last, lrep.rows_total],
                 vio=[*vrep.passes, vrep.rows_total, vrep.cov_updated])
    h.close()
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["nccl", "p2p", "p2p-ragged"])
def test_sharded_update_matches_oracle(flb, po, frames, tmp_path, mode):
    """Both collectives: NCCL all-reduce between per-pass kernels, and the fused NVLink exchange inside
    the persistent kernels (T1 with early stop has a rejected VIO step: the speculated pass is discarded on
    every rank alike).  'p2p-ragged': rank 1 owns no scan point and no patch and still takes part in every
    exchange."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    out = str(tmp_path / "gpu.npz")
    # FLB_TEST_WORLD=4 / 8 on a machine with that many GPUs: the same test at that world size
    world = max(2, min(int(os.environ.get("FLB_TEST_WORLD", "2")), torch.cuda.device_count(), 8))
    mp.spawn(_gpu_worker, args=(world, _free_port(), out, mode), nprocs=world, join=True)
    r = np.load(out)
    f = _trim(frames("T1"), mode)
    lio = po.Lio(f["map_xyz"], f["scan_body"])
    vio = po.Vio(f["image"], f["patch_pos"], f["patch_ref"], f["patch_level"], f["cam"])
    x = po.state_from_frame(f)
    lrep = lio.update(po.lio_params(f, 4), x, x.copy())
    vrep = vio.update(po.vio_params(f, 4), x, x.copy())
    assert list(r["lio"]) == [lrep.passes, lrep.knn_passes, lrep.n_eff_last, lrep.rows_total]
    assert list(r["vio"]) == [*vrep.passes, vrep.rows_total, vrep.cov_updated]
    ref = x.vector()
    # every rank ends in the bit-identical state (same reduced inputs -> same solve) ...
    assert all((r["states"][0] == r["states"][k]).all() for k in range(1, len(r["states"])))
    # ... which matches the unsharded CPU path
    assert np.abs(r["states"][0] - ref).max() / np.abs(ref).max() < 1e-9
    np.testing.assert_allclose(r["P"], x.P, rtol=1e-6, atol=1e-14)
