"""CPU tests of the N>1 path: scenario sharding + the single all-gather of result records,
world_size 2 over gloo (the GPU runs use the same code over NCCL)."""
import os

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import landing_controller_b200 as lc


def test_shard_bounds_cover_everything():
    for n in (1, 7, 1024, 16384, 1000):
        for w in (1, 2, 4, 8):
            b = [lc.shard_bounds(n, w, r) for r in range(w)]
            assert b[0][0] == 0 and b[-1][1] == n
            assert all(b[i][1] == b[i + 1][0] for i in range(w - 1))
            assert max(h - l for l, h in b) - min(h - l for l, h in b) <= 1


def test_grid_sweep_shapes():
    for B in (1024, 2048, 16384):
        d = lc.grid_sweep(B)
        assert d.shape == (B, 12) and len(np.unique(d, axis=0)) == B
    d = lc.grid_sweep(1024)
    assert set(np.round(np.unique(d[:, 2]), 3)) == {0.4, 0.5, 0.6, 0.7}
    assert np.isclose(d[:, 4].min(), -np.pi / 3) and np.isclose(d[:, 9].max(), 1.75)
    r = lc.random_sweep(100, seed=0)
    assert np.array_equal(r, lc.random_sweep(100, seed=0)) and r[:, 2].min() > 0.35


def test_interleaved_shards_partition_the_sweep():
    for n in (1, 7, 1024, 1000):
        for w in (1, 2, 4, 8):
            ids = [lc.shard_indices(n, w, r) for r in range(w)]
            assert np.array_equal(np.sort(np.concatenate(ids)), np.arange(n))
            assert max(map(len, ids)) - min(map(len, ids)) <= 1
            assert np.array_equal(lc.shard_indices(n, w, 0, "block"), np.arange(*lc.shard_bounds(n, w, 0)))
            order = lc.unshard_order(n, w)
            full = np.empty(n)
            full[order] = np.concatenate([i.astype(float) for i in ids])
            assert np.array_equal(full, np.arange(n))


def _worker(rank, world, port, n, nx, q, mode="block"):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    drops = lc.grid_sweep(1024)[:n]
    ids = lc.shard_indices(n, world, rank, mode)
    mine = drops[ids]
    # stand-in for the GPU solve: a deterministic function of the drop condition
    x = np.repeat(mine[:, :1] + mine[:, 2:3] * 10 + mine[:, 4:5] * 100 + mine[:, 9:10] * 1000, nx, axis=1)
    rec = lc.pack_records(x, mine[:, 2], ids % 3, ids)
    full = lc.gather_records(rec, n, world, rank, mode).numpy()
    if rank == 0:
        q.put(full)
    dist.barrier()
    dist.destroy_process_group()


import pytest


@pytest.mark.parametrize("mode", ["block", "interleaved"])
def test_all_gather_of_records_world2_gloo(mode):
    n, nx, world = 37, 5, 2  # ragged on purpose
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000) + (7 if mode == "block" else 0)
    procs = [ctx.Process(target=_worker, args=(r, world, port, n, nx, q, mode)) for r in range(world)]
    for p in procs:
        p.start()
    full = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    out = lc.unpack_records(full)
    drops = lc.grid_sweep(1024)[:n]
    assert out["x"].shape == (n, nx)
    assert np.array_equal(out["iters"], np.arange(n)) and np.array_equal(out["status"], np.arange(n) % 3)
    assert np.allclose(out["f"], drops[:, 2])
    assert np.allclose(out["x"][:, 0], drops[:, 0] + drops[:, 2] * 10 + drops[:, 4] * 100 + drops[:, 9] * 1000)


def test_reference_arm_line_schema():
    """bench.py --impl reference prints one JSON line with the contract's keys (CPU oracle, tiny sample)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--batch", "8",
                          "--steps", "1", "--warmup", "0", "--knots", "21"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "NLP/s" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"] > 0
    for k in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config"):
        assert k in line


def test_bench_dump_outputs_whole_and_sampled(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float64 .npy files, the whole sweep when it fits the size limit, otherwise the same
    seeded sample of scenarios on every call."""
    import sys
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)  # (bench sets it on import)
    import bench
    B, nx = 50, 10
    x = np.arange(B * nx, dtype=np.float64).reshape(B, nx)
    f, st, it = np.arange(B) * 0.5, np.arange(B, dtype=np.int32) % 5, np.arange(B, dtype=np.int32)
    load = lambda d: {n: np.load(os.path.join(d, n + ".npy")) for n in ("x", "f", "status", "iters", "scenario")}
    bench.dump_outputs(str(tmp_path / "all"), x, f, st, it)
    a = load(str(tmp_path / "all"))
    assert all(v.dtype == np.float64 for v in a.values())
    assert np.array_equal(a["x"], x) and np.array_equal(a["status"], st) and np.array_equal(a["scenario"], np.arange(B))
    monkeypatch.setattr(bench, "DUMP_LIMIT", 8 * (nx + 4) * 12)  # room for 12 scenarios
    bench.dump_outputs(str(tmp_path / "s1"), x, f, st, it)
    bench.dump_outputs(str(tmp_path / "s2"), x, f, st, it)
    s1, s2 = load(str(tmp_path / "s1")), load(str(tmp_path / "s2"))
    ids = s1["scenario"].astype(int)
    assert len(ids) == 12 and len(np.unique(ids)) == 12 and all(np.array_equal(s1[n], s2[n]) for n in s1)
    assert sum(v.nbytes for v in s1.values()) <= bench.DUMP_LIMIT
    assert np.array_equal(s1["x"], x[ids]) and np.array_equal(s1["f"], f[ids]) and np.array_equal(s1["iters"], it[ids])


def test_bench_sweep_records_undo_the_interleaved_all_gather(monkeypatch):
    """bench.py --dump-outputs under torchrun: the padded, rank-major all-gathered records back in sweep order."""
    import sys
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)
    import bench
    n, nx = 37, 4
    for world in (1, 2, 3, 8):
        x = np.arange(n * nx, dtype=np.float64).reshape(n, nx) + 0.25
        rec = lc.pack_records(x, np.arange(n) * 1.5, np.arange(n) % 5, np.arange(n) + 7)
        bmax = -(-n // world)
        gathered = np.full((world, bmax, nx + 3), np.nan)  # padding rows must never be read
        for r in range(world):
            ids = lc.shard_indices(n, world, r)
            gathered[r, :len(ids)] = rec[ids]
        out = bench.sweep_records(gathered, n, world)
        ref = lc.unpack_records(rec)
        assert all(np.array_equal(out[k], ref[k]) for k in ("x", "f", "status", "iters"))


def test_fast_oracle_fallback_names_the_failure(monkeypatch):
    """The timed CPU arm's -O3 build falls back to the -O2 library only with the reason in its label."""
    import tempfile
    import oracle_lib

    def no_tmp(**kw):
        raise PermissionError("temporary directory not writable")
    monkeypatch.setattr(tempfile, "mkdtemp", no_tmp)
    path, how = oracle_lib.build_oracle_fast()
    assert path == oracle_lib.ORACLE_SO and "-O2" in how and "temporary directory not writable" in how
