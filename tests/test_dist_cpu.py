"""N > 1 host logic on the CPU: two gloo ranks exercise the rank helpers bench.py uses (barrier, max / sum
over ranks, per-rank workloads, tile and sample sharding)."""
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_gloo_ranks(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(textwrap.dedent('''
        import sys
        sys.path.insert(0, %r)
        import numpy as np
        from spliser_b200 import synth
        from spliser_b200.dist import Ranks, samples_of, tile_of
        import bench
        r = Ranks("gloo")
        assert r.world == 2
        cfg, _ = bench.workload_config("small", 4000, r.rank)
        w = synth.generate(cfg)
        r.barrier()
        total = r.sum(len(w.records))
        slow = r.max(10.0 + r.rank)
        chk = r.sum(float(w.records.pos[:100].sum()))
        mine = float(w.records.pos[:100].sum())
        assert total == 8000 and slow == 11.0
        assert chk != 2 * mine            # the two ranks count different samples (per-rank seed)
        lo, hi = tile_of(r.rank, r.world, 101)
        assert r.sum(hi - lo) == 101
        assert samples_of(r.rank, r.world, 5) == ([0, 2, 4] if r.rank == 0 else [1, 3])
        r.close()
        print("rank", r.rank, "ok")
    ''' % ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29517", str(script)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert res.stdout.count("ok") == 2


def test_one_sample_tiled_over_two_gloo_ranks(tmp_path):
    """The N > 1 path of bench.py on the CPU: ONE sample sharded over two ranks by genomic tile -- read-balanced cuts, the tile's
    records, the tile's own junction rows (every rank builds its own site table), counting by the oracle standing in for the
    device, owned rows written out, rank 0 concatenates: the table equals the unsharded one in every column.  No data-path
    collective: the ranks only meet at barriers."""
    script = tmp_path / "t.py"
    script.write_text(textwrap.dedent('''
        import os, sys
        sys.path.insert(0, %r)
        import numpy as np
        from oracle import c_oracle
        from spliser_b200 import api, dist, synth
        from spliser_b200.dist import Ranks
        r = Ranks("gloo")
        out = %r
        w = synth.generate(synth.config_small(40000, seed=7, stranded=True, paired=True))     # the same sample on every rank
        nc = len(w.chroms)
        table = api.build_site_table(nc, w.junctions, w.flags)
        cuts = dist.balanced_tiles(w.records, table, nc, r.world)
        lo, hi = cuts[r.rank], cuts[r.rank + 1]
        rec_t = dist.tile_records(w.records, table, nc, r.rank, r.world, site_range=(lo, hi), seg_spans=dist.segment_max_spans(w.records))
        rows, junc_t, local = dist.tile_junctions(w.junctions, table, nc, (lo, hi), w.flags)
        assert len(rec_t) < len(w.records) and len(junc_t) <= len(w.junctions)
        part = c_oracle.process(rec_t, nc, junc_t, w.flags | 4, threads=2)
        class T: pass
        t = T()
        for k, v in part.items(): setattr(t, k, v)
        np.savez(os.path.join(out, "part_%%d.npz" %% r.rank), **dist.owned_part(t, local, rows))
        sent = r.sum(len(rec_t))
        r.barrier()
        if r.rank == 0:
            full = c_oracle.process(w.records, nc, w.junctions, w.flags | 4, threads=2)
            parts = [dict(np.load(os.path.join(out, "part_%%d.npz" %% q))) for q in range(r.world)]
            d = c_oracle.diff_tables(dist.concat_parts(parts, full), full)
            assert d is None, d
            assert 0.9 * len(w.records) <= sent < 1.2 * len(w.records)     # edge reads go to both tiles; reads that can touch no site go to none
        r.barrier()
        r.close()
        print("rank", r.rank, "ok")
    ''' % (ROOT, str(tmp_path))))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29521", str(script)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert res.stdout.count("ok") == 2


def test_bench_reference_arm_prints_the_contract_line(tmp_path):
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) on a small workload: ONE JSON line with the
    keys of the bench contract; under torchrun (N > 1) rank 0 alone prints it and the other rank exits 0 without work."""
    import json
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", SPLISER_BENCH_CACHE=str(tmp_path))
    tail = ["bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1", "--reads", "120000"]
    one = subprocess.run([sys.executable] + tail, capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert one.returncode == 0, one.stderr[-2000:]
    lines = [ln for ln in one.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "reads/s" and d["value"] > 0 and d["warmup"] >= 3
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    two = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", "29519"] + tail[:1] + ["--gpus", "2"] + tail[1:], capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert two.returncode == 0, two.stderr[-2000:]
    lines = [ln for ln in two.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["n_gpus"] == 2


def _bench_dump(tmp_path, tag, *args):
    """Runs bench.py with --dump-outputs (workload cache of its own) -> {column: array}."""
    import numpy as np
    out = tmp_path / ("dump_" + tag)
    env = dict(os.environ, SPLISER_BENCH_CACHE=str(tmp_path / ("cache_" + tag)))
    res = subprocess.run([sys.executable, "bench.py", "--workload", "small", "--reads", "60000", "--steps", "2", "--warmup", "1",
                          "--dump-outputs", str(out)] + list(args), capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    return {p.name[:-4]: np.load(str(p)) for p in out.iterdir()}


def test_bench_dump_outputs_of_the_reference_arm(tmp_path):
    """`bench.py --dump-outputs DIR`: every column of the last step's table as float64 .npy, the same in two runs that each
    generate the workload afresh, and equal to the oracle's table of that seeded workload."""
    import numpy as np
    import bench
    from oracle import c_oracle
    from spliser_b200 import synth
    a = _bench_dump(tmp_path, "a", "--impl", "reference")
    b = _bench_dump(tmp_path, "b", "--impl", "reference")
    assert sorted(a) == sorted(c_oracle.TABLE_FIELDS) and sorted(b) == sorted(a)
    w = synth.generate(bench.workload_config("small", 60000)[0])
    want = c_oracle.process(w.records, len(w.chroms), w.junctions, w.flags)
    assert len(want["pos"]) > 500 and want["sse"].any()
    for k in c_oracle.TABLE_FIELDS:
        assert a[k].dtype == np.float64 and np.array_equal(a[k], b[k], equal_nan=True), k
        assert np.array_equal(a[k], want[k].astype(np.float64), equal_nan=True), k


def test_bench_dump_outputs_sample_above_the_limit(tmp_path):
    """A table larger than the limit keeps a seeded sample: under the limit on disk, the same rows in every column of one
    length, the same entries from call to call."""
    import numpy as np
    import bench
    from oracle import c_oracle
    n, e = 20000, 30000
    lens = {"partner_off": n + 1, "comp_off": n + 1, "partner_pos": e, "partner_cnt": e, "comp_pos": e // 2}
    t = {k: np.arange(lens.get(k, n), dtype=np.int64) * (i + 1) for i, k in enumerate(c_oracle.TABLE_FIELDS)}
    limit = 400_000
    for tag in ("a", "b"):
        bench.dump_outputs(str(tmp_path / tag), t, limit=limit)
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= limit
    got = {k: np.load(str(tmp_path / "a" / (k + ".npy"))) for k in c_oracle.TABLE_FIELDS}
    for i, k in enumerate(c_oracle.TABLE_FIELDS):
        assert 0 < len(got[k]) < lens.get(k, n) and np.array_equal(got[k], np.load(str(tmp_path / "b" / (k + ".npy")))), k
        rows = got[k] / (i + 1)                                      # the sampled row indices
        ref = {"partner_off": "comp_off", "partner_pos": "partner_cnt"}.get(k, "chrom" if lens.get(k, n) == n else k)
        assert np.array_equal(rows, got[ref] / (c_oracle.TABLE_FIELDS.index(ref) + 1)), k


def test_host_topology_against_a_fake_sysfs(tmp_path):
    """The NUMA report bench.py attaches to every line (and the opt-in binding) reads sysfs only: a fake tree with two
    nodes, the GPU on node 1."""
    from spliser_b200.dist import bind_to_device_node, host_topology, parse_cpulist
    assert parse_cpulist("0-3,8,10-11") == [0, 1, 2, 3, 8, 10, 11] and parse_cpulist("") == [] and parse_cpulist("a,2") == [2]
    allowed = sorted(os.sched_getaffinity(0))
    half = allowed[len(allowed) // 2:] or allowed
    for n, cl in ((0, "900-903"), (1, ",".join(map(str, half)))):
        d = tmp_path / "devices/system/node" / ("node%d" % n)
        d.mkdir(parents=True)
        (d / "cpulist").write_text(cl + "\n")
    dev = tmp_path / "bus/pci/devices/0000:1b:00.0"
    dev.mkdir(parents=True)
    (dev / "numa_node").write_text("1\n")
    t = host_topology(0, sysfs=str(tmp_path), bus_id="00000000:1B:00.0")
    assert t["gpu_numa_node"] == 1 and t["numa_nodes"] == 2 and t["node_cpus"] == len(half)
    assert t["cpus_allowed"] == len(allowed) and t["cpus_allowed_on_gpu_node"] == len(half)
    if len(half) < len(allowed):
        try:
            assert bind_to_device_node(t) and sorted(os.sched_getaffinity(0)) == half
        finally:
            os.sched_setaffinity(0, allowed)
    # unknown GPU / single node / virtualised numa_node = -1: report only, never bind
    (dev / "numa_node").write_text("-1\n")
    t = host_topology(0, sysfs=str(tmp_path), bus_id="00000000:1B:00.0")
    assert t["gpu_numa_node"] == -1 and not bind_to_device_node(t)
    t = host_topology(0, sysfs=str(tmp_path / "absent"), bus_id="00000000:1B:00.0")
    assert t["gpu_numa_node"] is None and not bind_to_device_node(t)
