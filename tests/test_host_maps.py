"""Host layer (prosstt_b200.tree / sim_utils / device.TreeTables) against the fixtures
produced by running the reference: integer maps are bit-exact.  CPU only."""
import re
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, golden_lineage, load_maps, load_npz, pairs_to_dict
from prosstt_b200 import _native as nat
from prosstt_b200 import sim_utils as sut, simulation as sim, tree as ptree, tree_utils as tu
from prosstt_b200.device import TreeTables, choice_cdf

MAPS = load_maps()


def _tree(rec, **kw):
    time = pairs_to_dict(rec["time"])
    return ptree.Tree(topology=rec["topology"], time=time, num_branches=len(time),
                      branch_points=rec["branch_points"], modules=3, G=7, **kw)


@pytest.mark.parametrize("rec", MAPS, ids=[r["name"] for r in MAPS])
def test_tree_maps_match_reference(rec):
    t = _tree(rec)
    assert t.branches == rec["branches"] and t.root == rec["root"]
    bt = t.branch_times()
    assert [[k, list(v)] for k, v in bt.items()] == rec["branch_times"]
    zones = t.populate_timezone()
    assert zones == rec["timezone"]
    live = sut.assign_branches(bt, zones)
    assert [[k, v] for k, v in live.items()] == rec["assignments"]
    pt, br = sim.cover_whole_tree(t)
    assert pt == rec["cover_pt"] and br == rec["cover_br"]
    assert t.get_max_time() == rec["max_time"]
    assert [str(b) for b in sut.breadth_first_branches(t)] == [str(b) for b in rec["bfs"]]
    assert t.paths(t.root) == rec["paths"]
    par = t.get_parallel_branches()
    assert [[k if not hasattr(k, "item") else k.item(), list(v.tolist())] for k, v in par.items()] == rec["parallel"]
    assert abs(sum(np.sum(v) for v in t.density.values()) - rec["density_sum"]) < 1e-15


@pytest.mark.parametrize("rec", MAPS, ids=[r["name"] for r in MAPS])
def test_device_tables_flatten_the_same_maps(rec):
    t = _tree(rec)
    tb = TreeTables(t, "cpu")
    bt = t.branch_times()
    assert tb.P == sum(t.time.values)
    for i, b in enumerate(tb.names):
        assert tb.branch_start[i] == bt[b][0] and tb.T[i] == t.time[b]
    # packed positions are sample_density's concatenation (simulation.py:454-461)
    want_pt = np.concatenate([np.arange(bt[b][0], bt[b][1] + 1) for b in t.branches])
    assert np.array_equal(tb.pos_pt, want_pt)
    assert [tb.names[c] for c in tb.pos_branch] == [b for b in t.branches for _ in range(t.time[b])]
    # cover tables == cover_whole_tree
    assert tb.cover_pt.tolist() == rec["cover_pt"]
    assert [tb.names[c] for c in tb.cover_branch] == rec["cover_br"]
    for e in range(len(tb.cover_pt)):
        b = tb.cover_branch[e]
        assert tb.cover_row[e] == tb.row_base[b] + tb.cover_pt[e] - tb.branch_start[b]
    # candidates per zone == assign_branches
    live = sut.assign_branches(bt, t.populate_timezone())
    for z in range(len(tb.zone_lo)):
        got = [tb.names[c] for c in tb.cand_branch[tb.cand_off[z]:tb.cand_off[z + 1]]]
        assert got == live[z]
    assert tb.max_time == rec["max_time"]


def test_random_topology_matches_reference_stream():
    # gen_random_topology consumes np.random.choice exactly like tree.py:82-113
    for rec in MAPS:
        m = re.match(r"random_s(\d+)_bp(\d+)", rec["name"])
        if not m:
            continue
        np.random.seed(int(m.group(1)))
        top = ptree.Tree.gen_random_topology(int(m.group(2)))
        assert [[int(a), int(b)] for a, b in top] == rec["topology"]


def test_tree_defaults_and_errors():
    np.random.seed(0)
    t = ptree.Tree()
    assert t.branches == ["A", "B", "C"] and t.G == 500 and 6 <= t.modules <= 24
    assert dict(t.branch_times()) == {"A": [0, 39], "B": [40, 79], "C": [40, 79]}
    with pytest.raises(ValueError):
        t.add_genes({"A": np.zeros((40, 500))})
    with pytest.raises(ValueError):
        t.add_genes({"A": np.zeros((40, 500)), "B": np.zeros((40, 500)), "C": np.zeros((39, 500))})
    with pytest.raises(ValueError):
        t.set_density({"A": np.ones(40)})
    with pytest.raises(ValueError):
        t.set_density({"A": np.ones(40), "B": np.ones(40), "C": np.ones(3)})
    with pytest.raises(ValueError):
        t.set_velocity({"A": np.ones(40)})
    bad = ptree.Tree(topology=[[1, 2], [0, 1]], time={0: 3, 1: 3, 2: 3}, modules=1, G=1)
    with pytest.raises(ValueError):
        bad.branch_times()
    t2 = ptree.Tree(modules=4)
    t2.num_branches = 5
    with pytest.raises(ValueError):          # simulation.py:254-256, raised before any GPU work
        sim.simulate_lineage(t2, a=0.05)


def test_newick():
    t = ptree.Tree.from_newick("(A:50,B:50)C:50;", genes=10, modules=2)
    assert t.branches == ["C", "A", "B"] and t.root == "C"
    assert t.topology == [["C", "A"], ["C", "B"]] and t.num_branches == 3 and t.branch_points == 1
    assert dict(t.time) == {"C": 50, "A": 50, "B": 50}
    t = ptree.Tree.from_newick("((D,E)B:7,C:3)A;", genes=10, modules=2)
    assert t.branches == ["A", "B", "D", "E", "C"]
    assert dict(t.time) == {"A": 40, "B": 7, "D": 40, "E": 40, "C": 3}
    assert t.topology == [["A", "B"], ["A", "C"], ["B", "D"], ["B", "E"]]
    with pytest.raises(ValueError):
        tu.newick_loads("((A,B)C;")


def test_velocity_to_density():
    t = ptree.Tree(modules=2)
    vel = {b: np.linspace(1.0, 2.0, 40) for b in t.branches}
    t.set_velocity(vel)
    assert abs(sum(np.sum(v) for v in t.density.values()) - 1) < 1e-12
    assert t.density["A"][0] > t.density["A"][-1]          # slow cells pile up


def test_choice_cdf_validation():
    cdf = choice_cdf(np.full(8, 0.125))
    assert cdf[-1] == 1.0
    with pytest.raises(ValueError):
        choice_cdf([0.5, 0.6])
    with pytest.raises(ValueError):
        choice_cdf([1.5, -0.5])


def test_timeseries_input_and_groups():
    pts, cells, std = sut.process_timeseries_input([0, 10, 20], 100, 6.0)
    assert cells.tolist() == [33, 33, 33] and std.tolist() == [2.0, 2.0, 2.0]
    np.random.seed(1)
    groups = sut.create_groups(4, 30)
    assert len(groups) == 4 and sorted(g for grp in groups for g in grp) == sorted(list(range(30)) * 2)
    assert sut.flat_order(4).tolist() == [[0, 0, 1], [1, 0, 2], [2, 0, 3], [3, 1, 2], [4, 1, 3], [5, 2, 3]]


def test_host_side_draws_follow_the_reference_stream():
    """generate_negbin_params / simulate_coefficients / simulate_base_gene_exp stay on the
    global legacy numpy stream: same seed -> the reference's values."""
    from prosstt_b200 import count_model as cm
    d = load_npz("nbparams.npz")
    np.random.seed(5)
    a, b = cm.generate_negbin_params(type("T", (), {"G": 64})(), mean_alpha=0.2, mean_beta=2)
    assert np.array_equal(a, d["gen_alpha"]) and np.array_equal(b, d["gen_beta"])
    branches, time, top, L = golden_lineage("abc")
    np.random.seed(int(L["seed"]))
    t = ptree.Tree(topology=top, time=time, num_branches=3, branch_points=1, modules=int(L["K"]), G=int(L["G"]))
    H = sim.simulate_coefficients(t, a=float(L["a"]))
    assert np.array_equal(H, L["H"])                         # first draws after the seed


def test_library_loads_and_exports_every_declared_symbol():
    lib = nat.load()
    header = open(os.path.join(ROOT, "include", "prosstt_b200.h")).read()
    declared = set(re.findall(r"\b(pst_[a-z0-9_]+)\s*\(", header))
    assert declared == set(nat.declared_symbols())
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.pst_abi_version() == 2
    # loading launches nothing; asked of a fresh process, since earlier tests in this one may have launched kernels
    code = "import sys; sys.path.insert(0, %r); from prosstt_b200 import _native as nat; " \
           "print(nat.load().pst_launch_count())" % ROOT
    fresh = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert fresh.returncode == 0, fresh.stderr
    assert fresh.stdout.strip() == "0"


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    t = ptree.Tree(modules=2, G=8)
    with pytest.raises(nat.NativeError):
        sim.simulate_lineage(t, a=0.05)
    with pytest.raises(nat.NativeError):
        sim.sample_density(t, 10)


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "prosstt_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("no oracle", ""), f


def test_text_writers_match_files_written_by_the_reference(tmp_path):
    """Byte-for-byte: tests/golden/written_files.json holds what the reference's own writers
    (tree_utils.py:59-173) produce for conftest.writer_inputs()."""
    import json
    from conftest import writer_inputs
    X, uMs, H, labs, brns, scal, gscale, alpha, beta = writer_inputs()
    t = ptree.Tree(topology=[["A", "B"]], time={"A": 3, "B": 2}, num_branches=2, branch_points=0, modules=2, G=5)
    tu.save_matrices("job", str(tmp_path), X, uMs, H)
    tu.save_cell_params("job", str(tmp_path), labs, brns, scal)
    tu.save_gene_params("job", str(tmp_path), gscale, alpha, beta)
    tu.save_params("job", str(tmp_path), t, 7)
    want = json.load(open(os.path.join(ROOT, "tests", "golden", "written_files.json")))
    assert sorted(os.listdir(tmp_path)) == sorted(want)
    for name, text in want.items():
        assert open(tmp_path / name).read() == text, name


def test_text_writers_round_trip(tmp_path):
    """tree_utils.save_* write the reference's file set (tree_utils.py:59-173)."""
    import pandas as pd
    X = np.arange(12).reshape(3, 4)
    uMs = {"A": np.ones((2, 4)) * 0.5, "B": np.zeros((1, 4))}
    H = np.arange(8.0).reshape(2, 4)
    tu.save_matrices("job", str(tmp_path), X, uMs, H)
    tu.save_cell_params("job", str(tmp_path), [0, 1, 2], ["A", "A", "B"], [1.0, 0.5, 2.0])
    tu.save_gene_params("job", str(tmp_path), [1.0, 2, 3, 4], [0.1, 0.2, 0.3, 0.4], [2.0, 2, 2, 2])
    t = ptree.Tree(modules=3, G=4)
    tu.save_params("job", str(tmp_path), t, 7)
    back = pd.read_csv(tmp_path / "job_simulation.txt", sep="\t", index_col=0)
    assert list(back.columns) == ["gene_%d" % i for i in range(4)] and list(back.index) == ["cell_0", "cell_1", "cell_2"]
    assert np.array_equal(back.values, X)
    assert np.array_equal(np.loadtxt(tmp_path / "job_h.txt"), H)
    assert np.array_equal(np.loadtxt(tmp_path / "job_umsA.txt"), uMs["A"])
    cells = pd.read_csv(tmp_path / "job_cellparams.txt", sep="\t", index_col=0)
    assert list(cells.columns) == ["pseudotime", "branches", "scalings"] and list(cells["branches"]) == ["A", "A", "B"]
    genes = pd.read_csv(tmp_path / "job_geneparams.txt", sep="\t", index_col=0)
    assert list(genes.columns) == ["alpha", "beta", "genescale"]
    text = (tmp_path / "job_params.txt").read_text()
    assert "Genes: 4" in text and "#modules: 3" in text and text.endswith("random seed: 7")


def test_binary_formats_host_side(tmp_path):
    """formats.NpyShardWriter writes a valid .npy in row blocks; load_sparse_npz reads scipy's layout."""
    import scipy.sparse as sp
    from prosstt_b200 import formats
    X = np.arange(35, dtype=np.int32).reshape(7, 5)
    path = formats.shard_path(str(tmp_path / "sim"), 0, 1)
    assert path.endswith("sim.npy") and formats.shard_path("s", 3, 8) == "s.rank3of8.npy"
    with formats.NpyShardWriter(path, 7, 5) as w:
        w.append(X[:3])
        w.append(X[3:])
    assert np.array_equal(np.load(path), X) and np.load(path).dtype == np.int32
    w = formats.NpyShardWriter(str(tmp_path / "short.npy"), 7, 5)
    w.append(X[:3])
    with pytest.raises(ValueError):
        w.close()                                          # rows missing
    w = formats.NpyShardWriter(str(tmp_path / "long.npy"), 2, 5)
    with pytest.raises(ValueError):
        w.append(X)                                        # too many rows
    with pytest.raises(ValueError):
        w.append(X[:1, :4])                                # wrong width
    m = sp.csr_matrix(np.array([[0, 2, 0], [0, 0, 0], [5, 0, 7]], dtype=np.int32))
    sp.save_npz(str(tmp_path / "m.npz"), m)
    ip, ix, da, shape = formats.load_sparse_npz(str(tmp_path / "m.npz"))
    assert shape == (3, 3) and np.array_equal(formats.csr_to_dense(ip, ix, da, shape), m.toarray())
    sp.save_npz(str(tmp_path / "c.npz"), m.tocsc())
    with pytest.raises(ValueError):
        formats.load_sparse_npz(str(tmp_path / "c.npz"))


def test_widen_host_side():
    from prosstt_b200 import formats
    X16 = np.array([[1, 65535, 3], [65535, 0, 65534]], dtype=np.uint16)
    full = formats.widen(X16, {"index": np.array([1, 3]), "value": np.array([65535, 123456], dtype=np.int32)})
    assert full.dtype == np.int32 and full.tolist() == [[1, 65535, 3], [123456, 0, 65534]]
    X8 = np.array([[255, 254], [0, 255]], dtype=np.uint8)
    assert formats.widen(X8, (np.array([0, 3]), np.array([255, 1000], dtype=np.int32))).tolist() == [[255, 254], [0, 1000]]
    with pytest.raises(ValueError):
        formats.widen(X16, (np.array([1]), np.array([70000])))          # a saturated element is not listed
    with pytest.raises(TypeError):
        formats.widen(X16.astype(np.int16), (np.array([], dtype=np.int64), np.array([], dtype=np.int32)))


def test_epilogue_argument_checks_without_a_gpu():
    """stats / formats reject anything that is not a 2-D int32 CUDA tensor before touching the library."""
    import torch
    from prosstt_b200 import formats, stats
    cpu = torch.zeros((3, 4), dtype=torch.int32)
    for fn in (stats.count_stats, stats.log1p, formats.to_csr):
        with pytest.raises(TypeError):
            fn(cpu)
    with pytest.raises(TypeError):
        stats.transform_counts(cpu.float(), None, "log1p")
    with pytest.raises(TypeError):
        formats.widen(np.zeros((2, 2), dtype=np.int32), (np.array([]), np.array([])))


def test_host_side_helpers_of_the_device_to_host_path():
    """pst_host_widen / pst_host_apply_overflow / pst_host_checksum / pst_host_prepare are plain host code
    (threads, no CUDA): every supported width pair, ragged sizes, thread counts, the overflow fix-up."""
    import ctypes
    lib = nat.load()
    rng = np.random.RandomState(5)
    for n in (0, 1, 63, 64, 1000003):
        for sb, sdt, hi in ((8, np.uint8, 255), (16, np.uint16, 65535), (32, np.int32, 2 ** 31 - 1)):
            src = rng.randint(0, hi + 1, size=n, dtype=np.int64).astype(sdt)
            for db, ddt in ((32, np.int32), (64, np.int64)):
                dst = np.full(n, -1, dtype=ddt)
                for threads in (1, 3, 0):
                    dst[:] = -1
                    assert lib.pst_host_widen(src.ctypes.data, sb, dst.ctypes.data, db, n, threads) == 0
                    assert np.array_equal(dst, src.astype(ddt)), (n, sb, db, threads)
                # streaming-store form: same result for any alignment of the destination, nothing written
                # outside [0, n)
                for off in (0, 1, 5):
                    if n <= off:
                        continue
                    pad = np.full(n + 32, -7, dtype=ddt)
                    assert lib.pst_host_widen_stream(src[off:].ctypes.data, sb, pad[off + 3:].ctypes.data, db,
                                                     n - off, 3) == 0
                    assert np.array_equal(pad[off + 3:n + 3], src[off:].astype(ddt)), (n, sb, db, off)
                    assert (pad[:off + 3] == -7).all() and (pad[n + 3:] == -7).all()
    assert lib.pst_host_widen(None, 8, None, 32, 5, 1) == -1
    assert lib.pst_host_widen_stream(None, 8, None, 32, 5, 1) == -1
    a = np.zeros(4, np.int32)
    assert lib.pst_host_widen(a.ctypes.data, 32, a.ctypes.data, 16, 4, 1) == -1          # unsupported pair
    # overflow list: entries inside [base, base + n) overwrite, the rest are skipped
    dst = np.arange(10, dtype=np.int64)
    idx = np.array([3, 12, 25, 19], dtype=np.int64)
    val = np.array([300, 1200, 2500, 1900], dtype=np.int32)
    assert lib.pst_host_apply_overflow(dst.ctypes.data, 64, 10, 10, idx.ctypes.data, val.ctypes.data, 4) == 0
    assert dst.tolist() == [0, 1, 1200, 3, 4, 5, 6, 7, 8, 1900]
    d32 = np.zeros(5, dtype=np.int32)
    assert lib.pst_host_apply_overflow(d32.ctypes.data, 32, 0, 5, idx.ctypes.data, val.ctypes.data, 4) == 0
    assert d32.tolist() == [0, 0, 0, 300, 0]
    words = rng.randint(0, 2 ** 32, size=300001, dtype=np.uint64).astype(np.uint32)
    lib.pst_host_checksum.restype = ctypes.c_uint64
    for threads in (1, 4, 0):
        assert lib.pst_host_checksum(words.ctypes.data, words.nbytes, threads) == int(words.astype(np.uint64).sum())
    big = np.empty(8 << 20, dtype=np.uint8)
    assert lib.pst_host_prepare(big.ctypes.data, big.nbytes) in (0, 1)                   # advice only
    assert lib.pst_host_prepare(None, 0) == 1
    lay = (ctypes.c_int64 * 6)()
    assert lib.pst_draw_scratch_layout(1000, 400, 37, lay) == 0
    assert lib.pst_draw_scratch_words(1000, 400, 37) == lay[4] + 4 * lay[5] and lay[4] % 4 == 0
    assert lay[1] == 4 + 4 * lay[0] and lay[2] == lay[1] + 1000 and lay[3] == lay[2] + 38


def test_chunk_plan_covers_every_cell_once_in_order():
    """device._plan_chunks: the chunks of every chunked device->host call.  A budget gives chunks of
    budget // cell_bytes cells after a ramp of 1/8, 1/4 and 1/2 of that; an explicit chunk size has no ramp."""
    from prosstt_b200.device import _plan_chunks
    assert _plan_chunks(1000, None, 40, 40 * 80) == (80, [(0, 10), (10, 30), (30, 70)]
                                                     + [(lo, min(1000, lo + 80)) for lo in range(70, 1000, 80)])
    assert _plan_chunks(1000, 300, 40, 40 * 80) == (300, [(0, 300), (300, 600), (600, 900), (900, 1000)])
    assert _plan_chunks(0, None, 40, 1 << 30) == (1, [])
    assert _plan_chunks(0, 7, 40, 1 << 30) == (1, [])
    # n smaller than one chunk: the ramp still applies (chunk 5 -> 1, 1, 2, then the rest), an explicit size not
    assert _plan_chunks(5, None, 40, 1 << 30) == (5, [(0, 1), (1, 2), (2, 4), (4, 5)])
    assert _plan_chunks(5, 100, 40, 1 << 30) == (5, [(0, 5)])
    assert _plan_chunks(3, None, 40, 1) == (1, [(0, 1), (1, 2), (2, 3)])        # budget below one cell
    for n in (1, 2, 7, 100, 1001):
        for chunk_cells in (None, 1, 3, 97, 5000):
            for cell_bytes, budget in ((0, 64), (4, 64), (40, 4000), (4, 1 << 30)):
                chunk, bounds = _plan_chunks(n, chunk_cells, cell_bytes, budget)
                assert [c for lo, hi in bounds for c in range(lo, hi)] == list(range(n))
                assert all(1 <= hi - lo <= chunk for lo, hi in bounds) and chunk <= n
                if chunk_cells is not None:
                    assert all(hi - lo == min(chunk_cells, n) for lo, hi in bounds[:-1])


def test_result_pool_recycles_only_unreachable_matrices():
    """hostpool: the buffer of a result comes back when the array AND every view of it are gone, is handed
    out again for a matrix of similar size, and PST_HOST_POOL_GB=0 turns the pool off."""
    import gc
    from prosstt_b200 import hostpool as hp
    hp.release()
    a, fresh = hp.result_array((1000, 2000), np.int64)
    assert fresh and a.shape == (1000, 2000) and a.dtype == np.int64
    assert a.flags.writeable and a.flags.c_contiguous
    a[:] = 7
    view = a[10:20, ::2]
    del a
    gc.collect()
    assert hp.retained_bytes() == 0 and (view == 7).all()          # a view keeps the memory out of the pool
    del view
    gc.collect()
    assert hp.retained_bytes() == 16 << 20
    b, fresh = hp.result_array((999, 2000), np.int64)              # similar size: the same memory again
    assert not fresh and hp.retained_bytes() == 0 and b.shape == (999, 2000)
    c, fresh = hp.result_array((999, 2000), np.int64)              # the first is still alive: new memory
    assert fresh
    # private memory like np.empty's: what a forked child writes stays in the child
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", DeprecationWarning)        # "multi-threaded process": the child only writes and exits
        pid = os.fork()
    if pid == 0:
        b[:] = 9
        os._exit(0 if int(b[5, 5]) == 9 else 1)
    assert os.waitpid(pid, 0)[1] == 0 and int(b[5, 5]) == 7
    del b, c
    gc.collect()
    small, fresh = hp.result_array((100, 2000), np.int32)          # far smaller than what is retained: not reused
    assert fresh and small.flags.owndata
    hp.release()
    assert hp.retained_bytes() == 0
    old = os.environ.get("PST_HOST_POOL_GB")
    os.environ["PST_HOST_POOL_GB"] = "0"
    try:
        d, fresh = hp.result_array((1000, 2000), np.int64)
        assert fresh and d.flags.owndata
        del d
        gc.collect()
        assert hp.retained_bytes() == 0
    finally:
        if old is None:
            del os.environ["PST_HOST_POOL_GB"]
        else:
            os.environ["PST_HOST_POOL_GB"] = old


def test_default_transport_is_a_fixed_rule_of_cpu_and_threads(monkeypatch):
    """The transport nobody asked for (device.py:_shared_host_transport) must be the same on every rank of a
    job: a function of the CPU's store instructions and the rank's thread count only, overridable by
    PST_HOST_TRANSPORT; the thread count is the rank's share of the cores (LOCAL_WORLD_SIZE)."""
    from prosstt_b200 import device as pdev
    monkeypatch.delenv("PST_HOST_TRANSPORT", raising=False)
    streams = bool(nat.load().pst_host_stream_stores())
    need = 3 if streams else 10
    assert pdev._shared_host_transport(need) == "u8" and pdev._shared_host_transport(need - 1) == "direct"
    assert pdev._shared_host_transport(64) == "u8" and pdev._shared_host_transport(1) == "direct"
    monkeypatch.setenv("PST_HOST_TRANSPORT", "u16")
    assert pdev._shared_host_transport(1) == "u16" and pdev._shared_host_transport(64) == "u16"
    cores = len(os.sched_getaffinity(0))
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "1")
    assert pdev._host_threads() == cores
    monkeypatch.setenv("LOCAL_WORLD_SIZE", str(4 * cores))
    assert pdev._host_threads() == 1
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "not a number")
    assert pdev._host_threads() == cores
