"""The oracle (and, on the GPU, the CUDA kernels) against THE REFERENCE'S OWN DEVICE CODE.

tests/golden/ref_kernels.npz was produced by running the __global__ / __device__ function bodies of the reference's
Hash3DAnchored_cuda.cu and PersSampler_cuda.cu -- extracted where they lie under /root/reference and compiled for the
host between two small shims (oracle/ref_extract.py, ref_driver.cpp, ref_shim/; `make -C oracle ref`) -- on the inputs
stored beside the outputs.  This is what pins Hash3DAnchored, the octree traversal, the march, the occupancy vote and
the cold queries to the reference's code rather than to a reading of it.  It already paid for itself: it exposed
that the reference adds its per-level ROW offset to a SCALAR pointer (level windows overlap by half; see
level_base_row in oracle/gf_oracle.c), which the first restatement had missed.

Bars.  Integer results (table rows via the zero pattern, leaf lists, sample counts, anchors, vote statistics, pruned
leaves, point anchors) are exact.  fp32 results: the reference binary is built by nvcc, which fuses mul+add pairs
where it chooses; the fixture by g++, which fuses where IT chooses; the oracle spells out nvcc's choices.  So
straight-line results (hash blend, near/far, warp) agree to the last bit or a few ulp, and the march -- a recurrence
of up to 1024 steps -- to 1e-4 relative, the sample COUNTS still being identical.

Where oracle/_ref/*.so exists (built in this container by __graft_entry__.build()) the same comparisons also run
live on larger random inputs and on both contraction flavours."""
import os

import numpy as np
import pytest

from oracle import oracle as orc
from oracle import ref_host as rh
from tests.helpers import hash_inputs, load_rig

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernels.npz")
S = 1024


@pytest.fixture(scope="module")
def fx():
    d = np.load(GOLD)
    return {k: d[k] for k in d.files}


@pytest.fixture(scope="module")
def rig():
    return load_rig("rig8")


def rel_close(a, b, rtol, what):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    err = np.abs(a - b) / np.maximum(np.abs(b), 1e-3)
    assert err.max() <= rtol, f"{what}: max rel err {err.max():.3e} (> {rtol})"


# ------------------------------------------------------------------ Hash3DAnchored
@pytest.mark.parametrize("tag", ["h0", "h1"])
def test_hash_forward_is_the_reference_kernel_bit_for_bit(fx, tag):
    out = orc.hash_forward(fx[f"{tag}_feat"], fx[f"{tag}_prim"], fx[f"{tag}_bias"], fx[f"{tag}_pts"], fx[f"{tag}_anchors"])
    assert np.array_equal(out, fx[f"{tag}_out"].astype(np.float32))


@pytest.mark.parametrize("tag", ["h0", "h1"])
def test_hash_rows_reach_only_the_reference_windows(fx, tag):
    """The reference offsets a scalar pointer by l * local_size: level l owns rows [l*T/2, l*T/2 + T)."""
    L = int(fx[f"{tag}_local"])
    _, idx = orc.hash_forward(fx[f"{tag}_feat"], fx[f"{tag}_prim"], fx[f"{tag}_bias"], fx[f"{tag}_pts"],
                              fx[f"{tag}_anchors"], want_idx=True)
    base = (np.arange(16) * L // 2).reshape(1, 16, 1)
    assert np.all(idx >= base) and np.all(idx < base + L)
    # the reference's gradient lands on exactly the rows the oracle computes (rows of zero-gradient samples excluded)
    live = np.abs(fx[f"{tag}_grad"]).reshape(-1, 16, 2).max(-1) > 0
    touched = np.zeros(16 * L, bool)
    touched[idx[live]] = True
    ref_nonzero = (fx[f"{tag}_gtable"] != 0).any(-1)
    assert not ref_nonzero[~touched].any()                       # nothing outside
    assert not ref_nonzero[17 * L // 2:].any()                   # in particular nothing past 8.5 T
    assert ref_nonzero[touched].mean() > 0.9                     # (tiny products round to zero in fp16)


@pytest.mark.parametrize("tag", ["h0", "h1"])
def test_hash_backward_matches_the_reference_kernel(fx, tag):
    L = int(fx[f"{tag}_local"])
    args = (L, fx[f"{tag}_prim"], fx[f"{tag}_bias"])
    # six points, every row hit at most once per level pair: nothing accumulates, so the fp16 atomics are exact and
    # so must the oracle be (same x128 -> fp16 quantisation of the gradient and of every product)
    few = slice(0, 6)
    g = orc.hash_backward(*args, fx[f"{tag}_pts"][few], fx[f"{tag}_anchors"][few], fx[f"{tag}_grad"][few] * 50)
    ref = fx[f"{tag}_gtable_few"]
    _, idx = orc.hash_forward(fx[f"{tag}_feat"], fx[f"{tag}_prim"], fx[f"{tag}_bias"], fx[f"{tag}_pts"][few],
                              fx[f"{tag}_anchors"][few], want_idx=True)
    hits = np.bincount(idx.reshape(-1), minlength=16 * L)
    once = hits == 1
    assert once.sum() > 400
    assert np.array_equal(g[once].astype(np.float32), ref[once])
    # the full batch: the reference accumulates in fp16 (order-dependent), the oracle in fp64
    g = orc.hash_backward(*args, fx[f"{tag}_pts"], fx[f"{tag}_anchors"], fx[f"{tag}_grad"])
    ref = fx[f"{tag}_gtable"].astype(np.float64)
    assert np.linalg.norm(g - ref) <= 5e-3 * np.linalg.norm(ref)


# ------------------------------------------------------------------ PersSampler
def run_oracle_sampler(fx, rig, mode):
    return orc.sampler_get_samples(fx["s_rays_o"], fx["s_rays_d"], fx[f"s_{mode}_noise"], rig["tree_nodes"],
                                   rig["pers_trans"], want_oct=True)


def test_search_order_table_runs_the_reference_traversal(fx):
    assert np.array_equal(orc.search_order(), fx["s_search_order"])


@pytest.mark.parametrize("mode", ["eval", "train"])
def test_traversal_leaf_lists_are_the_reference_kernels(fx, rig, mode):
    a = run_oracle_sampler(fx, rig, mode)
    n_oct = fx[f"s_{mode}_n_oct"]
    assert np.array_equal(a["n_oct"], n_oct)
    k = fx[f"s_{mode}_oct_idx"].shape[1]
    assert np.array_equal(a["oct_idx"][:, :k], fx[f"s_{mode}_oct_idx"])
    assert np.array_equal(a["oct_nf"][:, :k], fx[f"s_{mode}_oct_nf"])        # slab test: no contraction to differ on
    assert np.array_equal(a["first_oct_dis"], fx[f"s_{mode}_first_oct_dis"])
    assert n_oct[-1] == 0 and n_oct[-2] == 0 and n_oct.max() > 8             # the two rays that miss; deep rays


@pytest.mark.parametrize("mode", ["eval", "train"])
def test_march_counts_anchors_and_positions(fx, rig, mode):
    a = run_oracle_sampler(fx, rig, mode)
    counts = fx[f"s_{mode}_counts"]
    assert np.array_equal(a["counts"], counts)                               # bit-exact sample counts
    se = fx[f"s_{mode}_pts_idx_start_end"]
    assert np.array_equal(se[:, 1] - se[:, 0], counts) and np.array_equal(se[:, 0], np.cumsum(counts) - counts)
    m = np.arange(S)[None, :] < counts[:, None]
    assert np.array_equal(a["anchors"][m], fx[f"s_{mode}_anchors"])          # (trans_idx, node_idx, block_idx)
    rel_close(a["ts"][m], fx[f"s_{mode}_ts"], 1e-4, "t")
    rel_close(a["dists"][m], fx[f"s_{mode}_dists"], 1e-4, "dist")
    assert np.abs(a["warp_pts"][m] - fx[f"s_{mode}_warp_pts"]).max() <= 2e-4   # warp coordinates are O(1)
    assert (a["ts"][m] == fx[f"s_{mode}_ts"]).mean() > 0.9                   # and most are the same bits
    assert bool(fx[f"s_{mode}_dirs_ok"])


def test_vote_statistics_and_pruning(fx, rig):
    a = run_oracle_sampler(fx, rig, "eval")
    nodes = rig["tree_nodes"].copy()
    ws, as_, vc = fx["v_ws_in"].copy(), fx["v_as_in"].copy(), np.zeros(nodes.size // 128, np.int64)
    orc.update_oct_nodes(a["counts"], a["anchors"][..., 1].reshape(-1), fx["v_weights"].astype(np.float32).reshape(-1),
                         fx["v_alphas"].astype(np.float32).reshape(-1), nodes, ws, as_, vc)
    assert np.array_equal(ws, fx["v_ws"]) and np.array_equal(as_, fx["v_as"]) and np.array_equal(vc, fx["v_cnt"])
    assert np.array_equal(nodes.view(np.int64).reshape(-1, 16)[:, 12], fx["v_trans_idx"])


def test_cold_queries(fx, rig):
    got = orc.trans_query_frame(rig["tree_nodes"], rig["pers_trans"], fx["q_anchors"], fx["q_pts"])
    assert np.array_equal(got == 0, fx["q_out"] == 0)                        # the rows the kernel leaves untouched
    assert np.abs(got - fx["q_out"]).max() <= 1e-5 * max(1.0, np.abs(fx["q_out"]).max())
    pa = orc.points_anchors(fx["s_rays_o"][:64], fx["s_rays_d"][:64], fx["p_t_cur"], rig["tree_nodes"])
    assert np.array_equal(pa, fx["p_anchors"])
    from tests.golden.make_golden_ref_kernels import edge_pool_of
    pts, ids = orc.edge_samples(edge_pool_of(rig["tree_nodes"]), rig["pers_trans"], fx["e_idx"], fx["e_coord"])
    assert np.array_equal(ids, fx["e_ids"])
    assert np.abs(pts - fx["e_pts"]).max() <= 1e-5 * max(1.0, np.abs(fx["e_pts"]).max())


# ------------------------------------------------------------------ live, where the reference build exists
live = pytest.mark.skipif(not (rh.available("off") and rh.available("fma")),
                          reason="oracle/_ref not built (needs /root/reference: build container only)")


@live
@pytest.mark.parametrize("flavour", ["off", "fma"])
def test_live_hash_forward_large(flavour):
    feat, prim, bias, pts, anchors = hash_inputs(20000, 7, 14, seed=3, along_rays=False)
    o = orc.hash_forward(feat, prim, bias, pts, anchors)
    r = rh.hash_forward(feat, prim, bias, pts, anchors, flavour=flavour)
    if flavour == "fma":
        assert np.array_equal(o, r)
    else:   # no contraction at all: a handful of blends round the other way, by one fp16 ulp
        assert (o == r).mean() > 0.999 and np.abs(o - r).max() <= 2.0 ** -10 * np.abs(r).max()


@live
@pytest.mark.parametrize("flavour", ["off", "fma"])
def test_live_sampler_2000_rays(rig, flavour):
    from gfnerf_b200.persoctree import rig_rays
    R = 2000
    o, d, _ = rig_rays(rig["c2w"], rig["intri"], R, seed=41)
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    noise = np.random.RandomState(7).uniform(0.5, 1.5, S + R + 10).astype(np.float32)
    a = orc.sampler_get_samples(o, d, noise, rig["tree_nodes"], rig["pers_trans"], want_oct=True)
    b = rh.get_samples(o, d, noise, rig["tree_nodes"], rig["pers_trans"], orc.search_order(), flavour=flavour)
    assert np.array_equal(a["n_oct"], b["n_oct"]) and np.array_equal(a["oct_idx"], b["oct_idx"])
    assert np.array_equal(a["oct_nf"], b["oct_nf"])
    # counts: the march compares accumulated fp32 positions with leaf borders, so a different contraction may move a
    # border sample across; with g++'s contraction no ray does, without any contraction a few may
    same = a["counts"] == b["counts"]
    assert same.mean() >= (1.0 if flavour == "fma" else 0.99), same.mean()
    m = (np.arange(S)[None, :] < a["counts"][:, None]) & same[:, None]
    tol = 1e-4 if flavour == "fma" else 1e-2
    rel_close(a["ts"][m], b["ts"][m], tol, "t")
    if flavour == "fma":
        assert np.array_equal(a["anchors"][m], b["anchors"][m])
        assert np.abs(a["world_pts"][m] - b["world_pts"][m]).max() <= 1e-4 * np.abs(b["world_pts"][m]).max()


@pytest.mark.parametrize("name", ["rig8", "rig20"])
def test_octree_marks_match_the_reference_fixture(name):
    """orc_mark_invisible_nodes / orc_set_block_idxs against the reference's own MarkInvisibleNodesKernel /
    SetBlockIdxsNearestKernel outputs stored in tests/golden/ref_marks.npz (tests/golden/make_golden_marks.py): the
    per-node trans_idx and block_idx are identical, and nothing else in the 128-byte blobs moves."""
    fx = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_marks.npz"))
    tree = load_rig(name)["tree_nodes"]
    nodes = orc.mark_invisible_nodes(tree, fx[f"{name}_intri"], fx[f"{name}_w2c"], fx[f"{name}_bounds"])
    nodes = orc.set_block_idxs(nodes, fx[f"{name}_centers"])
    blob, before = nodes.view(np.int64).reshape(-1, 16), tree.view(np.int64).reshape(-1, 16)
    assert np.array_equal(blob[:, 12], fx[f"{name}_trans_idx"]) and np.array_equal(blob[:, 13], fx[f"{name}_block_idx"])
    keep = [c for c in range(16) if c not in (12, 13)]
    assert np.array_equal(blob[:, keep], before[:, keep])
    assert not np.isin(blob[:, 13], (5, 6)).any()                             # ties: the first of equal minima


@live
def test_live_threaded_launches_give_the_serial_results(rig):
    """oracle/_ref with ref_set_threads(n > 1) -- what bench.py's CPU arm (kind "reference") runs: the thread instances
    of a launch spread over host threads, the shim's atomics real atomics.  Everything that does not depend on the
    ORDER of atomics is identical to the serial emulation: samples, anchors, ranges, hash encodings, vote statistics;
    the fp16 gradient sums agree like two runs of the reference on a GPU do."""
    from gfnerf_b200.persoctree import rig_rays
    R = 192
    o, d, _ = rig_rays(rig["c2w"], rig["intri"], R, seed=31)
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    noise = np.random.RandomState(2).uniform(0.5, 1.5, S + R + 10).astype(np.float32)
    feat, prim, bias, _, _ = hash_inputs(8, rig["pers_trans"].size // 576, 12, seed=4)
    out = {}
    try:
        for n in (1, 5):
            rh.set_threads(n, "fma")
            smp = rh.get_samples(o, d, noise, rig["tree_nodes"], rig["pers_trans"], orc.search_order(), flavour="fma")
            m = smp["counts"][:, None] > np.arange(S)[None]
            pts = ((smp["warp_pts"][m] + 1.5) / 3).astype(np.float32)
            anc = np.ascontiguousarray(smp["anchors"][m][:, 0])
            enc = rh.hash_forward(feat, prim, bias, pts, anc, "fma")
            g = (np.random.RandomState(3).normal(size=(pts.shape[0], 32)) * 1e-3).astype(np.float32)
            gt = rh.hash_backward(feat.shape[0] // 16, prim, bias, pts, anc, g, "fma")
            nodes, ws, as_ = rig["tree_nodes"].copy(), np.full(rig["tree_nodes"].size // 128, 3, np.int64), \
                np.full(rig["tree_nodes"].size // 128, 3, np.int64)
            vc = np.zeros_like(ws)
            w = np.random.RandomState(4).uniform(0, 0.02, size=(R, S)).astype(np.float32)
            rh.update_oct_nodes(smp["pts_idx_start_end"], smp["anchors"][..., 1].reshape(-1), w.reshape(-1),
                                (w * 2).reshape(-1), nodes, ws, as_, vc, flavour="fma")
            out[n] = (smp, enc, gt, nodes, ws, as_, vc)
    finally:
        rh.set_threads(1, "fma")
    a, b = out[1], out[5]
    for k in ("counts", "pts_idx_start_end", "anchors", "ts", "dists", "warp_pts", "world_pts", "first_oct_dis", "n_oct"):
        assert np.array_equal(a[0][k], b[0][k]), k
    assert np.array_equal(a[1], b[1])
    assert all(np.array_equal(x, y) for x, y in zip(a[3:], b[3:]))
    assert np.linalg.norm(a[2] - b[2]) <= 2e-2 * np.linalg.norm(a[2])         # fp16 sums in another order


def _camera_subset(rig, n=6):
    c2w = rig["c2w"][:n]
    m = np.tile(np.eye(4, dtype=np.float32)[None], (c2w.shape[0], 1, 1))
    m[:, :3, :] = c2w
    w2c = np.ascontiguousarray(np.linalg.inv(m)[:, :3, :].astype(np.float32))
    return w2c, np.ascontiguousarray(rig["intri"][:n]), np.ascontiguousarray(rig["bounds"][:n])


@live
def test_live_mark_invisible_nodes_is_the_reference_kernel(rig):
    """The oracle's MarkInvisibleNodes (the checker of gf_octree_mark_invisible, tests/test_octree_device_gpu.py) against
    the reference's MarkInvisibleNodesKernel / CheckVisible (PersSampler_cuda.cu:680-723) compiled for the host, on the
    rig's tree with a camera subset so that a good part of the nodes really is out of sight.  The oracle spells out
    nvcc's contraction of the reference's expressions (the GPU test holds the kernel to the nvcc-built reference
    kernel bit for bit); g++ contracts them its own way, so a node whose bounding sphere touches a frustum edge within
    fp rounding may fall either way here."""
    w2c, intri, bound = _camera_subset(rig)
    tidx0 = rig["tree_nodes"].view(np.int64).reshape(-1, 16)[:, 12].copy()
    mine = orc.mark_invisible_nodes(rig["tree_nodes"], intri, w2c, bound)
    n_marked = ((mine.view(np.int64).reshape(-1, 16)[:, 12] == -1) & (tidx0 != -1)).sum()
    assert 0 < n_marked < (tidx0 != -1).sum()
    for flavour in ("off", "fma"):
        nodes_ref = rig["tree_nodes"].copy()
        rh.mark_invisible_nodes(nodes_ref, intri, w2c, bound, flavour=flavour)
        # only trans_idx may change, and on at most two borderline nodes differently
        assert (mine != nodes_ref).sum() <= 2 * 8, (flavour, (mine != nodes_ref).sum())
    # no camera at all: every node loses its transform (the reference's count stays 0)
    none = orc.mark_invisible_nodes(rig["tree_nodes"], intri[:0], w2c[:0], bound[:0])
    assert (none.view(np.int64).reshape(-1, 16)[:, 12] == -1).all()


@live
def test_live_nearest_block_is_the_reference_kernel(rig):
    """The oracle's SetBlockIdxsNearest (the checker of gf_octree_set_block_idxs) against SetBlockIdxsNearestKernel
    (PersSampler_cuda.cu:746-766), incl. exact ties (duplicated centres: the first wins, strict `<`)."""
    centers = np.random.RandomState(0).uniform(-4, 4, size=(5, 3)).astype(np.float32)
    centers = np.concatenate([centers, centers[1:3]], 0)                      # blocks 5, 6 duplicate 1, 2
    got = orc.set_block_idxs(rig["tree_nodes"], centers).view(np.int64).reshape(-1, 16)[:, 13]
    assert got.max() <= 4 and got.min() >= 0
    for flavour in ("off", "fma"):
        nodes_ref = rig["tree_nodes"].copy()
        rh.set_block_idxs(nodes_ref, centers, flavour=flavour)
        want = nodes_ref.view(np.int64).reshape(-1, 16)[:, 13]
        assert (got != want).sum() <= 2, (flavour, (got != want).sum())       # (fp32 norm rounding at near-ties)
    # nothing closer than 1e9: the index stays -1
    far = orc.set_block_idxs(rig["tree_nodes"], np.full((2, 3), 3e9, np.float32))
    assert (far.view(np.int64).reshape(-1, 16)[:, 13] == -1).all()


def _history(rig, trial, rng):
    """A training history on the rig's tree: some leaves voted empty, random statistics and visit counts."""
    nodes = rig["tree_nodes"].copy()
    tidx = nodes.view(np.int64).reshape(-1, 16)[:, 12]
    n = tidx.shape[0]
    leaves = np.nonzero(tidx >= 0)[0]
    tidx[rng.choice(leaves, size=int(len(leaves) * (0.2 + 0.3 * trial)), replace=False)] = -1
    return (nodes, rng.randint(-100, 5000, size=n).astype(np.int64), rng.randint(-100, 5000, size=n).astype(np.int64),
            rng.randint(0, 12, size=n).astype(np.int64))


def _our_proc_octree(nodes, w, a, v, compact, subdivide, brute):
    import ctypes as C
    from gfnerf_b200 import _lib
    L, n_out = _lib.lib(), C.c_int64(0)
    args = (nodes.ctypes.data, nodes.size // 128, w.ctypes.data, a.ctypes.data, v.ctypes.data, int(compact),
            int(subdivide), int(brute))
    _lib.check(L.gf_octree_proc(*args, None, None, None, 0, C.byref(n_out)))
    n = n_out.value
    o_nodes, o_w, o_a = np.empty(n * 128, np.uint8), np.empty(n, np.int64), np.empty(n, np.int64)
    _lib.check(L.gf_octree_proc(*args, o_nodes.ctypes.data, o_w.ctypes.data, o_a.ctypes.data, n, C.byref(n_out)))
    return o_nodes, o_w, o_a


def test_proc_octree_and_edge_pool_match_the_reference_digests(fx, rig):
    """gf_octree_proc / gf_octree_edge_pool against digests of what the reference's own PersOctree::ProcOctree and
    ConstructEdgePool bodies produced on the same inputs (node count + sha256 of node blob / weight / alpha stats)."""
    import hashlib
    from tests.golden.make_golden_ref_kernels import edge_pool_of
    dig = lambda x: int(hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()[:15], 16)
    rng = np.random.RandomState(5)
    for trial in range(3):
        nodes, w, a, v = _history(rig, trial, rng)
        for tag, flags in (("c", (True, False, False)), ("cs", (True, True, False)), ("csb", (True, True, True))):
            out = _our_proc_octree(nodes, w, a, v, *flags)
            assert [out[0].size // 128] + [dig(x) for x in out] == fx[f"o_{trial}_{tag}"].tolist(), (trial, tag)
    ep = edge_pool_of(rig["tree_nodes"])
    used = np.arange(ep.size) % 64 < 52
    assert [ep.size // 64, dig(ep[used])] == fx["o_edge_pool"].tolist()


@live
@pytest.mark.parametrize("compact,subdivide,brute", [(True, False, False), (True, True, False), (True, True, True),
                                                      (False, True, False), (False, False, False)])
def test_live_proc_octree_is_the_reference_function(rig, compact, subdivide, brute):
    """gf_octree_proc (csrc/octree_host.cu) against the reference's own PersOctree::ProcOctree body
    (PtsSampler/PersSampler.cpp:154-417) on the same blobs: node array byte for byte, statistics identical; and the
    milestone sequence of UpdateOctNodes (:662-667): ProcOctree(true, true, .) then ProcOctree(true, false, false)."""
    rng = np.random.RandomState(5)
    for trial in range(3):
        nodes, w, a, v = _history(rig, trial, rng)
        if not compact:
            # without the compaction pass pruned leaves stay linked: the reference's CHECK_GE (PersSampler.cpp:315)
            # aborts -- and so does ours; a compacted tree goes through both
            with pytest.raises(RuntimeError, match="CHECK"):
                rh.proc_octree(nodes, w, a, v, compact, subdivide, brute)
            with pytest.raises(RuntimeError, match="removed"):
                _our_proc_octree(nodes, w, a, v, compact, subdivide, brute)
            nodes, w, a = rh.proc_octree(nodes, w, a, v, True, False, False)
            v = rng.randint(0, 12, size=w.shape[0]).astype(np.int64)
        ref = rh.proc_octree(nodes, w, a, v, compact, subdivide, brute)
        got = _our_proc_octree(nodes, w, a, v, compact, subdivide, brute)
        assert got[0].size == ref[0].size
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])
        if subdivide:   # the second call of a milestone, on the first call's output (visit counts restart at 0)
            z = np.zeros(ref[1].shape[0], np.int64)
            ref2 = rh.proc_octree(ref[0], ref[1], ref[2], z, True, False, False)
            got2 = _our_proc_octree(got[0], got[1], got[2], z, True, False, False)
            assert all(np.array_equal(x, y) for x, y in zip(got2, ref2))


@live
def test_live_edge_pool_is_the_reference_function(rig):
    """gf_octree_edge_pool against the reference's own PersOctree::ConstructEdgePool body (:833-895)."""
    from tests.golden.make_golden_ref_kernels import edge_pool_of
    rng = np.random.RandomState(2)
    for trial in range(2):
        nodes = _history(rig, trial, rng)[0] if trial else rig["tree_nodes"].copy()
        ref = rh.construct_edge_pool(nodes)
        got = edge_pool_of(nodes)
        assert ref.size > 0 and ref.size % 64 == 0
        # the 12 padding bytes of each 64-byte record (52 used) are indeterminate in the reference's push_back
        used = np.arange(ref.size) % 64 < 52
        assert got.size == ref.size and np.array_equal(got[used], ref[used])


# ------------------------------------------------------------------ GPU: the CUDA kernels against the same fixture
@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["h0", "h1"])
def test_cuda_hash_forward_is_the_reference_kernel_bit_for_bit(fx, tag):
    import torch
    from gfnerf_b200 import _lib
    L, n = int(fx[f"{tag}_local"]), fx[f"{tag}_pts"].shape[0]
    n_vol = fx[f"{tag}_prim"].shape[1]
    dev = "cuda"
    scales_d, scales_h = torch.empty(16, device=dev), np.zeros(16, np.float32)
    _lib.check(_lib.lib().gf_hash_level_scales(_lib.ptr(scales_d), scales_h.ctypes.data, _lib.cur_stream()))
    f16 = torch.from_numpy(fx[f"{tag}_feat"]).to(dev).half().contiguous()
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    tp, ta, tprim, tbias = T(fx[f"{tag}_pts"]), T(fx[f"{tag}_anchors"]), T(fx[f"{tag}_prim"].astype(np.int32)), T(fx[f"{tag}_bias"])
    out = torch.empty((n, 32), device=dev)
    _lib.check(_lib.lib().gf_hash_forward(n, None, n_vol, L, _lib.ptr(f16), _lib.ptr(tprim), _lib.ptr(tbias),
                                          _lib.ptr(scales_d), _lib.ptr(tp), _lib.ptr(ta), 1, None, _lib.ptr(out),
                                          _lib.cur_stream()))
    got, ref = out.cpu().numpy(), fx[f"{tag}_out"].astype(np.float32)
    # The fixture was computed on the host, where exp2f (the level scale, Hash3DAnchored_cuda.cu:28) is glibc's; the
    # device's exp2f may round the non-integer levels one ulp the other way, which moves the blend weights by ~1e-4 of
    # a cell and a fraction of the fp16-rounded outputs by one ulp.  (Against the oracle fed with the DEVICE scales the
    # kernel is bit-exact: tests/test_hash_gpu.py.)  Levels 0 and 15 have exact scales 8 and 1024: bit-exact here too.
    ulp = np.maximum(np.abs(ref), 2.0 ** -14) * 2.0 ** -10
    assert np.all(np.abs(got - ref) <= 2 * ulp + 4e-5)          # table values are O(1e-2)
    print("bit-equal fraction vs the reference kernel:", float((got == ref).mean()))
    assert (got == ref).mean() > 0.3
    assert np.array_equal(got[:, :2], ref[:, :2])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["eval", "train"])
def test_cuda_sampler_counts_and_anchors_are_the_reference_kernels(fx, rig, mode):
    import torch
    from tests.helpers import make_sampler
    from gfnerf_b200 import _lib
    s = make_sampler(rig, mode=1)
    R, dev = fx["s_rays_o"].shape[0], "cuda"
    to, td = torch.from_numpy(fx["s_rays_o"]).cuda(), torch.from_numpy(fx["s_rays_d"]).cuda()
    noise = torch.from_numpy(fx[f"s_{mode}_noise"]).cuda()
    # below GetSamples' normalisation of rays_d (the fixture's directions are the unit vectors the kernels saw)
    z = lambda *sh, dt=torch.float32: torch.zeros(sh, dtype=dt, device=dev)
    world, warp, dirs, anchors = z(R, S, 3), z(R, S, 3), z(R, S, 3), z(R, S, 3, dt=torch.int64)
    dists, ts, se, first, cnt = z(R, S), z(R, S), z(R, 2, dt=torch.int64), z(R, 1), z(R, dt=torch.int32)
    out = _lib.SamplerOut(world_pts=_lib.ptr(world), warp_pts=_lib.ptr(warp), dirs=_lib.ptr(dirs),
                          dists=_lib.ptr(dists), ts=_lib.ptr(ts), anchors_i64=_lib.ptr(anchors), anchors_i32=None,
                          pts_idx_start_end=_lib.ptr(se), counts=_lib.ptr(cnt), first_oct_dis=_lib.ptr(first),
                          n_oct=None, packed=None)
    s._launch(to, td, noise, out)
    torch.cuda.synchronize()
    counts = fx[f"s_{mode}_counts"]
    assert np.array_equal(cnt.cpu().numpy(), counts)
    assert np.array_equal(se.cpu().numpy(), fx[f"s_{mode}_pts_idx_start_end"])
    m = np.arange(S)[None, :] < counts[:, None]
    assert np.array_equal(anchors.cpu().numpy()[m], fx[f"s_{mode}_anchors"])
    rel_close(ts.cpu().numpy()[m], fx[f"s_{mode}_ts"], 1e-4, "t")
    rel_close(dists.cpu().numpy()[m], fx[f"s_{mode}_dists"], 1e-4, "dist")
    assert np.abs(warp.cpu().numpy()[m] - fx[f"s_{mode}_warp_pts"]).max() <= 2e-4
    np.testing.assert_allclose(first.cpu().numpy().reshape(-1), fx[f"s_{mode}_first_oct_dis"], rtol=1e-6)


# ------------------------------------------------------------------ GPU: beside the reference's kernels built by nvcc
# `make -C oracle ref_cuda` (needs the reference's source tree).  The bit-level pin the host build cannot give: nvcc's own
# FMA contraction of the reference's expressions.  First run (r02a, profiles/r02a_ref_cuda.log): hash forward, counts,
# anchors, first_oct_dis identical; t / warp differed in the last bits through two contractions read off the
# reference's SASS and now followed by kernel + oracle (the GEMV's rounded product is the second one; the leaf-crossing
# step is fused into `cur_t +=`).  Where that library is not built, a seeded sample of the same outputs stored in
# tests/golden/ref_cuda.npz stands in for it (tests/golden/make_golden_ref_cuda.py).
REF_CUDA_GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_cuda.npz")


def beside_nvcc_inputs(rig):
    """The inputs of the comparison with the nvcc-built reference kernels: a hash-encoding batch along rays and a
    sampler batch of 4096 rig rays (unit directions) with its march noise."""
    from gfnerf_b200.persoctree import rig_rays
    feat, prim, bias, pts, anchors = hash_inputs(200000, 7, 16, seed=3, along_rays=True)
    R = 4096
    o, d, _ = rig_rays(rig["c2w"], rig["intri"], R, seed=77)
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    noise = np.random.RandomState(5).uniform(0.5, 1.5, S + R + 10).astype(np.float32)
    return dict(feat=feat, prim=prim, bias=bias, pts=pts, anchors=anchors, o=o, d=d, noise=noise)


def cuda_beside_nvcc(rig, inp):
    """gf_hash_forward and the sampler's launch on `beside_nvcc_inputs` -> (sampler, dict of device tensors)"""
    import torch
    from gfnerf_b200 import _lib
    from tests.helpers import make_sampler
    dev = "cuda"
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    feat, prim, bias, pts, anchors = (inp[k] for k in ("feat", "prim", "bias", "pts", "anchors"))
    L = feat.shape[0] // 16
    scales_d, scales_h = torch.empty(16, device=dev), np.zeros(16, np.float32)
    _lib.check(_lib.lib().gf_hash_level_scales(_lib.ptr(scales_d), scales_h.ctypes.data, _lib.cur_stream()))
    f16 = T(feat).half().contiguous()
    tp, ta, tprim, tbias = T(pts), T(anchors), T(prim.astype(np.int32)), T(bias)
    hash_out = torch.empty((pts.shape[0], 32), device=dev)
    _lib.check(_lib.lib().gf_hash_forward(pts.shape[0], None, prim.shape[1], L, _lib.ptr(f16), _lib.ptr(tprim),
                                          _lib.ptr(tbias), _lib.ptr(scales_d), _lib.ptr(tp), _lib.ptr(ta), 1, None,
                                          _lib.ptr(hash_out), _lib.cur_stream()))
    s = make_sampler(rig, mode=1)
    R = inp["o"].shape[0]
    z = lambda *sh, dt=torch.float32: torch.zeros(sh, dtype=dt, device=dev)
    world, warp, dirs, anc = z(R, S, 3), z(R, S, 3), z(R, S, 3), z(R, S, 3, dt=torch.int64)
    dists, ts, se, first, cnt = z(R, S), z(R, S), z(R, 2, dt=torch.int64), z(R, 1), z(R, dt=torch.int32)
    so = _lib.SamplerOut(world_pts=_lib.ptr(world), warp_pts=_lib.ptr(warp), dirs=_lib.ptr(dirs),
                         dists=_lib.ptr(dists), ts=_lib.ptr(ts), anchors_i64=_lib.ptr(anc), anchors_i32=None,
                         pts_idx_start_end=_lib.ptr(se), counts=_lib.ptr(cnt), first_oct_dis=_lib.ptr(first),
                         n_oct=None, packed=None)
    s._launch(T(inp["o"]), T(inp["d"]), T(inp["noise"]), so)
    torch.cuda.synchronize()
    return s, dict(hash_out=hash_out, counts=cnt, first_oct_dis=first.view(-1), ts=ts, dists=dists, warp_pts=warp,
                   world_pts=world, anchors=anc)


@pytest.mark.gpu
def test_cuda_beside_the_reference_kernels_built_by_nvcc(rig):
    import torch
    inp = beside_nvcc_inputs(rig)
    s, got = cuda_beside_nvcc(rig, inp)
    # the stored sample: every value bit for bit (hash rows, per-ray counts and first crossings, the samples of the
    # stored rays)
    gold = np.load(REF_CUDA_GOLD)
    h = lambda k: got[k].cpu().numpy()
    assert np.array_equal(h("hash_out")[gold["hash_rows"]], gold["hash_out"])
    assert np.array_equal(h("counts"), gold["counts"]) and np.array_equal(h("first_oct_dis"), gold["first_oct_dis"])
    rays = gold["rays"]
    m = np.arange(S)[None, :] < gold["counts"][rays][:, None]
    for k in ("ts", "dists", "warp_pts", "world_pts", "anchors"):
        assert np.array_equal(h(k)[rays][m], gold[k]), k
    if not rh.cuda_available():
        return
    # live, beside the library: hash forward on the same table, points, primes -> bit-identical encodings
    dev = "cuda"
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    ref = rh.cuda_hash_forward(T(inp["feat"]), T(inp["prim"].astype(np.int32)), T(inp["bias"]), T(inp["pts"]),
                               T(inp["anchors"]))
    out = got["hash_out"]
    print("hash forward bit-equal fraction vs nvcc-built reference:", float((out == ref).float().mean()))
    assert torch.equal(out, ref)
    # sampler: leaf ranges, counts and anchors identical; positions reported
    r = rh.cuda_get_samples(T(inp["o"]), T(inp["d"]), T(inp["noise"]), s.tree_nodes_gpu_, s.pers_trans_gpu_,
                            T(orc.search_order()))
    cnt, ts, dists, warp, world, anc = (got[k] for k in ("counts", "ts", "dists", "warp_pts", "world_pts", "anchors"))
    same = (cnt == r["counts"])
    print("sampler: rays with identical sample counts:", float(same.float().mean()), "of", cnt.shape[0])
    m = (torch.arange(S, device=dev)[None, :] < cnt[:, None]) & same[:, None]
    for name, a, b in (("t", ts, r["ts"]), ("dist", dists, r["dists"]), ("warp", warp, r["warp_pts"]),
                       ("world", world, r["world_pts"])):
        mm = m if a.dim() == 2 else m[..., None].expand_as(a)
        print(f"  {name}: bit-equal fraction {float((a[mm] == b[mm]).float().mean()):.6f}, "
              f"max abs diff {float((a[mm] - b[mm]).abs().max()):.3e}")
    assert bool(same.all())
    assert torch.equal(anc[m], r["anchors"][m])
    assert torch.equal(got["first_oct_dis"], r["first_oct_dis"])
    for a, b in ((ts, r["ts"]), (dists, r["dists"]), (warp, r["warp_pts"]), (world, r["world_pts"])):
        mm = m if a.dim() == 2 else m[..., None].expand_as(a)
        assert torch.equal(a[mm], b[mm])
