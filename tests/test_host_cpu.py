"""CPU-side checks (run with -m "not gpu"): the C-ABI library builds/loads and exports exactly what
include/uem_b200.h declares, the host layer refuses CPU tensors (no fallback), the sharding / packing
helpers are right, and the world_size-2 exchange works over gloo."""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    text = open(os.path.join(ROOT, "include", "uem_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    out = {}
    for m in re.finditer(r"UEM_API\s+([\w\s\*]+?)\s*\b(uem_\w+)\s*\(([^;]*?)\)\s*;", text, flags=re.S):
        args = m.group(3).strip()
        n = 0 if args in ("", "void") else len(args.split(","))
        out[m.group(2)] = n
    return out


@pytest.fixture(scope="module")
def built_lib():
    from uemda_b200 import build
    return build.build()


def test_library_exports_every_declared_symbol(built_lib):
    decl = _header_functions()
    assert len(decl) >= 30
    nm = subprocess.run(["nm", "-D", "--defined-only", built_lib], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (uem_\w+)", nm))
    assert set(decl) == exported, (set(decl) ^ exported)


def test_ctypes_signatures_match_header(built_lib):
    from uemda_b200 import _lib
    decl = _header_functions()
    assert set(_lib.SIGNATURES) == set(decl), set(_lib.SIGNATURES) ^ set(decl)
    for name, (_, args) in _lib.SIGNATURES.items():
        assert len(args) == decl[name], (name, len(args), decl[name])
    lib = _lib.load()  # loading needs no GPU
    assert lib.uem_version() == 1
    # pure host helpers can be called without a device
    assert lib.uem_class_stats_bytes(8, 6) >= 8 * 8 * 4
    assert lib.uem_class_max_ws_bytes(8, 6, 512 * 512) > 0
    assert lib.uem_mine_ws_bytes(8, 6, 512, 512, 32, 32, 2048, 1025) > 8 * 6 * 32 * 32 * 4


def test_options_and_exchange_geometry_are_host_only_removed_options_refused(built_lib):
    """uem_set_option and the exchange-region geometry are pure host code: callable without a device; unknown options
    (among them the removed refine_form, refine_slot_skew and pdl_pearson) and out-of-range worlds are refused with an
    error, not ignored."""
    from uemda_b200 import _lib
    lib = _lib.load()
    defaults = {"l2_stream": 1, "l2_last_use": 1, "l2_region": 1, "l2_keep": 0, "refine_ctas_per_sm": 0,
                "region_ctas_per_sm": 0, "proto_ctas_per_sm": 0}
    for name, v in defaults.items():
        assert lib.uem_set_option(name.encode(), v) == 0, name
    for name in ("no_such_option", "refine_form", "refine_slot_skew", "pdl_pearson"):
        assert lib.uem_set_option(name.encode(), 1) != 0, name
        assert name.encode() in lib.uem_last_error()
    one = lib.uem_xchg_region_bytes(1, 3, 6, 2048)
    eight = lib.uem_xchg_region_bytes(8, 3, 6, 2048)
    assert one > 3 * 6 * 2048 * 8 and (eight - 2048) == 8 * (one - 2048)   # header + depth x world x slot
    assert lib.uem_xchg_region_bytes(17, 3, 6, 2048) < 0 and lib.uem_xchg_region_bytes(2, 5, 6, 2048) < 0


def test_uvem_loss_backward_requires_workspace(built_lib):
    """uem_uvem_loss_backward_f32 has one form, which needs its scratch: ws = NULL is refused with an error before any
    pointer is touched (so this runs without a device)."""
    import ctypes
    from uemda_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(256)   # never dereferenced
    assert lib.uem_uvem_loss_backward_f32(p, None, 2, 6, 8, 8, 64, 64, p, p, p, p, None, None, None) != 0
    assert b"ws" in lib.uem_last_error()


def test_sass_is_sm100a(built_lib):
    out = subprocess.run(["cuobjdump", "-lelf", built_lib], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out[:400]


def test_no_cpu_fallback():
    from uemda_b200 import _lib, ops
    from uemda_b200.gast.pseudo_generation import pseudo_selection
    from uemda_b200.scatter import scatter
    x = torch.rand(1, 3, 8, 8)
    with pytest.raises(_lib.UemLibraryError):
        ops.class_max(x)
    with pytest.raises(_lib.UemLibraryError):
        pseudo_selection(x, return_type="tensor")
    with pytest.raises(_lib.UemLibraryError):
        scatter(torch.rand(1, 16, 3), torch.zeros(1, 16, 1, dtype=torch.long), dim=1, reduce="max")
    if not torch.cuda.is_available():
        from uemda_b200.gast.alignment import Aligner
        with pytest.raises(RuntimeError):
            Aligner(None, 8, 3)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "uemda_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.replace("uem_oracle", "oracle") or "import oracle" not in text, f
                assert not re.search(r"^\s*(from|import)\s+oracle", text, flags=re.M), f


def test_f32_rounding_helper():
    from uemda_b200.ops import _uvem_coefs, f32
    assert f32(0.8) == float(torch.tensor(0.8, dtype=torch.float32))
    m, t, ig, cl, cr = _uvem_coefs(0.2, 0.7, 4.0)
    assert cl == float(torch.tensor(-1 / (0.2 ** 2), dtype=torch.float32))
    assert cr == float(torch.tensor(-1 / ((0.7 - 0.2) ** 2), dtype=torch.float32))


def test_shard_range_covers_everything():
    from uemda_b200.mining import shard_range
    for n in (0, 1, 7, 8, 2016, 2017):
        for ws in (1, 2, 3, 4, 8):
            spans = [shard_range(n, r, ws) for r in range(ws)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(ws - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_pack_unpack_roundtrip():
    from uemda_b200.mining import pack_stats, unpack_stats
    c, k = 6, 32
    sums = torch.randn(c, k)
    counts = torch.randint(0, 1 << 40, (c,))
    hist = torch.randint(0, 1 << 40, (c + 1,))
    s, n, h = unpack_stats(pack_stats(sums, counts, hist), c, k, True)
    assert torch.equal(s, sums) and torch.equal(n, counts) and torch.equal(h, hist)


def test_synth_is_deterministic():
    from uemda_b200.synth import WORKLOADS, make_inputs
    a = make_inputs(WORKLOADS["tiny"], seed=5)
    b = make_inputs(WORKLOADS["tiny"], seed=5)
    for key in ("soft", "feat", "sup", "label_s", "pred1"):
        assert torch.equal(a[key], b[key])
    sup = a["sup"]
    assert sup.dtype == torch.int64 and int(sup.max()) == a["ignore_id"]
    frac = float((sup == a["ignore_id"]).float().mean())
    assert 0.2 < frac < 0.95  # the 7x7 edge shrink marks a large share of pixels as 'ignored'


def test_bench_dump_is_bounded_and_repeatable(tmp_path):
    """bench.py --dump-outputs: one float32 .npy per output, an output larger than its share written as its own values at
    sorted, unique, seeded flat indices (the same on every run), and at most DUMP_BYTES in all."""
    import numpy as np
    import bench
    g = torch.Generator().manual_seed(1)
    arrays = {"refined": torch.rand(8, 6, 512, 512, generator=g), "hard": torch.randint(-1, 6, (8, 512, 512), generator=g),
              "prototypes": torch.randn(6, 2048, generator=g)}
    info = bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    total = 0
    for name in arrays:
        x, y = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert x.dtype == np.float32 and np.array_equal(x, y), name
        total += x.nbytes
    assert total <= bench.DUMP_BYTES
    assert info["refined"] == [arrays["refined"].numel(), np.load(tmp_path / "a" / "refined.npy").size]
    assert info["refined"][1] < info["refined"][0]
    idx = bench.dump_sample_index(arrays["refined"].numel(), bench.DUMP_BYTES // (4 * len(arrays)))
    assert idx.numel() == info["refined"][1] and bool((idx[1:] > idx[:-1]).all())   # sorted, no repeats
    assert np.array_equal(np.load(tmp_path / "a" / "refined.npy"), arrays["refined"].reshape(-1)[idx].numpy())
    assert np.array_equal(np.load(tmp_path / "a" / "hard.npy"), arrays["hard"].numpy().astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "a" / "prototypes.npy"), arrays["prototypes"].numpy())


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["UEM_ROOT"])
from uemda_b200.mining import pack_stats, unpack_stats, shard_range, pack_local, fold_gathered
from oracle import uem_oracle as O
from uemda_b200.synth import Workload, make_inputs
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
wl = Workload("t", 4, 5, 32, 32, 24, 8, 9)
inp = make_inputs(wl, seed=3)
lo, hi = shard_range(wl.b, rank, world)
down = O.downscale_label(inp["label_s"], wl.scale, wl.c)
# rank-local partial statistics, exchanged exactly as ShardedMiner does (sum + max)
s, n = O.class_feature_sums(inp["feat_s"][lo:hi], down[lo:hi], wl.c)
hist, valid = O.class_histogram(down[lo:hi], wl.c)
buf = pack_stats(s, n.reshape(-1).long(), torch.cat([hist, valid.reshape(1).long()]))
dist.all_reduce(buf, op=dist.ReduceOp.SUM)
mx = inp["sup"][lo:hi].max().reshape(1)
dist.all_reduce(mx, op=dist.ReduceOp.MAX)
S, N, Hh = unpack_stats(buf, wl.c, wl.k, True)
s_all, n_all = O.class_feature_sums(inp["feat_s"], down, wl.c)
h_all, v_all = O.class_histogram(down, wl.c)
assert torch.allclose(S, s_all, rtol=1e-5, atol=1e-5)
assert torch.equal(N, n_all.reshape(-1).long())
assert torch.equal(Hh[:-1], h_all) and int(Hh[-1]) == int(v_all)
# ClassBalance over a sharded batch (balance.py:45-52 is batch-global): the frequency EMA fed by the all-reduced
# histogram equals the un-sharded one; fed by the rank-local histogram it does not
freq0 = torch.ones(wl.c) / wl.c
want_freq, want_w = O.class_balance_step(freq0, down, wl.c)[:2]
red = torch.cat([hist, valid.reshape(1).long()]).clone()
dist.all_reduce(red, op=dist.ReduceOp.SUM)
got_freq = (1.0 - 0.99) * (red[:-1].float() / (red[-1].float() + 1e-7)) + 0.99 * freq0
assert torch.equal(got_freq, want_freq), (got_freq, want_freq)
assert int(mx) == int(inp["sup"].max())
# the three-phase form: one all_gather of [sums | counts | max id], folded in rank order on every rank
packed = pack_local(s, n.reshape(-1).long(), inp["sup"][lo:hi].max().reshape(1))
gathered = torch.empty(world, packed.numel(), dtype=torch.float64)
dist.all_gather_into_tensor(gathered.reshape(-1), packed)
S2, N2, M2 = fold_gathered(gathered, wl.c, wl.k)
assert torch.allclose(S2, s_all, rtol=1e-5, atol=1e-5) and torch.equal(N2, n_all.reshape(-1).long())
assert int(M2) == int(inp["sup"].max())
# sharded refine with the GLOBAL ignored id == un-sharded refine (alignment.py:241 is batch-global)
full = O.label_refine(inp["sup"], inp["feat"], [inp["pred1"], inp["pred2"]], inp["soft"], inp["prototypes"])
sup_l = inp["sup"][lo:hi].clone()
# emulate the global max inside the oracle by appending one sentinel pixel-free check: ids equal to mx are ignored
part = O.label_refine(torch.cat([sup_l, inp["sup"]]), torch.cat([inp["feat"][lo:hi], inp["feat"]]),
                      [torch.cat([inp["pred1"][lo:hi], inp["pred1"]]), torch.cat([inp["pred2"][lo:hi], inp["pred2"]])],
                      torch.cat([inp["soft"][lo:hi], inp["soft"]]), inp["prototypes"])[: hi - lo]
assert torch.equal(part, full[lo:hi])
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_world_size_2_gloo_exchange(tmp_path):
    """The N>1 host logic on CPU: shard -> local stats -> packed all_reduce(SUM) + all_reduce(MAX)."""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    env = dict(os.environ, UEM_ROOT=ROOT, MASTER_ADDR="127.0.0.1", MASTER_PORT="29613", WORLD_SIZE="2",
               OMP_NUM_THREADS="2")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
