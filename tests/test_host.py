"""CPU tests of the host-side logic: init parity with the reference, state_dict layout, synthetic batches,
the C-ABI library (loads, exports every declared symbol) and the loud failure without a GPU."""
import ctypes
import os
import re

import pytest
import torch

from conftest import ROOT, load_golden, relerr
from dostransformer_b200 import _lib
from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer
from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon
from dostransformer_b200.synthetic import make_edos_batch, make_large_cell_batch, make_phonon_batch


def _summ_ok(model, fx):
    sd = model.state_dict()
    assert [(k, tuple(v.shape), str(v.dtype)) for k, v in sd.items()] == fx["state_keys"]
    for k, s in fx["weights"].items():
        v = sd[k]
        assert abs(v.double().norm().item() - s["norm"]) <= 1e-12 * max(1.0, s["norm"]), k
        assert torch.equal(v.flatten()[:8], s["head"]), k


def test_edos_init_and_state_dict_match_reference():
    fx = load_golden("edos_h256.pt")
    torch.manual_seed(fx["init_seed"])
    m = DOSTransformer(3, 2, 200, 41, 2, 256, torch.device("cpu"), 0.0)
    _summ_ok(m, fx)
    assert sum(p.numel() for p in m.parameters()) == 9_428_109


def test_phonon_init_and_state_dict_match_reference():
    fx = load_golden("phonon_h256.pt")
    torch.set_default_dtype(torch.float64)
    torch.manual_seed(fx["init_seed"])
    m = DOSTransformer_phonon(3, 2, 118, 4, 256, torch.device("cpu"), 0.0)
    _summ_ok(m, fx)
    assert m.fc.weight.dtype == torch.float64


def test_phonon_ctor_accepts_the_launchers_argument_order():
    # main_phDOS.py:68 passes (layers, transformer, 118, 4, hidden, out_dim, device)
    m = DOSTransformer_phonon(1, 1, 118, 4, 32, 51, torch.device("cpu"))
    assert m.n_energies == 51 and m.attn_drop == 0.0 and m.embeddings.weight.shape == (51, 32)
    m2 = DOSTransformer_phonon(1, 1, 118, 4, 32, torch.device("cpu"), 0.1)
    assert m2.attn_drop == 0.1


def test_small_fixture_state_dict_loads():
    fx = load_golden("edos_small.pt")
    m = DOSTransformer(*fx["ctor_args"])
    m.load_state_dict(fx["state_dict"], strict=True)


def test_no_cpu_fallback():
    m = DOSTransformer(1, 1, 200, 41, 2, 32, "cpu", 0.0)
    g = make_edos_batch(2, seed=1, mean_atoms=4.0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(g)


def test_dropin_aliases():
    import dostransformer_b200
    dostransformer_b200.install_dropin()
    from embedder_eDOS.DOSTransformer import DOSTransformer as A
    from embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon as Bc
    from layers import TransformerEncoder
    assert A is DOSTransformer and Bc is DOSTransformer_phonon and TransformerEncoder is not None
    import sys
    for k in ("embedder_eDOS", "embedder_phDOS", "layers", "embedder_eDOS.DOSTransformer",
              "embedder_phDOS.DOSTransformer_phonon"):
        sys.modules.pop(k, None)


def test_synthetic_edos_layout():
    g = make_edos_batch(16, seed=3)
    B = 16
    n = torch.bincount(g.batch, minlength=B)
    assert g.x.shape[1] == 200 and g.edge_attr.shape[1] == 41 and g.glob.shape == (2 * B,)
    assert g.y_ft.shape == (B * 201,) and len(g.mp_id) == B and g.system.max() < 7
    assert torch.all(g.batch[1:] >= g.batch[:-1])
    last = n.cumsum(0) - 1
    assert torch.all(g.x[last] == 0)                      # the zero "prompt" node of every crystal
    row, col = g.edge_index
    assert g.edge_index.shape[1] == 12 * int((n - 1).sum())
    assert torch.all(g.batch[row] == g.batch[col])
    assert not torch.isin(row, last).any() and not torch.isin(col, last).any()
    assert (g.y_ft < 0).any() and g.y_ft.max() <= 1.0 + 1e-6
    g2 = make_edos_batch(16, seed=3)
    assert torch.equal(g.x, g2.x) and torch.equal(g.edge_index, g2.edge_index)


def test_synthetic_phonon_and_large_cell():
    g = make_phonon_batch(3, seed=4)
    assert g.x.dtype == torch.float64 and g.x.shape[1] == 118 and g.phdos.shape == (3, 51)
    row, col = g.edge_index
    assert g.edge_vec.shape == (row.numel(), 3)
    self_edges = row == col
    assert torch.all(g.edge_vec[::24] == 0) and self_edges[::24].all()
    assert "edge_index" in g and g["edge_vec"] is g.edge_vec
    big = make_large_cell_batch(2, seed=5)
    n = torch.bincount(big.batch)
    assert n.min() >= 201 and big.edge_index.shape[1] == 24 * int((n - 1).sum())


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "dost.h")).read()
    declared = set(re.findall(r"\b(dost_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    lib = _lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/dost.h but not exported"
    assert declared == set(_lib.EXPORTED_SYMBOLS)
    assert lib.dost_abi_version() == _lib.ABI_VERSION == 15
    # argument validation works without a GPU (no launch happens)
    assert lib.dost_gemm(None, None, 0, None) == -1
    assert b"null descriptor" in lib.dost_last_error()
    assert isinstance(lib.dost_csr_workspace_bytes(10, 4), int)


def test_ops_raise_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.lib()


def test_fused_adamw_interface_mirrors_torch():
    """Constructor defaults, param_groups and the state_dict layout of torch.optim.AdamW (no device work)."""
    from dostransformer_b200.optim import AdamW
    ps = [torch.nn.Parameter(torch.zeros(3, 2)), torch.nn.Parameter(torch.zeros(5))]
    opt = AdamW(ps, lr=1e-4, weight_decay=1e-2)
    ref = torch.optim.AdamW(ps, lr=1e-4, weight_decay=1e-2)
    for k in ("lr", "betas", "eps", "weight_decay"):
        assert opt.param_groups[0][k] == ref.param_groups[0][k]
    opt.step()                                  # nothing has a gradient: a no-op, like torch
    sd = opt.state_dict()
    assert sd["state"] == {} and sd["param_groups"][0]["params"] == [0, 1]
    opt.zero_grad()
    with pytest.raises(ValueError):
        AdamW([])


def test_oracle_collate_inverts_split_batch():
    """Integer / byte work of the batch assembly, host side: oracle.collate(split_batch(b)) == b bit for bit, and the
    packed store's metadata (table kinds, counts) on a CPU-resident store."""
    from dostransformer_b200.collate import PackedCrystals, split_batch
    from oracle.dost_oracle import collate
    for b in (make_edos_batch(9, seed=21), make_phonon_batch(6, seed=22)):
        graphs = split_batch(b)
        c = collate([{k: g[k] for k in g.keys()} for g in graphs])
        for k in b.keys():
            if k == "max_num_nodes":
                continue
            if torch.is_tensor(b[k]):
                assert c[k].dtype == b[k].dtype and torch.equal(c[k], b[k]), k
            else:
                assert c[k] == b[k], k
        n = torch.bincount(b.batch)
        assert torch.equal(c["ptr"], torch.cat([n.new_zeros(1), n.cumsum(0)]))
        pk = PackedCrystals.from_graphs(graphs, device="cpu")
        assert len(pk) == b.num_graphs and pk.kinds["x"] == "node" and pk.kinds["system"] == "crystal"
        assert pk.kinds["edge_attr" if "edge_attr" in b else "edge_vec"] == "edge"
        assert int(pk.node_count.sum()) == b.x.shape[0] and int(pk.edge_count.sum()) == b.edge_index.shape[1]
        assert int(pk.edge_index.min()) == 0 and int(pk.edge_index.max()) == int(n.max()) - 1 - ("glob" in b)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            if torch.cuda.is_available():
                raise RuntimeError("no CPU fallback")      # GPU box: the CPU-resident store is rejected below instead
            pk.collate([0, 1])


def test_header_is_plain_c_and_struct_layouts_match_ctypes(tmp_path):
    """include/dost.h must compile as C (it is the FFI contract) and every descriptor struct must have the layout the
    ctypes mirror in _lib.py assumes: size and the offset of every field, taken from gcc."""
    import ctypes
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    pairs = {"dost_seg_t": _lib.Seg, "dost_gemm_t": _lib.Gemm, "dost_planes_t": _lib.PlanesC, "dost_gemm_bf16_t": _lib.GemmBf16}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{os.path.join(ROOT, "include", "dost.h")}"',
             'int main(void) {']
    for cname, cls in pairs.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(src)], check=True, capture_output=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    got = {(a, b): int(c) for a, b, c in (ln.split() for ln in out.strip().splitlines())}
    for cname, cls in pairs.items():
        assert got[(cname, "size")] == ctypes.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert got[(cname, fname)] == getattr(cls, fname).offset, (cname, fname)
    # and nothing in the C struct is missing from the mirror: equal size + equal last-field offset covers trailing fields


def test_sweep_plan_covers_every_crystal_once():
    import numpy as np
    from dostransformer_b200.evaluate import sweep_plan
    rng = np.random.default_rng(0)
    counts = rng.integers(2, 60, size=1000)
    for world in (1, 3, 8):
        plan = sweep_plan(counts, 64, world)
        assert len(plan) == world
        allids = np.concatenate([b.numpy() for r in plan for b in r])
        assert sorted(allids.tolist()) == list(range(1000))
        # contiguous by length: inside a batch the atom counts span a narrow range, batches are balanced across ranks
        for r in plan:
            for b in r:
                c = counts[b.numpy()]
                assert c.max() - c.min() <= 6
        assert max(len(r) for r in plan) - min(len(r) for r in plan) <= 1


def test_bench_reference_arm_contract_and_product_arm_needs_gpu():
    """bench.py --impl reference prints one JSON line with the contract's keys (CPU oracle port, bounded sample); the
    product arm refuses to run without a CUDA device instead of falling back to the CPU."""
    import json
    import subprocess
    import sys
    env = dict(os.environ, OMP_NUM_THREADS="4")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-sample", "4"], capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "crystals/s" and d["higher_is_better"] is True and d["value"] > 0
    # kind "reference" = the reference's own modules (/root/reference here, oracle/_ref on the GPU box); "port" = the oracle
    from oracle import reference_loader
    want_kind = "reference" if reference_loader.available() else "port"
    assert d["vs_baseline"] is None and d["cpu_baseline"]["kind"] == want_kind and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in d["config"]
    if not torch.cuda.is_available():
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                           capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_bench_dump_outputs_dtypes_and_budget(tmp_path):
    """bench.py --dump-outputs: float64 arrays are written as float64, all others as float32; past the byte budget every
    array keeps the same seeded sample of its elements, run after run, and a scalar is never cut away."""
    import numpy as np
    import bench
    arrays = {"loss": torch.tensor(1.5), "grad.w": torch.arange(1000.0).view(10, 100),
              "grad.h": torch.arange(50, dtype=torch.float16), "grad.d": torch.arange(300, dtype=torch.float64)}
    bench.dump_outputs(str(tmp_path / "full"), arrays)
    for k, v in arrays.items():
        got = np.load(tmp_path / "full" / f"{k}.npy")
        assert got.dtype == (np.float64 if v.dtype == torch.float64 else np.float32) and got.shape == tuple(v.shape), k
        assert np.array_equal(got, v.double().numpy()), k
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, budget=2000)
    total = 0
    for k, v in arrays.items():
        a, b = np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy")
        assert np.array_equal(a, b) and a.ndim == 1 and 1 <= a.size < max(2, v.numel()), k
        assert np.isin(a, v.double().numpy()).all() and np.unique(a).size == a.size, k      # distinct elements of v
        total += a.nbytes
    assert total <= 2000 + 8


def test_bucket_padding_is_a_semantic_no_op_for_the_real_crystals():
    """synthetic.pad_edos_batch (the shape bucketing behind graphed.GraphedStep): on the CPU oracle, the padded batch's
    outputs, loss over the first n_valid crystals and gradients equal those of the unpadded batch (the padding length
    Nmax, which sets every crystal's phantom-key count, is unchanged because no dummy is larger than a real crystal)."""
    from dostransformer_b200.graphed import batch_signature
    from dostransformer_b200.synthetic import pad_edos_batch
    from oracle import dost_oracle as O
    torch.manual_seed(0)
    sd = O.state_dict_of(DOSTransformer(2, 1, 200, 41, 2, 32, "cpu", 0.0))
    g = make_edos_batch(5, seed=8, mean_atoms=6.0)
    p = pad_edos_batch(g, node_bucket=32, dummies=2)
    B = 5
    assert p.n_valid == B and p.x.shape[0] % 32 == 0 and p.edge_index.shape[1] == 12 * (p.x.shape[0] - p.system.numel())
    n = torch.bincount(p.batch)
    assert n.min() >= 2 and int(n[B:].max()) <= int(n[:B].max())
    leaf = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    dg, x, ds = O.edos_forward(leaf, g, training=True)
    loss = O.edos_loss(dg, ds, g.y_ft)
    loss.backward()
    leaf_p = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    dgp, xp, dsp = O.edos_forward(leaf_p, p, training=True)
    loss_p = O.edos_loss(dgp[:B], dsp[:B], p.y_ft.reshape(-1, 201)[:B].reshape(-1))
    loss_p.backward()
    assert relerr(dgp[:B], dg) < 1e-5 and relerr(dsp[:B], ds) < 1e-5 and relerr(xp[:x.shape[0]], x) < 1e-5
    assert abs(loss_p.item() - loss.item()) < 1e-6 * abs(loss.item())
    for k, v in leaf.items():
        if torch.is_tensor(v) and v.requires_grad and v.grad is not None:
            assert leaf_p[k].grad is not None
            err = ((leaf_p[k].grad - v.grad).norm() / v.grad.norm().clamp_min(1e-30)).item()
            assert err < 5e-4, (k, err)
    # a handful of signatures for many batches
    sigs = {batch_signature(pad_edos_batch(make_edos_batch(64, seed=100 + s))) for s in range(12)}
    assert len(sigs) <= 6


def test_staged_reference_copy_is_byte_identical(tmp_path, monkeypatch):
    """oracle/build_ref.py stages the reference's model files for machines without the reference: the same bytes as the
    source, their SHA-256 in the manifest, and the staged copy still found once the source is gone.  A stand-in source
    tree takes the reference's place."""
    import hashlib
    import json
    from oracle import build_ref
    src, dst = tmp_path / "reference", tmp_path / "staged"
    for i, rel in enumerate(build_ref.FILES):
        (src / rel).parent.mkdir(parents=True, exist_ok=True)
        (src / rel).write_bytes(f"# {rel}\n".encode() + bytes(range(256)) * i)
    monkeypatch.setattr(build_ref, "SRC", str(src))
    monkeypatch.setattr(build_ref, "DST", str(dst))
    assert build_ref.build() == str(dst)
    man = json.load(open(dst / "MANIFEST.json"))
    assert set(man["sha256"]) == set(build_ref.FILES)
    for rel, sha in man["sha256"].items():
        data = (src / rel).read_bytes()
        assert (dst / rel).read_bytes() == data and hashlib.sha256(data).hexdigest() == sha, rel
    monkeypatch.setattr(build_ref, "SRC", str(tmp_path / "absent"))
    assert build_ref.build() == str(dst)


def test_kernel_path_gates_are_host_decisions(monkeypatch):
    """Which kernels a call takes is decided on the host from shapes, the precision context and the DOST_* switches: the
    fused attention (<= 256 keys, H in {64, 128, 192, 256}, a tensor-core precision), the 1-bit ReLU gates of the FFN (TMA-store
    epilogue: M >= 32, N % 32 == 0), the key-side buffer bound of the attention (the batch's own largest crystal, not the
    data-parallel padding length).  No device is touched."""
    from dostransformer_b200 import _lib as L
    from dostransformer_b200 import ops
    with ops.precision("bf16x3"):
        assert ops.fused_attention_ok(256, 201) and ops.fused_attention_ok(128, 1, 0.3) and ops.fused_attention_ok(64, 256)
        assert not ops.fused_attention_ok(256, 257) and not ops.fused_attention_ok(32, 40) and not ops.fused_attention_ok(320, 40)
        monkeypatch.setenv("DOST_NO_ATTN_FUSED", "1")
        L.reload_switches()
        assert not ops.fused_attention_ok(256, 201)
        monkeypatch.delenv("DOST_NO_ATTN_FUSED")
        L.reload_switches()
    with ops.precision("fp32"):
        assert not ops.fused_attention_ok(256, 201)
    assert ops.gate_bits_ok(205824, 1024) and not ops.gate_bits_ok(16, 1024) and not ops.gate_bits_ok(4096, 1000)
    monkeypatch.setenv("DOST_GEMM_TMA_EPI", "0")
    assert not ops.gate_bits_ok(205824, 1024)
    monkeypatch.delenv("DOST_GEMM_TMA_EPI")
    t = torch.zeros(1, dtype=torch.int32)
    csr = ops.CSR(t, None, t, 0)
    g = ops.CrystalGraph(0, 0, 0, t, t, t, t, csr, csr, csr, csr, t, 201, 111)
    assert g.nkeys_host == 112                       # own largest crystal (111) + the phantom column, not the global 201
    assert ops.CrystalGraph(0, 0, 0, t, t, t, t, csr, csr, csr, csr, t, 201, None).nkeys_host == 202
    assert ops.CrystalGraph(0, 0, 0, t, t, t, t, csr, csr, csr, csr, t, None, None).nkeys_host is None


def test_index_cache_keeps_outgrown_tensors_alive():
    """ops._arange_i32 serves views of one cached index tensor per device.  When a longer one is needed the old tensor is
    retired, not freed: launches recorded in a CUDA graph keep reading it (the GPU-side regression is
    tests/test_gpu_graphed.py::test_cached_index_tensors_outlive_captured_graphs)."""
    from dostransformer_b200 import ops
    dev = torch.device("cpu")
    a = ops._arange_i32(10, dev)
    base = ops._ARANGE_CACHE[(str(dev),)]
    assert a.data_ptr() == base.data_ptr() and torch.equal(a, torch.arange(10, dtype=torch.int32))
    n_retired = len(ops._ARANGE_RETIRED)
    b = ops._arange_i32(base.numel() + 5, dev)
    assert b.numel() == base.numel() + 5 and int(b[-1]) == base.numel() + 4
    assert ops._ARANGE_CACHE[(str(dev),)] is not base
    assert len(ops._ARANGE_RETIRED) == n_retired + 1 and ops._ARANGE_RETIRED[-1] is base
    assert torch.equal(a, torch.arange(10, dtype=torch.int32))          # the earlier view still reads its own storage
    c = ops._arange_i32(7, dev)                                          # smaller requests re-use the new tensor
    assert c.data_ptr() == ops._ARANGE_CACHE[(str(dev),)].data_ptr() and len(ops._ARANGE_RETIRED) == n_retired + 1


def test_reference_arm_under_torchrun_prints_one_line():
    """The driver launches both arms the same way.  Under torch.distributed.run with 2 ranks the reference arm runs on
    rank 0 alone and prints ONE JSON line; rank 1 exits 0 without work."""
    import json
    import subprocess
    import sys
    env = dict(os.environ, OMP_NUM_THREADS="4")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29731", os.path.join(ROOT, "bench.py"), "--impl", "reference",
                        "--gpus", "2", "--steps", "1", "--warmup", "0", "--cpu-sample", "4"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0 and d["e2e"]["value"] == d["value"]
