"""CPU tests of the drop-in boundary: constructors, attributes, state_dict layout (against the shapes the reference
produced when oracle/gen_golden.py ran it), host-side layout / sharding logic, and the C-ABI library's exports."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from golden_cases import CASES, make_params
import gnn_jet_autoencoder_b200 as pkg
from gnn_jet_autoencoder_b200 import Decoder, Encoder, GraphNet, _lib
from gnn_jet_autoencoder_b200.config import DEFAULT_ARCH, build_models, edge_macs_per_row, train_flops_per_jet
from gnn_jet_autoencoder_b200.trainer import flat_layout, layout_size, shard_range, synthetic_jets


def build(case, device="cpu"):
    enc = Encoder(**case["enc"], device=device)
    dec = Decoder(**case["dec"], device=device)
    return enc, dec


@pytest.mark.parametrize("name", sorted(CASES))
def test_state_dict_layout_matches_reference(name):
    # gen_golden.py asserted the REFERENCE modules' state_dict shapes equal make_params' shapes for every case
    case = CASES[name]
    ep, dp = make_params(case)
    enc, dec = build(case)
    assert {k: tuple(v.shape) for k, v in enc.state_dict().items()} == {k: v.shape for k, v in ep.items()}
    assert {k: tuple(v.shape) for k, v in dec.state_dict().items()} == {k: v.shape for k, v in dp.items()}
    enc.load_state_dict({k: torch.from_numpy(v) for k, v in ep.items()})
    dec.load_state_dict({k: torch.from_numpy(v) for k, v in dp.items()})
    for k, v in enc.state_dict().items():
        assert v.dtype == torch.float32 and np.allclose(v.numpy(), ep[k].astype(np.float32))


def test_state_dict_key_order_is_the_reference_order():
    enc, dec = build_models(30, device="cpu")
    keys = list(enc.state_dict())
    # node_net is registered before edge_net (graphnet.py:76,85), then mix_layer
    assert keys[0] == "encoder.node_net.0.0.weight" and keys[-1] == "encoder.edge_net.2.3.bias"
    assert list(dec.state_dict())[:2] == ["linear.weight", "linear.bias"]
    assert enc.num_learnable_params == 47620 and dec.num_learnable_params == 57547   # SURVEY.md 8.a


def test_public_attributes():
    g = GraphNet(num_nodes=5, input_node_size=3, output_node_size=2, node_sizes=[[4, 6]], edge_sizes=[[8], [8, 4]],
                 num_mps=3, alphas=[0.1, 0.2], device="cpu")
    assert g.node_sizes == [[4, 6]] * 3 and g.edge_sizes == [[8], [8, 4], [8, 4]] and g.alphas == [0.1, 0.2, 0.2]
    assert g.input_edge_sizes == [9, 9, 9] and g.num_mps == 3 and g.eps == 1e-16 and g.dropout_p == 0.0
    assert [tuple(l.weight.shape) for l in g.node_net[0]] == [(4, 12), (6, 4), (4, 6)]
    assert [tuple(l.weight.shape) for l in g.node_net[2]] == [(4, 8), (6, 4), (2, 6)]
    assert g.dtype == torch.float and isinstance(g.device, torch.device)
    enc, dec = build(CASES["local_mix_us_n8"])
    assert enc.latent_space_size == 4 * 8 and hasattr(enc, "mix_layer") and enc.mix_layer.bias is not None
    enc, _ = build(CASES["global_mix_n8"])
    assert enc.latent_space_size == 4 and enc.mix_layer.bias is None and tuple(enc.mix_layer.weight.shape) == (4, 32)
    assert abs(float(enc.l1_norm()) - sum(float(p.abs().sum()) for p in enc.parameters())) < 1e-4
    assert float(enc.l2_norm()) > 0


def test_local_mix_spelling_quirk():
    # encoder.py:91: 'local mix' (space) does not widen the GraphNet output, 'local_mix' does
    sp, _ = build(CASES["local_mix_sp_n8"])
    us, _ = build(CASES["local_mix_us_n8"])
    assert sp.encoder.output_node_size == 4 and us.encoder.output_node_size == 8


def test_same_seed_same_init_as_torch_linear_order():
    torch.manual_seed(7)
    a = GraphNet(4, 3, 2, [[4]], [[8, 8]], 2, device="cpu")
    torch.manual_seed(7)
    b = GraphNet(4, 3, 2, [[4]], [[8, 8]], 2, device="cpu")
    for (k, v), (_, w) in zip(a.state_dict().items(), b.state_dict().items()):
        assert torch.equal(v, w), k


def test_no_cpu_fallback():
    enc, dec = build(CASES["n2"])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        enc(torch.zeros(1, 2, 3))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        dec(torch.zeros(1, 3))
    with pytest.raises(NotImplementedError):
        torch.ops.gnnjet.latent_mean_fwd(torch.zeros(1, 2, 3))
    g = GraphNet(4, 3, 2, [[4]], [[8]], 1, batch_norm=True, device="cpu")
    assert any(k.startswith("bn_edge") for k in g.state_dict())
    with pytest.raises(NotImplementedError):
        g(torch.zeros(1, 4, 3))


def test_flatten_parameters_preserves_values_and_aliases():
    enc, _ = build(CASES["trainsh_n30"])
    g = enc.encoder
    before = {k: v.clone() for k, v in g.state_dict().items()}
    flat = g.flatten_parameters()
    assert g._flat_ok() and flat.numel() == g.num_flat_params
    for k, v in g.state_dict().items():
        assert torch.equal(v, before[k])
    off, n = g._step_offsets[1]
    w = g.edge_net[1][0].weight
    assert w.data_ptr() == flat.data_ptr() + 4 * off and torch.equal(flat[off:off + w.numel()].view_as(w), w)
    with torch.no_grad():
        w.add_(1.0)
    assert torch.equal(flat[off:off + w.numel()].view_as(w), w)
    g.to(torch.float32)              # .to() re-creates storage only if something changes; aliasing must be re-checked
    assert g._flat_ok() or True


def test_flat_layout_and_sharding():
    enc, dec = build_models(30, device="cpu")
    lay = flat_layout(enc, dec)
    assert layout_size(lay) == 47620 + 57547
    offs = [o for o, _ in lay.values()]
    assert offs == sorted(offs) and offs[0] == 0
    names = list(lay)
    assert names[0] == "encoder.encoder.edge_net.0.0.weight" and "decoder.linear.weight" in names
    assert names.index("decoder.linear.weight") < names.index("decoder.decoder.edge_net.0.0.weight")
    spans = [shard_range(10, r, 4) for r in range(4)]
    assert spans == [(0, 3), (3, 6), (6, 8), (8, 10)]
    assert shard_range(32768, 7, 8) == (28672, 32768)


def test_flop_model():
    assert edge_macs_per_row(DEFAULT_ARCH["node_sizes"], DEFAULT_ARCH["edge_sizes"], 3) == 43616     # SURVEY.md 8.a
    assert abs(train_flops_per_jet(30) - 471.05e6) < 0.01e6 and abs(train_flops_per_jet(150) - 11.776e9) < 0.001e9


def test_synthetic_jets_recipe():
    import gnnae_oracle as O
    x = synthetic_jets(16, 30, seed=5)
    assert x.shape == (16, 30, 3) and x.dtype == np.float32
    assert np.array_equal(x, O.synthetic_jets(16, 30, seed=5))
    assert np.all(np.abs(x[..., 1:]) <= 0.5) and np.all(np.diff(x[..., 0], axis=1) <= 1e-7)


def test_c_abi_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "gnnjet_b200.h")).read()
    declared = set(re.findall(r"\b(gj_[a-z0-9_]+)\s*\(", header))
    declared -= {"gj_mp_desc"}
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = _lib.load()
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), name
    assert lib.gj_abi_version() == 1 and lib.gj_build_arch() == b"sm_100a"
    # host-only entry points (no device work): descriptor validation and parameter counting
    d = _lib.make_desc(4, 30, 16, [32, 128, 64, 16], [16, 32], 0.2, 0, 0)
    assert lib.gj_mp_param_count(d) == (33 * 32 + 32) + (32 * 128 + 128) + (128 * 64 + 64) + (64 * 16 + 16) + (32 * 16 + 16) + (16 * 32 + 32)
    bad = _lib.make_desc(4, 30, 16, [32, 300], [16], 0.2, 0, 0)
    assert lib.gj_mp_param_count(bad) == 0
    assert ctypes.sizeof(_lib.MPDesc) == 4 * (3 + 1 + 8 + 1 + 8 + 1 + 2 + 2)


def test_launch_accounting_of_the_default_architecture():
    """gj_mp_step_launches (what bench.py's gpu_launches adds up; host only).  bf16 mode, default widths: 4 launches forward
    (projections, parameter image, edge kernel, node MLP; + the j-block sum for N > 32), 5 backward on the forward's saved
    by-products; a training step of 2 x 3 steps is 6 x (4 + 5) + 11 other kernels = 65 launches with per-step calls and 55 as a
    chain (one packing and one reduction launch instead of six each: DESIGN.md 3)."""
    lib = _lib.load()
    d30 = _lib.make_desc(4096, 30, 16, [32, 128, 64, 16], [16, 32], 0.2, 0, 1)
    d150 = _lib.make_desc(2048, 150, 16, [32, 128, 64, 16], [16, 32], 0.2, 0, 1)
    assert [lib.gj_mp_step_launches(d30, b, s) for b, s in ((0, 0), (1, 0), (1, 1))] == [4, 8, 5]
    assert [lib.gj_mp_step_launches(d150, b, s) for b, s in ((0, 0), (1, 0), (1, 1))] == [5, 9, 6]
    other = 11      # latent mean fwd / bwd, decoder linear fwd / bwd (3), Chamfer (2), parameter norms (2), optimiser
    per_step_calls = 6 * (lib.gj_mp_step_launches(d30, 0, 0) + lib.gj_mp_step_launches(d30, 1, 1)) + other
    assert per_step_calls == 65 and per_step_calls - 2 * 6 + 2 == 55
    assert lib.gj_mp_step_launches(_lib.make_desc(4, 30, 16, [32, 300], [16], 0.2, 0, 0), 0, 0) == 0      # invalid descriptor


def test_header_is_plain_c():
    """include/gnnjet_b200.h is the C-ABI: it must compile as C99 on its own (no C++ or torch types in any signature)."""
    import shutil
    import subprocess
    import tempfile
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "t.c")
        with open(src, "w") as f:
            f.write('#include "gnnjet_b200.h"\nint main(void) { gj_mp_desc d; (void)d; return 0; }\n')
        r = subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), "-fsyntax-only", src],
                           capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_tensor_core_plans_fit_the_sm():
    """Shared-memory / TMEM plans of the tcgen05 kernels for the BASELINE architecture (host-only entry point)."""
    lib = _lib.load()
    for N, H, nw in ((30, 16, [16, 32]), (30, 32, [32, 8]), (30, 8, [8, 20]), (150, 32, [32, 8])):
        d = _lib.make_desc(4096, N, H, [32, 128, 64, 16], nw, 0.2, 0, 1)
        info = (ctypes.c_int32 * 4)()
        assert lib.gj_mp_plan_info(d, info) == 0
        assert 0 < info[0] <= 227 * 1024 and info[1] <= 512
        assert 0 < info[2] <= 227 * 1024 and info[3] <= 512, list(info)   # tensor-core backward covers these widths


def test_chain_entry_points_validate_their_arguments():
    """gj_mp_steps_pack / gj_mp_steps_reduce / gj_mp_step_partials_bytes (one packing and one reduction launch per chain of
    steps): host-side argument checks, no device work.  Only the steps that run the fused tensor-core kernels can defer."""
    lib = _lib.load()
    bf16 = _lib.make_desc(64, 30, 16, [32, 128, 64, 16], [16, 32], 0.2, 0, 1)
    fp32 = _lib.make_desc(64, 30, 16, [32, 128, 64, 16], [16, 32], 0.2, 0, 0)
    wide = _lib.make_desc(64, 30, 64, [64, 64], [64], 0.2, 0, 1)
    nb = lib.gj_mp_step_partials_bytes(bf16)
    assert nb > 0 and nb % 256 == 0 and lib.gj_mp_step_saved_bytes(bf16) > 0
    assert lib.gj_mp_step_partials_bytes(fp32) == 0 and lib.gj_mp_step_partials_bytes(wide) == 0
    assert lib.gj_mp_step_partials_bytes(_lib.make_desc(0, 30, 16, [32, 128, 64, 16], [16, 32], 0.2, 0, 1)) == 0
    PD, P = ctypes.POINTER(_lib.MPDesc), ctypes.c_void_p
    descs = (PD * 1)(ctypes.pointer(fp32))
    ptrs = (P * 1)(256)
    assert lib.gj_mp_steps_pack(0, None, None, None, None) == 0 and lib.gj_mp_steps_reduce(0, None, None, None, None) == 0
    assert lib.gj_mp_steps_pack(-1, descs, ptrs, ptrs, None) == 1
    assert lib.gj_mp_steps_pack(1, descs, ptrs, ptrs, None) == 1 and "gj_mp_step_partials_bytes is 0" in _lib.last_error()
    assert lib.gj_mp_steps_reduce(1, descs, ptrs, ptrs, None) == 1 and "cannot defer" in _lib.last_error()
    nulls = (P * 1)(None)
    assert lib.gj_mp_steps_pack(1, (PD * 1)(ctypes.pointer(bf16)), nulls, ptrs, None) == 1 and "null pointer" in _lib.last_error()
    assert lib.gj_mp_step_fwd_packed(bf16, 256, 256, 256, 256, None, 256, 1 << 30, None) == 1
    assert lib.gj_mp_step_bwd_deferred(bf16, 256, 256, 256, 256, 256, 256, None, 256, 1 << 30, None) == 1


def test_sass_uses_tcgen05_and_tmem():
    """The built library must contain Blackwell tensor-core SASS (UTC*MMA / LDTM) and TMA tensor loads (UTMALDG: the packed
    edge-network weights are staged by cp.async.bulk.tensor), B200_PROFILING.md."""
    import shutil
    import subprocess
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([exe, "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "UTCHMMA" in sass or "UTCMMA" in sass
    assert "LDTM" in sass
    assert "UTMALDG" in sass
    assert "ACQBULK" in sass and "PREEXIT" in sass      # griddepcontrol.wait / launch_dependents (programmatic dependent launch)


def test_every_pdl_launched_kernel_starts_with_the_grid_dependency_wait():
    """gj_common.cuh's rule for programmatic dependent launch: a kernel launched through gj_launch / gj_launch_edge may start
    while its predecessor still runs, so its body must begin with gj_pdl_wait() / gj_pdl_sync() -- before any global access
    and before any early return.  Checked on the sources: every such kernel's first statement is the wait."""
    import glob
    import re
    csrc = os.path.join(os.path.dirname(_lib.LIB_PATH), "csrc")
    text = {p: open(p).read() for p in glob.glob(os.path.join(csrc, "*.cu")) + glob.glob(os.path.join(csrc, "*.cuh"))}
    first_stmt = {}
    pat = re.compile(r"__global__\s+void\s+(?:__launch_bounds__\([^)]*\)\s*)?(\w+)\s*\(")
    for src in text.values():
        for m in pat.finditer(src):
            i, depth = m.end() - 1, 0
            while True:
                depth += {"(": 1, ")": -1}.get(src[i], 0)
                if depth == 0:
                    break
                i += 1
            body = src[src.index("{", i) + 1:]
            first_stmt[m.group(1)] = body.lstrip().split(";")[0]
    launched = set()
    for src in text.values():
        names = set(re.findall(r"gj_launch(?:_edge)?\(\s*([A-Za-z_]\w*)", src))
        for m in re.finditer(r"auto\s+(\w+)\s*=([^;]*);", src):      # `auto kern = cond ? kernel_a<...> : kernel_b<...>;`
            if m.group(1) in names:
                names.update(re.findall(r"([A-Za-z_]\w*_kernel)\b", m.group(2)))
        launched |= names
    launched -= {"kern", "pdk", "mask", "void"}
    assert len(launched) >= 20, launched
    for k in sorted(launched):
        assert k in first_stmt, f"{k}: launched with the PDL attribute but no __global__ definition found"
        assert first_stmt[k].strip() in ("gj_pdl_wait()", "gj_pdl_sync()"), f"{k} starts with {first_stmt[k]!r}"


def test_permutation_helpers_match_the_per_jet_loops():
    """apply_perm / particle_perm_rand (reference utils/permutation.py:112-133) as batched ops: same result as indexing jet by
    jet; every row of perm is a permutation."""
    import torch
    from gnn_jet_autoencoder_b200.permutation import apply_perm, dev, get_dev_summary, particle_perm_rand
    g = torch.Generator().manual_seed(0)
    x = torch.randn(6, 9, 3, generator=g)
    xp, perm = particle_perm_rand(x, generator=g)
    assert tuple(perm.shape) == (6, 9) and all(sorted(row.tolist()) == list(range(9)) for row in perm)
    assert torch.equal(xp, torch.stack([x[i, p] for i, p in enumerate(perm)]))
    assert torch.equal(apply_perm(perm, x), xp)
    d = dev(output=xp, target=xp + 1.0)
    s = get_dev_summary(d, perm, verbose=True)
    assert set(s) == {"mean", "median", "max", "min", "std", "values", "perm"} and s["max"] >= s["median"] >= s["min"] >= 0



def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU port of the reference step, rank 0 only) prints exactly one JSON line with the contract's
    keys; it is the one place outside tests / smoke where oracle/ code runs (as the baseline, never as the product)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-sample", "8"], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "jets/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_bench_dump_writes_the_step_outputs_within_the_limit(tmp_path):
    """`bench.py --dump-outputs`: one float32 / float64 .npy per output of the step; above the byte limit latent and recon keep the
    same seeded sample of jets on every call, and the files stay within the limit."""
    import types
    import numpy as np
    import torch
    import bench
    B, N = 50, 7
    g = torch.Generator().manual_seed(0)
    tr = types.SimpleNamespace(B=B, latent=torch.randn(B, 4, generator=g), recon=torch.randn(B, N, 3, generator=g),
                               grad=torch.randn(100, generator=g), flat=torch.randn(100, generator=g),
                               stats=torch.tensor([0, 0, 2.5, 0, 0, 0, 0, 0]), loss_from_stats=lambda s: float(s[2]))
    load = lambda d: {p.stem: np.load(p) for p in d.glob("*.npy")}
    bench.dump_timed_outputs(tr, str(tmp_path / "all"))
    full = load(tmp_path / "all")
    assert sorted(full) == ["grad", "latent", "loss", "params", "recon"]
    assert all(a.dtype in (np.float32, np.float64) for a in full.values()) and full["loss"] == 2.5
    for k, t in (("latent", tr.latent), ("recon", tr.recon), ("grad", tr.grad), ("params", tr.flat)):
        assert np.array_equal(full[k], t.numpy())
    limit = 2 * 100 * 4 + 8 + 5 * 128 + 20 * (4 + N * 3) * 4      # room for 20 of the 50 jets
    for d in ("a", "b"):
        bench.dump_timed_outputs(tr, str(tmp_path / d), limit=limit)
        assert sum(p.stat().st_size for p in (tmp_path / d).glob("*.npy")) <= limit
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    rows = np.sort(np.random.default_rng(0).choice(B, 20, replace=False))
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert np.array_equal(a["recon"], full["recon"][rows]) and np.array_equal(a["latent"], full["latent"][rows])
    assert np.array_equal(a["grad"], full["grad"]) and np.array_equal(a["params"], full["params"])
