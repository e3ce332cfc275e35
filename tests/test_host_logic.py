"""CPU-side tests: host logic of the drop-in surface, the C-ABI export table, and the 2-rank gather (gloo)."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import torch

import quanto_b200 as q
from oracle import quanto_oracle as O
from quanto_b200 import _native
from quanto_b200.parallel import _unpack_rows, shard_weight
from quanto_b200.tensor.packed import pack_weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "quanto_b200.h")).read()
    declared = set(re.findall(r"QB200_API\s+[\w\s\*]+?\b(qb200_\w+)\s*\(", header))
    assert declared == set(_native.EXPORTS), declared ^ set(_native.EXPORTS)
    lib = ctypes.CDLL(_native.lib_path())
    for name in declared:
        assert hasattr(lib, name), name
    assert _native.load().qb200_version() >= 100


def test_ops_registered_with_reference_schemas():
    for name in ("unpack", "qbytes_mm", "quantize_symmetric", "quantize_affine", "qbits_mm", "dequantize_qbits"):
        assert hasattr(torch.ops.quanto, name)
    s = str(torch.ops.quanto.qbytes_mm.default._schema)
    assert "Tensor A, Tensor B, Tensor scales" in s
    s = str(torch.ops.quanto.quantize_symmetric.default._schema)
    assert "ScalarType dtype" in s and "int? axis" in s


def test_no_cpu_fallback():
    with pytest.raises(NotImplementedError):
        torch.ops.quanto.unpack(torch.zeros(4, dtype=torch.uint8), 4)
    with pytest.raises(NotImplementedError):
        torch.ops.quanto.qbytes_mm(torch.zeros(2, 16, dtype=torch.int8), torch.zeros(4, 16, dtype=torch.int8),
                                   torch.ones(4, 1))


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "optimum-quanto_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("# oracle", ""), os.path.join(dirpath, f)


@pytest.mark.parametrize("bits", [2, 4])
@pytest.mark.parametrize("shape", [(10,), (12,), (10, 8), (12, 8), (64, 128)])
def test_pack_weights_matches_oracle(bits, shape):
    g = torch.Generator().manual_seed(0)
    u = torch.randint(0, 2**bits, shape, dtype=torch.uint8, generator=g)
    packed = pack_weights(u, bits)
    assert np.array_equal(packed.numpy(), O.pack_weights(u.numpy(), bits))
    assert np.array_equal(_unpack_rows(packed, bits, shape[0]).numpy(), u.numpy())
    pt = q.PackedTensor.pack(u, bits)
    assert pt.shape == u.shape and pt.dtype == torch.uint8 and pt.bits == bits


def test_group_ungroup_roundtrip():
    w = torch.arange(4 * 256, dtype=torch.float32).reshape(4, 256)
    for axis in (0, -1):
        t = w if axis == 0 else w.t().contiguous()
        g = q.group(t, axis, 128)
        assert tuple(g.shape) == tuple(q.grouped_shape(t.shape, axis, 128))
        assert torch.equal(q.ungroup(g, axis, t.shape), t)
    assert np.array_equal(q.group(w, 0, 128).numpy(), O.group(w.numpy(), 0, 128))
    with pytest.raises(ValueError):
        q.group(w, 1, 128)


@pytest.mark.parametrize("wq", ["qint4", "qint2"])
def test_qbits_weight_serialization_roundtrip(wq):
    torch.manual_seed(0)
    lin = torch.nn.Linear(256, 64, bias=True).to(torch.bfloat16)
    ql = q.QLinear.from_module(lin, weights=q.qtypes[wq])
    assert ql.weight_group_size == 128 and not ql.frozen
    ql.freeze()
    assert ql.frozen and isinstance(ql.weight, q.WeightQBitsTensor)
    sd = ql.state_dict()
    assert set(sd) == {"weight._data._data", "weight._scale", "weight._shift", "bias", "input_scale", "output_scale"}
    per_byte = 8 // q.qtypes[wq].bits
    assert sd["weight._data._data"].shape == (64 * 256 // 128 // per_byte, 128)
    ql2 = q.QLinear.from_module(lin, weights=q.qtypes[wq])
    ql2.load_state_dict(sd)
    assert ql2.frozen and torch.equal(ql2.weight, ql.weight)
    # canonical packing agrees with the oracle's pack of the same nibbles
    rows = 64 * 256 // 128
    u = _unpack_rows(sd["weight._data._data"], q.qtypes[wq].bits, rows)
    assert np.array_equal(O.pack_weights(u.numpy(), q.qtypes[wq].bits), sd["weight._data._data"].numpy())


def test_group_size_rule():
    from quanto_b200.nn import _pick_group_size
    assert [_pick_group_size(k) for k in (4096, 14336, 160, 96, 128, 200)] == [128, 128, 32, None, None, None]


def test_qlinear_state_dict_matches_reference_fixture(golden_dir):
    """The reference's own serialized QLinear (tests/golden/qlinear.npz) loads into our QLinear unchanged."""
    z = np.load(os.path.join(golden_dir, "qlinear.npz"))
    tdt = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}

    def tt(arr, dtype):
        if dtype in (torch.float16, torch.bfloat16):
            return torch.from_numpy(arr.view(np.int16).copy()).view(dtype)
        return torch.from_numpy(arr.copy())

    for i in range(int(z["n"])):
        p = f"c{i}_"
        dtype = tdt[str(z[p + "tag"])]
        N, K, M, G = (int(v) for v in z[p + "shape"])
        wq = q.qtypes[str(z[p + "wq"])]
        aq = None if str(z[p + "aq"]) == "none" else q.qtypes[str(z[p + "aq"])]
        lin = torch.nn.Linear(K, N, bias=True).to(dtype)
        ql = q.QLinear.from_module(lin, weights=wq, activations=aq)
        sd = {"bias": tt(z[p + "bias"], dtype), "input_scale": tt(z[p + "input_scale"], dtype).reshape(()),
              "output_scale": tt(z[p + "output_scale"], dtype).reshape(())}
        for key in z.files:
            if key.startswith(p + "sd_"):
                name = key[len(p) + 3:]
                arr = z[key]
                if name.endswith("_data") and wq.bits == 8 and wq.is_floating_point:
                    sd[name] = torch.from_numpy(arr.copy()).view(wq.dtype)
                elif name.endswith("_data"):
                    sd[name] = torch.from_numpy(arr.copy())
                elif arr.dtype == np.uint8:  # zero-point shift
                    sd[name] = torch.from_numpy(arr.copy())
                else:
                    sd[name] = tt(arr, dtype)
        ql.load_state_dict(sd)
        assert ql.frozen
        out = ql.state_dict()
        for k, v in sd.items():
            a, b = out[k], v
            if a.dtype.is_floating_point and a.element_size() == 1:
                a, b = a.view(torch.uint8), b.view(torch.uint8)
            assert torch.equal(a, b), (i, k)


def test_shard_weight_is_canonical_slice():
    torch.manual_seed(1)
    lin = torch.nn.Linear(256, 64).to(torch.float16)
    ql = q.QLinear.from_module(lin, weights=q.qint4)
    ql.freeze()
    w = ql.weight
    full = _unpack_rows(w._data._data, 4, 128)
    parts = [shard_weight(w, r, 4) for r in range(4)]
    assert all(p.shape == (16, 256) and isinstance(p, q.WeightQBitsTensor) for p in parts)
    assert torch.equal(torch.cat([_unpack_rows(p._data._data, 4, 32) for p in parts]), full)
    assert torch.equal(torch.cat([p._scale for p in parts]), w._scale)
    lin8 = torch.nn.Linear(64, 32).to(torch.float16)
    q8 = q.WeightQBytesTensor(q.qint8, 0, lin8.weight.size(), lin8.weight.stride(),
                              torch.randint(-127, 127, (32, 64), dtype=torch.int8), torch.rand(32, 1).half(), None)
    p8 = [shard_weight(q8, r, 2) for r in range(2)]
    assert torch.equal(torch.cat([p._data for p in p8]), q8._data)
    with pytest.raises(ValueError):
        shard_weight(q8, 0, 3)


def _gloo_worker(rank, world, port, ret):
    import torch.distributed as dist

    from quanto_b200.parallel import gather_columns
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    full = torch.arange(6 * 8, dtype=torch.float32).reshape(6, 8)
    local = full[:, rank * 4:(rank + 1) * 4].contiguous()
    out = gather_columns(local)
    ret[rank] = bool(torch.equal(out, full))
    dist.destroy_process_group()


def test_gather_columns_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    mgr = ctx.Manager()
    ret = mgr.dict()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert ret[0] and ret[1]


def test_torch_port_matches_oracle(golden_dir):
    """The timed CPU-baseline port (oracle/torch_port.py) reproduces the golden dequantisation bit for bit."""
    from oracle import torch_port as P
    z = np.load(os.path.join(golden_dir, "qbits.npz"))
    p = "c0_"
    N, K, G, M = (int(v) for v in z[p + "shape"])
    packed = torch.from_numpy(z[p + "packed"])
    scale = torch.from_numpy(z[p + "scale"].view(np.int16)).view(torch.bfloat16)
    shift = torch.from_numpy(z[p + "shift"].view(np.int16)).view(torch.bfloat16)
    deq = P.dequantize_qbits(packed, scale, shift, N, K, G)
    assert np.array_equal(deq.view(torch.int16).numpy().view(np.uint16), z[p + "deq"])
    a = torch.randint(-127, 127, (32, 64), dtype=torch.int8)
    w = torch.randint(-127, 127, (48, 64), dtype=torch.int8)
    s = (torch.rand(48, 1) / 1e3).to(torch.bfloat16)
    y = P.qbytes_mm(a, w, s)
    ref = O.qbytes_int_mm(a.numpy(), w.numpy(), s.float().numpy().reshape(-1), "bf16")
    assert np.array_equal(y.view(torch.int16).numpy().view(np.uint16), ref)


def test_freeze_host_side_matches_reference_fixture(golden_dir):
    """Host mirror of the weight-freeze step on CPU tensors vs tests/golden/freeze.npz (made by the real reference):
    MaxOptimizer / AbsmaxOptimizer / absmax_scale, the quantize_affine composition and pack_weights."""
    import quanto_b200 as q
    from quanto_b200.library import _affine_mode, quantize_affine_any
    z = np.load(os.path.join(golden_dir, "freeze.npz"))
    tdt = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}

    def tt(arr, tag):
        return torch.from_numpy(arr.copy()) if tag == "f32" else torch.from_numpy(arr.view(np.int16).copy()).view(tdt[tag])

    for i in range(int(z["n_affine"])):
        p = f"a{i}_"
        tag, bits, zp = str(z[p + "tag"]), int(z[p + "bits"]), bool(int(z[p + "zeropoint"]))
        N, K, G = (int(v) for v in z[p + "shape"])
        W = tt(z[p + "W"], tag).reshape(N, K)
        qt = q.qint4 if bits == 4 else q.qint2
        scale, shift = q.MaxOptimizer()(W, qtype=qt, axis=0, group_size=G or None, zeropoint=zp)
        assert np.array_equal(scale.view(torch.int16).numpy().view(np.uint16) if tag != "f32" else scale.numpy(), z[p + "scale"])
        data = quantize_affine_any(W, bits, 0, G or None, scale, shift)
        assert np.array_equal(data.numpy(), z[p + "data"])
        assert np.array_equal(q.pack_weights(data, bits).numpy(), z[p + "packed"])
        grouped = W if not G else W.reshape(-1, G)
        assert _affine_mode(grouped, scale, shift) == 1
    for i in range(int(z["n_absmax"])):
        p = f"s{i}_"
        tag = str(z[p + "tag"])
        W = tt(z[p + "W"], tag)
        qt = {"int8": q.qint8, "e4m3fn": q.qfloat8_e4m3fn, "e5m2": q.qfloat8_e5m2}[str(z[p + "out_tag"])]
        for got, want in ((q.AbsmaxOptimizer()(W, qtype=qt, axis=0), z[p + "scale"]),
                          (q.absmax_scale(W, qt, axis=0), z[p + "scale"]),
                          (q.absmax_scale(W, qt).reshape(1), z[p + "scale_tensor"])):
            got = got.numpy() if tag == "f32" else got.contiguous().view(torch.int16).numpy().view(np.uint16)
            assert np.array_equal(got.reshape(-1), want.reshape(-1)), (i, tag)
    # CPU weights never take the one-launch path (there is no CPU kernel to take)
    lin = torch.nn.Linear(256, 64, bias=False).to(torch.bfloat16)
    ql = q.QLinear.from_module(lin, weights=q.qint4)
    assert ql._fused_qweight() is None


def test_bench_algorithmic_figures_match_the_scope_table():
    """bench.py's roofline numerators are SURVEY.md 8(d)'s algorithmic flops / bytes (also stated in DESIGN.md)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    flops, byts = bench.algorithmic("int4", 4096, 14336, 4096)
    assert flops == 2 * 4096 * 14336 * 4096 and abs(flops - 4.810e11) / 4.810e11 < 1e-3
    assert byts == 182_190_080  # 33,554,432 (A) + 29,360,128 (packed W) + 1,835,008 (scale, shift) + 117,440,512 (out)
    assert bench.algorithmic("int4", 1, 14336, 4096)[1] == 31_232_000
    assert bench.algorithmic("int8", 4096, 14336, 4096)[1] == 192_966_656
    assert bench.algorithmic("int8", 4096, 4096, 4096)[1] == 67_117_056
    # one Llama-3-8B decode step streams 3,707,764,736 B of int4 weights + scales / shifts (lm_head excluded)
    per_layer = sum(n * k // 2 + 2 * (n * k // bench.GROUP) * 2 for _, n, k in bench.LLAMA3_8B_LAYER)
    assert per_layer * 32 == 3_707_764_736
    assert bench.metric_name("qlinear_bf16_int4_m4096") == "qlinear_bf16xint4_tflops"
    assert set(bench.WORKLOADS) >= {"qlinear_bf16_int4_m4096", "decode_m1", "int8_m4096", "llama3_8b_decode_b1"}


def test_bench_dump_outputs_sample_and_files(tmp_path):
    """bench.py --dump-outputs: small results are written whole, a large M as the same two rows of every 32-row band on
    every run, as float32 .npy files, never more than 64 MB in all."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert np.array_equal(bench.dump_rows(32), np.arange(32))
    rows = bench.dump_rows(4096)
    assert len(rows) == 256 and np.all(np.diff(rows) > 0) and np.array_equal(np.bincount(rows // 32), np.full(128, 2))
    assert np.array_equal(rows, bench.dump_rows(4096))
    bench.write_outputs(str(tmp_path / "out"), {"decode_m1": np.ones((1, 8), np.float32)})
    got = np.load(tmp_path / "out" / "decode_m1.npy")
    assert got.dtype == np.float32 and got.shape == (1, 8)
    with pytest.raises(SystemExit):
        bench.write_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_LIMIT_BYTES // 4 + 1, np.float32)})
    assert not (tmp_path / "big").exists()


def test_qlinear_output_hook_passthrough_and_fused_forward_guards():
    """Host logic of the fused output quantisation (nn.py): the hook passes an already quantized output through, the
    fused forward declines CPU weights / unfrozen weights / a removed hook, and the hook bookkeeping follows removal."""
    import quanto_b200 as q
    lin = torch.nn.Linear(64, 32, bias=True).to(torch.bfloat16)
    ql = q.QLinear.from_module(lin, weights=q.qint8, activations=q.qint8)
    assert set(ql._quantize_hooks) == {"input", "output"}
    data = torch.randint(-5, 5, (4, 32), dtype=torch.int8)
    already = q.ActivationQBytesTensor(q.qint8, data.size(), data.stride(), data, torch.tensor(0.5, dtype=torch.bfloat16))
    assert ql.quantize_output(ql, None, already) is already
    x = q.ActivationQBytesTensor(q.qint8, torch.Size([4, 64]), (64, 1), torch.zeros(4, 64, dtype=torch.int8),
                                 torch.tensor(0.1, dtype=torch.bfloat16))
    assert ql._forward_quantized_output(x) is None  # weight not frozen (a float Parameter)
    wd = torch.randint(-127, 127, (32, 64), dtype=torch.int8)
    ql.weight = torch.nn.Parameter(q.WeightQBytesTensor(q.qint8, 0, wd.size(), wd.stride(), wd,
                                                         torch.rand(32, 1).to(torch.bfloat16), q.qint8), requires_grad=False)
    assert ql.frozen and ql._forward_quantized_output(x) is None  # frozen, but on the CPU: no kernel to call
    assert ql._forward_quantized_output(torch.zeros(4, 64, dtype=torch.bfloat16)) is None  # float input
    ql.disable_output_quantization()
    assert set(ql._quantize_hooks) == {"input"}
    ql.disable_output_quantization()  # idempotent


@pytest.mark.parametrize("bits", [4, 2])
@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_shard_packed_rows_equals_unpack_slice_repack(bits, world):
    """Direct sharding of the packed bytes (SURVEY 8f rank 3) == unpack -> slice -> pack_weights, for every rank; and the
    state-dict loader built on it reads only the rank's rows."""
    from quanto_b200.parallel import load_column_shard, shard_packed_rows
    torch.manual_seed(world + bits)
    N, K, G = 64, 256, 128
    rows = N * K // G
    values = torch.randint(0, 2**bits, (rows, G), dtype=torch.uint8)
    packed = q.pack_weights(values, bits)
    scale, shift = torch.rand(rows, 1).to(torch.bfloat16), torch.rand(rows, 1).to(torch.bfloat16)
    qt = q.qint4 if bits == 4 else q.qint2
    w = q.WeightQBitsTensor(qt, 0, G, torch.Size([N, K]), (K, 1), q.PackedTensor(packed, bits, values.size(), values.stride()),
                            scale, shift)
    per = rows // world
    for rank in range(world):
        want = q.pack_weights(values[rank * per:(rank + 1) * per], bits)
        got = shard_packed_rows(packed, bits, rows, rank * per, (rank + 1) * per)
        assert got is not None and torch.equal(got, want), (bits, world, rank)
        sh = shard_weight(w, rank, world)  # takes the direct path
        assert torch.equal(sh._data._data, want) and sh.shape == (N // world, K)
        assert torch.equal(sh._scale, scale[rank * per:(rank + 1) * per])

        class CountingRows:  # stands in for a lazily sliced checkpoint tensor (safetensors get_slice)
            def __init__(self, t):
                self.t, self.rows_read = t, 0

            def __getitem__(self, sl):
                out = self.t[sl]
                self.rows_read += out.shape[0]
                return out

        lazy = CountingRows(packed)
        sd = {"weight._data._data": lazy, "weight._scale": scale, "weight._shift": shift}
        ld = load_column_shard(sd, "weight.", qt, (N, K), G, rank, world)
        assert isinstance(ld, q.WeightQBitsTensor) and torch.equal(ld._data._data, want)
        assert torch.equal(ld._shift, shift[rank * per:(rank + 1) * per]) and ld._group_size == G
        assert lazy.rows_read == per  # only the rank's share of the packed rows (8/bits planes x per/(8/bits) rows)
    # any run whose planes stay inside one plane of the full tensor works ...
    pl = 8 // bits
    assert torch.equal(shard_packed_rows(packed, bits, rows, 1, 1 + pl), q.pack_weights(values[1:1 + pl], bits))
    # ... a length that is not a multiple of the plane count, or a plane straddling two planes of the full tensor, is
    # declined (never mis-sharded)
    assert shard_packed_rows(packed, bits, rows, 0, 3) is None
    packed_rows = rows // pl
    assert shard_packed_rows(packed, bits, rows, packed_rows - 2, packed_rows - 2 + 4 * pl) is None


def test_release_library_ignores_debug_flags_and_env():
    """VERDICT r1 weak #8: the wrong-result knock-outs are compiled out of the release library, the setter is a no-op, and
    no environment variable steers the dispatch (loading the library with QB200_DEBUG_FLAGS set changes nothing)."""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r); from quanto_b200 import _native as n; l = n.load(); "
            "l.qb200_debug_set_flags(1023); print(l.qb200_developer_build(), l.qb200_debug_flags())" %
            os.path.join(ROOT, "optimum-quanto_b200"))
    env = dict(os.environ, QB200_DEBUG_FLAGS="1023")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, check=True).stdout.split()
    assert out == ["0", "0"], out


def test_test_override_keys_are_validated():
    from quanto_b200 import _native as n
    lib = n.load()
    assert lib.qb200_test_override(n.OVR_INT4_TILE_N, 224) == 0
    assert lib.qb200_test_override(n.OVR_INT4_TILE_N, 0) == 0
    assert lib.qb200_test_override(99, 1) == 1  # QB200_ERR_ARG
    with n.test_override(n.OVR_EPILOGUE, 2):
        pass


def test_ring_gemv_cut_of_k_does_not_depend_on_n():
    """Bit-identical column-parallel decode rests on this: the way the ring kernel cuts K (64-byte slabs per warp, passes
    over K) decides the order of every output's sum, so a shard [N / P, K] must be cut exactly like the full [N, K] matrix.
    qb200_qbits_ring_plan is a host-only query of the dispatcher's plan (no GPU involved)."""
    import ctypes

    from quanto_b200 import _native as n
    lib = n.load()
    out = (ctypes.c_int * 5)()
    seen = 0
    for group in (64, 128):
        for zp in (0, 1):
            for k in (2048, 4096, 8192, 11264, 14336):
                for m in range(1, 17):
                    cuts = set()
                    for N in (16, 256, 512, 1024, 1792, 2048, 3584, 4096, 7168, 14336, 28672, 128256):
                        for grid in (148, 132):
                            if lib.qb200_qbits_ring_plan(m, N, k, group, zp, grid, out):
                                cuts.add((out[0], out[1], out[3]))
                                assert out[4] <= 227 * 1024 and out[2] >= 2
                    assert len(cuts) <= 1, (group, zp, k, m, cuts)
                    seen += len(cuts)
    assert seen > 200  # the kernel takes most of these problems
    # the shapes of the Llama-3-8B decode step at batch 1 and 8 run on it, the K = 14336 projection at batch 8 in passes
    assert lib.qb200_qbits_ring_plan(1, 14336, 4096, 128, 0, 148, out) and (out[0], out[1]) == (4, 1)
    assert lib.qb200_qbits_ring_plan(8, 4096, 14336, 128, 0, 148, out) and out[1] > 1


@pytest.mark.parametrize("world", [2, 4, 8])
def test_load_column_shard_from_a_safetensors_checkpoint(tmp_path, world):
    """SURVEY 8f rank 3: a rank's canonical [N / P, K] int4 weight straight from a quanto-format safetensors file (keys
    weight._data._data / _scale / _shift), read through lazy slices, equals the shard of the fully loaded weight."""
    from safetensors.torch import save_file

    from quanto_b200.parallel import load_column_shard_safetensors
    torch.manual_seed(world)
    N, K, G = 128, 512, 128
    rows = N * K // G
    values = torch.randint(0, 16, (rows, G), dtype=torch.uint8)
    packed = q.pack_weights(values, 4)
    scale, shift = torch.rand(rows, 1).to(torch.bfloat16), torch.rand(rows, 1).to(torch.bfloat16)
    path = str(tmp_path / "qlinear.safetensors")
    save_file({"proj.weight._data._data": packed, "proj.weight._scale": scale, "proj.weight._shift": shift,
               "proj.bias": torch.zeros(N)}, path)
    full = q.WeightQBitsTensor(q.qint4, 0, G, torch.Size([N, K]), (K, 1),
                               q.PackedTensor(packed, 4, values.size(), values.stride()), scale, shift)
    for rank in range(world):
        got = load_column_shard_safetensors(path, "proj.weight.", q.qint4, (N, K), G, rank, world)
        want = shard_weight(full, rank, world)
        assert got.shape == want.shape and got._group_size == G
        assert torch.equal(got._data._data, want._data._data)
        assert torch.equal(got._scale, want._scale) and torch.equal(got._shift, want._shift)
    with pytest.raises(KeyError):
        load_column_shard_safetensors(path, "missing.weight.", q.qint4, (N, K), G, 0, world)
