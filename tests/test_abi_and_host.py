"""CPU-side tests: the C-ABI library loads and exports every symbol include/pf_b200.h declares,
argument errors follow the error convention without touching a GPU, host-side planning logic is
right, and the oracle still reproduces the committed golden vectors."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import pf_oracle as O
from pocketflow_b200 import lib, ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32


def header_symbols():
    out = []
    for fn in sorted(os.listdir(os.path.join(ROOT, 'include'))):
        src = open(os.path.join(ROOT, 'include', fn)).read()
        src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
        out += re.findall(r'\b(pf_[a-z0-9_]+)\s*\(', src)
    return sorted(set(out))


def test_library_exports_every_declared_symbol():
    L = lib.load()
    syms = header_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(L, s), 'libpf_b200.so does not export %s' % s
    assert set(lib.SIGNATURES) == set(syms), set(lib.SIGNATURES) ^ set(syms)
    assert L.pf_abi_version() == 1


def test_missing_library_fails_loudly(monkeypatch):
    monkeypatch.setattr(lib, '_lib', None)
    monkeypatch.setattr(lib, 'LIB_PATH', '/nonexistent/libpf_b200.so')
    with pytest.raises(lib.PFLibraryMissing):
        lib.load()


def test_argument_errors_map_to_valueerror():
    L = lib.load()
    st = L.pf_uq_act_quant(None, None, -1, None, 8, None)
    assert st == -1
    with pytest.raises(ValueError):
        lib.check(st, 'pf_uq_act_quant')
    assert b'n < 0' in L.pf_last_error()
    assert L.pf_uq_act_quant(None, None, 16, None, 0, None) == -1       # bits out of range
    assert L.pf_softmax_ce_fwd_bwd(None, None, None, 0, 10, 4.0, 4.0, None, None, None, None) == -1
    assert L.pf_uq_weight_quant(None, None, 0, None, 0, None) == 0         # empty work = no-op
    assert L.pf_momentum_step(None, None, None, None, 0, None, 0.9, 0.0, 1.0, None) == 0
    with pytest.raises(RuntimeError):
        lib.check(700, 'x')


def test_comm_entry_points_bind_nccl_at_run_time_and_validate_arguments():
    """pf_comm_* (the step's collective behind the C ABI): NCCL is bound with dlopen, not linked — the version query and
    the unique id need no GPU; argument errors come back as status codes, never as crashes."""
    import ctypes
    L = lib.load()
    v = ctypes.c_int32(0)
    st = L.pf_comm_nccl_version(ctypes.byref(v))
    if st != 0:
        pytest.skip('libnccl.so.2 is not loadable here: ' + L.pf_last_error().decode())
    assert v.value >= 20000
    a, b = ctypes.create_string_buffer(128), ctypes.create_string_buffer(128)
    assert L.pf_comm_unique_id(a) == 0 and L.pf_comm_unique_id(b) == 0 and a.raw != b.raw
    assert L.pf_comm_unique_id(None) == -1
    h = ctypes.c_void_p()
    assert L.pf_comm_init(a, 2, 5, ctypes.byref(h)) == -1                 # rank out of range: refused before NCCL
    assert L.pf_comm_init(None, 1, 0, ctypes.byref(h)) == -1
    assert L.pf_allreduce_flat(None, None, 0, None) == 0                  # empty range = no-op
    assert L.pf_allreduce_flat(None, None, 16, None) == -1                # no communicator / buffer
    assert L.pf_broadcast_flat(None, None, 16, 0, None) == -1
    assert L.pf_comm_destroy(None) == 0


def test_struct_layouts_match_header():
    assert ops.UQ_SEG.itemsize == 48 and ops.UQ_SEG.fields['ncols'][1] == 32
    assert ops.WORK.itemsize == 32 and ops.WORK.fields['start'][1] == 8
    assert ops.WS_SEG.itemsize == 32


def test_bucket_layouts():
    assert ops.uq_bucket_layout((3, 3, 64, 128), False, 'channel', 256) == (1, 73728)
    assert ops.uq_bucket_layout((3, 3, 64, 128), True, 'channel', 256) == (128, 73728)
    assert ops.uq_bucket_layout((3, 3, 64, 128), True, 'split', 256) == (288, 73728)
    assert ops.uq_bucket_layout((10,), True, 'split', 4) == (3, 12)
    with pytest.raises(ValueError):
        ops.uq_bucket_layout((4, 4), True, 'bogus', 4)


@pytest.mark.parametrize('numels', [[1], [8192], [8193, 5], [100000, 7, 0, 16384]])
def test_flat_works_cover_exactly(numels):
    w = ops.flat_works(numels)
    for s, n in enumerate(numels):
        mine = w[w['seg'] == s]
        covered = np.zeros(n, np.int32)
        for r in mine:
            assert r['start'] % 4 == 0 and r['kind'] == 0
            covered[r['start']:r['start'] + r['count']] += 1
        assert np.all(covered == 1)


def test_minmax_works_cover_exactly():
    segs = np.zeros(4, dtype=ops.UQ_SEG)
    segs[0] = (0, 0, 3 * 3 * 64 * 64, 3 * 3 * 64 * 64, 64, 0, 8, 0)       # channel
    segs[1] = (0, 0, 2048 * 1001, 2048 * 1001, 1001, 64, 8, 0)           # ncols % 4 != 0
    segs[2] = (0, 0, 1000, 1024, 4, 1068, 8, 0)                           # split, padded
    segs[3] = (0, 0, 50000, 50000, 1, 1072, 8, 0)                         # per-layer
    w = ops.minmax_works(segs)
    for s in range(3):
        nc = int(segs[s]['ncols'])
        nr = int(segs[s]['padded']) // nc
        cov = np.zeros((nr, nc), np.int32)
        for r in w[w['seg'] == s]:
            assert r['kind'] == 1 and (nc % 4 or (r['c0'] % 4 == 0 and r['ncol_tile'] % 4 == 0))
            assert r['ncol_tile'] <= 1024
            cov[r['start']:r['start'] + r['count'], r['c0']:r['c0'] + r['ncol_tile']] += 1
        assert np.all(cov == 1)
    assert np.all(w[w['seg'] == 3]['kind'] == 0)


def test_percentile_rank_matches_oracle():
    for n in (1, 2, 10, 777, 2359296):
        for r in (0.0, 0.1, 0.25, 0.5, 0.75, 0.999, 1.0):
            assert ops.ws_rank_desc(n, r) == O.ws_mask_rank(n, r)
        for q in (0.0, 5.88, 50.0, 94.1, 100.0):
            assert ops.percentile_rank_desc(n, q) == O.percentile_index(n, q)


def test_ordered_encoding_roundtrip():
    f = np.array([0.0, -0.0, 1.5, -1.5, 3e38, -3e38, 1e-40, -1e-40, np.inf, -np.inf], F32)
    u = f.view(np.uint32)
    enc = np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.uint32)
    assert np.array_equal(ops.decode_ordered(enc).view(np.uint32), u)
    keep = np.array([i for i in range(len(f)) if i != 1])       # -0.0 == 0.0 for argsort, enc(-0) < enc(+0)
    order = keep[np.argsort(f[keep], kind='stable')]
    assert np.all(np.diff(enc[order].astype(np.int64)) > 0)


def test_oracle_reproduces_golden():
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'hotpath_v1.npz'))
    for i in range(6):
        w = g['w%d' % i]
        for bits in (2, 4, 8):
            assert np.array_equal(O.uniform_quantize(w, bits), g['w%d_layer_b%d' % (i, bits)])
            assert np.array_equal(O.uniform_quantize(w, bits, use_buckets=True, bucket_type='channel'),
                                  g['w%d_channel_b%d' % (i, bits)])
            assert np.array_equal(O.uniform_quantize(w, bits, use_buckets=True, bucket_type='split', bucket_size=16),
                                  g['w%d_split_b%d' % (i, bits)])
    assert np.array_equal(O.uniform_quantize(g['act'], 8, mode='activation'), g['act_b8'])
    for r in (0.0, 0.3, 0.5, 0.9):
        v2, b2, m2, thr = O.ws_build_mask(g['ws_w'], g['ws_bkup'], g['ws_mask'], r)
        tag = 'ws_r%02d' % int(r * 100)
        assert np.array_equal(m2, g[tag + '_mask']) and np.array_equal(v2, g[tag + '_w'])
    qx, c, idx = O.nonuniform_quantize(g['nuq_w'], 4)
    assert np.array_equal(qx, g['nuq_q']) and np.array_equal(c, g['nuq_c'])


def test_space_to_depth_maps_reproduce_the_strided_conv():
    """Host logic of the stride-2 stem: x' = space-to-depth(x), w' = gather(w, fwd_map) turns the RxS stride-2 conv
    into a ceil(R/2) x ceil(S/2) stride-1 conv (float64 on the CPU), and bwd_map inverts fwd_map."""
    import torch
    import torch.nn.functional as F
    from pocketflow_b200 import ops
    for (n, h, c, k, r, pt) in [(2, 23, 3, 8, 7, 3), (1, 16, 3, 4, 3, 0), (2, 20, 4, 6, 5, 2)]:
        g = torch.Generator().manual_seed(n + h + r)
        x = torch.randn(n, h, h, c, generator=g, dtype=torch.float64)
        w = torch.randn(r, r, c, k, generator=g, dtype=torch.float64)
        pb = max(r - 1 - pt, 0)
        p = (h + pt + pb - r) // 2 + 1
        ref = F.conv2d(F.pad(x.permute(0, 3, 1, 2), (pt, pb, pt, pb)), w.permute(3, 2, 0, 1), stride=2).permute(0, 2, 3, 1)
        r2, s2, fwd, bwd = ops.s2d_weight_maps(r, r, c, 16)
        hp = p + r2 - 1
        xs = torch.zeros(n, hp, hp, 16, dtype=torch.float64)
        for yq in range(hp):
            for xq in range(hp):
                for dy in range(2):
                    for dx in range(2):
                        ih, iw = 2 * yq + dy - pt, 2 * xq + dx - pt
                        if 0 <= ih < h and 0 <= iw < h:
                            xs[:, yq, xq, (dy * 2 + dx) * c:(dy * 2 + dx) * c + c] = x[:, ih, iw, :]
        w2 = torch.zeros(r2 * s2 * 16, k, dtype=torch.float64)
        wf = w.reshape(-1, k)
        for j, src in enumerate(fwd):
            if src >= 0:
                w2[j] = wf[src]
        out = F.conv2d(xs.permute(0, 3, 1, 2), w2.reshape(r2, s2, 16, k).permute(3, 2, 0, 1)).permute(0, 2, 3, 1)
        assert out.shape == ref.shape and (out - ref).abs().max().item() < 1e-10
        assert all(fwd[bwd[i]] == i for i in range(r * r * c))


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver times beside the GPU arm): exactly ONE line on stdout, valid
    JSON, with the contract's keys; runs without a GPU."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1',
                          '--workload', 'lenet_uq8_b128'], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.split('\n') if ln.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
              'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['value'] > 0 and d['config']['workload'] == 'lenet_uq8_b128'
    assert set(('value', 'unit', 'cores', 'kind', 'sample')) <= set(d['cpu_baseline'])
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0


def test_bench_dump_outputs_is_reproducible_and_bounded(tmp_path):
    """bench.dump_outputs: float32 .npy per loss term and per variable, large variables sampled at the same indices in
    every run, the whole dump within DUMP_LIMIT_BYTES even when the model has many large variables."""
    import bench
    rng = np.random.default_rng(5)
    losses = {'loss': F32(2.5), 'ce': F32(2.25)}
    state = {'model/conv/kernel:0': rng.standard_normal((3, 3, 64, 128)).astype(F32),
             'model/bn/beta:0': rng.standard_normal(64).astype(F32)}
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), losses, state)
    names = sorted(os.listdir(str(tmp_path / 'a')))
    assert names == ['loss.ce.npy', 'loss.loss.npy', 'var.model.bn.beta_0.npy', 'var.model.conv.kernel_0.npy']
    for n in names:
        a, b = np.load(str(tmp_path / 'a' / n)), np.load(str(tmp_path / 'b' / n))
        assert a.dtype == F32 and np.array_equal(a, b), n
    assert np.array_equal(np.load(str(tmp_path / 'a' / 'var.model.bn.beta_0.npy')), state['model/bn/beta:0'])
    k = np.load(str(tmp_path / 'a' / 'var.model.conv.kernel_0.npy'))
    assert k.shape == (bench.DUMP_SAMPLE,) and np.isin(k, state['model/conv/kernel:0']).all()
    big = {'v%d' % i: np.zeros(bench.DUMP_SAMPLE + 1, F32) for i in range(300)}
    bench.dump_outputs(str(tmp_path / 'c'), losses, big)
    assert sum(os.path.getsize(str(p)) for p in (tmp_path / 'c').iterdir()) <= bench.DUMP_LIMIT_BYTES + 128 * 302


def test_run_scripts_parse_flags_and_map_value_errors_to_exit_status_1(capsys):
    """nets/*_run.py: every learner's flags are known before parsing; a bad execution mode or learner name is a
    ValueError -> exit status 1 (nets/resnet_at_cifar10_run.py:62-66), not a traceback to the shell."""
    import importlib
    from pocketflow_b200.flags import FLAGS
    from pocketflow_b200.nets import run_utils
    for net in ('lenet_at_cifar10', 'resnet_at_cifar10', 'resnet_at_ilsvrc12', 'mobilenet_at_ilsvrc12'):
        FLAGS.reset()
        mod = importlib.import_module('pocketflow_b200.nets.' + net + '_run')
        assert run_utils.run(mod.ModelHelper, ['--learner', 'uniform', '--uql_weight_bits', '8', '--ws_prune_ratio', '0.5',
                                               '--exec_mode', 'bogus', '--nuql_equivalent_bits=3', '--noenbl_dst']) == 1
        assert FLAGS.uql_weight_bits == 8 and FLAGS.ws_prune_ratio == 0.5 and FLAGS.enbl_dst is False
        assert 'unrecognized' in capsys.readouterr().err
        FLAGS.reset()
        assert run_utils.run(mod.ModelHelper, ['--learner', 'dis-chn-pruned']) == 1
        assert 'outside the hot-path scope' in capsys.readouterr().err
        assert run_utils.run(mod.ModelHelper, ['--no_such_flag', '1']) == 1
    FLAGS.reset()
