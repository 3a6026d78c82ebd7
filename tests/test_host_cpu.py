"""CPU: host-side logic of the drop-in (no kernels are launched): the C-ABI library loads and exports every
declared symbol, weight readers agree with the oracle's, schedule / topology helpers match the reference's
semantics, and the product never routes through the oracle."""
import os
import re
import subprocess
import sys
import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    from pipeedge_b200 import _lib
    with open(os.path.join(ROOT, 'include', 'pipeedge_b200.h'), encoding='utf-8') as fh:
        header = fh.read()
    declared = set(re.findall(r'^\s*(?:const\s+)?[a-z_0-9]+\*?\s+(pe_[a-z0-9_]+)\s*\(', header, flags=re.M))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SYMBOLS), (declared ^ set(_lib.SYMBOLS))
    for name in declared:
        assert hasattr(_lib.LIB, name), name
    assert _lib.LIB.pe_abi_version() == _lib.PE_ABI_VERSION == 2
    assert _lib.LIB.pe_quant_words(152064, 8) == 38016     # C5 hop: 4.87 MB of codes per 32 items
    assert _lib.LIB.pe_quant_words(10, 6) == 2              # 5 codes per word
    assert _lib.LIB.pe_quant_words(10, 0) == 0


def test_no_gpu_means_loud_failure_not_fallback():
    """Without a CUDA device every compute entry point refuses (PE_ERR_DEVICE) - there is no CPU path."""
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from pipeedge_b200 import _lib
    rc = _lib.LIB.pe_layernorm(None, None, None, 1e-12, None, None, 1, 4, None)
    assert rc == -3 and b'no CUDA device' in _lib.LIB.pe_last_error()
    import ctypes
    handle = ctypes.c_void_p()
    for rc in (_lib.LIB.pe_link_open_local(1 << 20, 4, 0, ctypes.byref(handle)),
               _lib.LIB.pe_link_open_host(1 << 20, 4, ctypes.byref(handle)),
               _lib.LIB.pe_linear_residual_layernorm(None, None, None, None, None, None, 1e-12, None, 0, None, 1, 768, 768, 1,
                                                     None)):
        assert rc < 0, "link / fused kernels must refuse to run without an sm_100 device"
    assert _lib.LIB.pe_linear_ln_cluster(768) == 8 and _lib.LIB.pe_linear_ln_cluster(1024) == 8
    assert _lib.LIB.pe_linear_ln_cluster(128) == 4 and _lib.LIB.pe_linear_ln_cluster(160) == 0      # host-only planning
    from pipeedge_b200.models.transformers._stage import EncoderStage
    from pipeedge_b200.synth import MODEL_SPECS, hf_config, synth_weights
    spec = MODEL_SPECS['test/vit-tiny']
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        EncoderStage('vit', hf_config(spec), 1, 4, synth_weights(spec), spec.tokens)


def test_clamp_factor_matches_scipy_lambertw():
    from scipy.special import lambertw
    from pipeedge_b200 import _lib
    for bit in range(1, 17):
        for gelu in (0, 1):
            want = np.float32(lambertw(3.0 * 4.0 ** (bit + gelu)).real)
            assert np.float32(_lib.LIB.pe_quant_clamp_factor(bit, gelu)) == want, (bit, gelu)


@pytest.mark.parametrize('name', ['test/vit-tiny', 'test/deit-tiny', 'test/bert-tiny', 'test/vit-huge-tiny'])
def test_weight_readers_agree_with_oracle(name):
    """npz layout -> kernel layout ([3H,H] fused QKV etc.) vs the oracle's own restatement of the loaders."""
    from oracle import shards as osh
    from pipeedge_b200.models.transformers import _stage
    from pipeedge_b200.synth import MODEL_SPECS, synth_weights
    spec = MODEL_SPECS[name]
    w = synth_weights(spec, seed=0)
    inner = osh._bert_inner(spec, w)   # pylint: disable=protected-access
    for block in range(spec.blocks):
        got = _stage._BLOCK_READERS[spec.family](inner, block, spec.hidden, range(4))   # pylint: disable=protected-access
        ref = osh.block_params(spec.family, inner, block, spec.hidden)
        np.testing.assert_array_equal(np.asarray(got['w_qkv']),
                                      torch.cat([ref['wq'], ref['wk'], ref['wv']], 0).numpy())
        np.testing.assert_array_equal(np.asarray(got['b_qkv']), torch.cat([ref['bq'], ref['bk'], ref['bv']]).numpy())
        for ours, theirs in (('w_o', 'wo'), ('b_o', 'bo'), ('w_fc1', 'w1'), ('b_fc1', 'b1'), ('w_fc2', 'w2'),
                             ('b_fc2', 'b2'), ('ln1_w', 'ln1_w'), ('ln1_b', 'ln1_b'), ('ln2_w', 'ln2_w'),
                             ('ln2_b', 'ln2_b')):
            np.testing.assert_array_equal(np.asarray(got[ours]), ref[theirs].numpy(), err_msg=ours)


def test_sublayer_ranges_and_partitions():
    from pipeedge_b200.models.transformers._stage import sublayer_ranges
    from oracle.shards import sublayer_ranges as oracle_ranges
    for lo in range(1, 14):
        for hi in range(lo, 14):
            assert sublayer_ranges(lo, hi) == oracle_ranges(lo, hi)
    sys.path.insert(0, ROOT)
    import bench
    assert bench.even_partition(48, 2) == [(1, 24), (25, 48)]
    assert bench.even_partition(48, 8)[1] == (7, 12)
    assert bench.even_partition(96, 4) == [(1, 24), (25, 48), (49, 72), (73, 96)]
    assert sum(hi - lo + 1 for lo, hi in bench.even_partition(48, 5)) == 48


def test_model_cfg_registry_and_topology():
    sys.path.insert(0, ROOT)
    import model_cfg
    assert model_cfg.get_model_layers('google/vit-base-patch16-224') == 48
    assert model_cfg.get_model_layers('google/vit-large-patch16-224') == 96
    assert model_cfg.get_model_default_weights_file('textattack/bert-base-uncased-CoLA') == 'BERT-B-CoLA.npz'
    cfg = model_cfg.get_model_config('google/vit-large-patch16-224')
    assert (cfg.hidden_size, cfg.num_attention_heads, cfg.intermediate_size, cfg.num_hidden_layers) == (1024, 16, 4096, 24)
    assert set(model_cfg.get_model_names()) >= {'bert-base-uncased', 'facebook/deit-tiny-distilled-patch16-224'}
    # topology (model_cfg.py:128-166), inspected through the threads the stage creates
    mk = model_cfg.dist_p2p_pipeline_stage_factory
    cb = lambda x: None   # noqa: E731
    st = mk([0, 1, 2], 0, 0, 0, cb, cb)._threads      # data rank = stage 0 of 3
    assert st['recv']._src_rank == 2 and st['send']._dst_rank == 1 and 'res' in st and 'work' in st
    st = mk([0, 1, 2], 0, 2, 2, cb, cb)._threads      # last stage sends results to the data rank
    assert st['recv']._src_rank == 1 and st['send']._dst_rank == 0 and 'res' not in st
    st = mk([1, 2], 0, 0, None, None, cb)._threads    # data rank outside the pipeline: relay, no worker
    assert st['recv']._src_rank == 2 and st['send']._dst_rank == 1 and 'work' not in st
    assert mk([0], 0, 0, 0, cb, cb)._threads.keys() == {'work', 'res'}   # degenerate single stage
    assert not mk([0, 1], 0, 3, None, None, cb)._threads                 # idle rank
    with pytest.raises(ValueError):
        mk([1, 0], 0, 0, 1, cb, cb)                                      # data rank must be stage 0


def test_runtime_schedule_resolution():
    sys.path.insert(0, ROOT)
    import runtime
    assert runtime.get_pipeline_sched(1, None, None, None, 'google/vit-base-patch16-224') == ([(1, 48)], [0], [0])
    layers, quant, ranks = runtime.get_pipeline_sched(2, [(1, 24), (25, 48)], [8, 0], None, 'google/vit-base-patch16-224')
    assert (layers, quant, ranks) == ([(1, 24), (25, 48)], [8, 0], [0, 1])
    with pytest.raises(RuntimeError):
        runtime.get_pipeline_sched(2, None, [8, 0], None, 'google/vit-base-patch16-224')
    with pytest.raises(RuntimeError):
        runtime.get_pipeline_sched(2, None, None, None, 'google/vit-base-patch16-224')   # sched-pipeline: out of scope


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing shipped may import it; bench.py only inside its CPU arm."""
    offenders = []
    for base in ('pipeedge_b200', 'runtime.py', 'model_cfg.py', 'devices.py'):
        path = os.path.join(ROOT, base)
        files = [path] if os.path.isfile(path) else [os.path.join(d, f) for d, _, fs in os.walk(path) for f in fs
                                                     if f.endswith('.py')]
        for file in files:
            with open(file, encoding='utf-8') as fh:
                if re.search(r'^\s*(from|import)\s+oracle\b', fh.read(), flags=re.M):
                    offenders.append(file)
    assert not offenders, offenders
    with open(os.path.join(ROOT, 'bench.py'), encoding='utf-8') as fh:
        src = fh.read()
    assert len(re.findall(r'^\s*(from|import)\s+oracle\b', src, flags=re.M)) == 1   # cpu_forward_timer only
    assert '/root/reference' not in src


def test_bench_reference_arm_cli(tmp_path):
    """`bench.py --impl reference` prints one JSON line with the contract's keys (tiny sample), times exactly `--steps`
    forwards, and `--dump-outputs` writes the last forward's logits: the oracle's logits for the seeded input."""
    import json
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1',
                          '--warmup', '1', '--dump-outputs', str(tmp_path)], capture_output=True, text=True, timeout=600,
                         check=True)
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['unit'] == 'images/s' and line['higher_is_better'] is True
    assert line['cpu_baseline']['kind'] == 'port' and line['e2e']['h2d_bytes_per_step'] == 0
    assert line['value'] > 0 and line['steps'] == 1
    from oracle import shards as osh
    from pipeedge_b200.synth import MODEL_SPECS, synth_input, synth_weights
    spec = MODEL_SPECS['google/vit-base-patch16-224']
    want = osh.shard_forward(spec, synth_weights(spec, seed=0), 1, spec.layers, synth_input(spec, 8, seed=1)).numpy()
    got = np.load(tmp_path / 'logits.npy')
    assert got.dtype == np.float32 and got.shape == (8, 1000)
    np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4)


def _gemm_plan(m, n, k, epi):
    import ctypes
    from pipeedge_b200 import _lib
    out = (ctypes.c_int * 6)()
    _lib.check(_lib.LIB.pe_debug_gemm_plan(m, n, k, epi, out))
    return dict(zip(('cm', 'cn', 'bn', 'stages', 'tiles', 'ctas'), out))


def test_gemm_tile_plans_of_the_headline_shapes():
    """`plan_gemm` is host code: the ViT-B ubatch-8 plans are the ones the sweep in profiles/r01d_plan_sweep.txt found
    best (DESIGN.md 4a), and the ring depth follows from the 144 / 224 KiB budgets."""
    from pipeedge_b200 import _lib
    m = 8 * 197
    assert _gemm_plan(m, 2304, 768, _lib.PE_EPI_F16) == {'cm': 1, 'cn': 1, 'bn': 224, 'stages': 5, 'tiles': 143, 'ctas': 143}
    assert _gemm_plan(m, 768, 768, _lib.PE_EPI_F32)['bn'] == 96
    fc1 = _gemm_plan(m, 3072, 768, _lib.PE_EPI_GELU_F16)
    assert (fc1['bn'], fc1['tiles'], fc1['ctas'], fc1['stages']) == (160, 260, 148, 4)   # two tiles per CTA: no aliasing
    fc2 = _gemm_plan(m, 768, 3072, _lib.PE_EPI_F32)
    assert (fc2['bn'], fc2['tiles'], fc2['stages']) == (96, 104, 8)


def test_gemm_tile_plan_invariants():
    """Any shape: BN a multiple of 32 in [32, 256], 2..8 stages that fit the shared-memory budget, a grid of at most
    148 CTAs covering all tiles."""
    import random
    from pipeedge_b200 import _lib
    rng = random.Random(3)
    for _ in range(300):
        m, n, k = rng.randint(1, 9000), rng.randint(1, 6000), 8 * rng.randint(1, 700)
        epi = rng.choice([_lib.PE_EPI_F16, _lib.PE_EPI_GELU_F16, _lib.PE_EPI_RESID_F32, _lib.PE_EPI_F32, _lib.PE_EPI_TANH_F32])
        p = _gemm_plan(m, n, k, epi)
        assert p['bn'] % 32 == 0 and 32 <= p['bn'] <= 256 and p['cm'] * p['cn'] <= 8
        assert p['tiles'] == -(-m // 128) * -(-n // p['bn'])
        assert 1 <= p['ctas'] <= 148 and p['ctas'] <= p['tiles'] * p['cm'] * p['cn']
        stage_bytes = 128 * 128 + p['bn'] * 128
        budget = (144 + 80) * 1024 if p['tiles'] <= p['ctas'] else 144 * 1024
        assert 2 <= p['stages'] <= 8 and (p['stages'] * stage_bytes <= budget or p['stages'] == 2)
    with pytest.raises(_lib.PipeEdgeB200Error):
        _gemm_plan(0, 8, 8, _lib.PE_EPI_F32)


def test_parse_yaml_sched_matches_the_reference(tmp_path):
    """`runtime.parse_yaml_sched` / `get_pipeline_sched` on the scheduler's YAML vs what the reference's own function
    returned for the same documents (`tests/golden/sched.json`, made by `oracle/make_goldens.py sched`)."""
    import json
    import yaml
    import runtime as rt
    with open(os.path.join(ROOT, 'tests', 'golden', 'sched.json'), encoding='utf-8') as fh:
        cases = json.load(fh)
    assert len(cases) >= 8
    for case in cases:
        sched = yaml.safe_load(case['yaml'])
        if 'error' in case:
            with pytest.raises((ValueError, RuntimeError)) as info:
                rt.parse_yaml_sched(sched, case['hosts'])
            assert type(info.value).__name__ == case['error']
        else:
            layers, ranks = rt.parse_yaml_sched(sched, case['hosts'])
            assert [list(l) for l in layers] == case['layers'] and ranks == case['ranks']
    # through get_pipeline_sched with a schedule file, as `runtime.py RANK 8 -H gpu0,...,gpu7 --sched-file f` would
    eight = next(c for c in cases if c.get('hosts') and len(c['hosts']) == 8)
    path = tmp_path / 'sched.yml'
    path.write_text(eight['yaml'])
    layers, quant, ranks = rt.get_pipeline_sched(8, None, None, None, 'google/vit-base-patch16-224', hosts=eight['hosts'],
                                                 sched_file=str(path))
    assert [list(l) for l in layers] == eight['layers'] and ranks == eight['ranks'] and quant == [0] * 8
    with pytest.raises(RuntimeError, match="hosts count"):
        rt.get_pipeline_sched(4, None, None, None, 'google/vit-base-patch16-224', hosts=eight['hosts'], sched_file=str(path))
