"""Control flow of bench.py's B200 arm with every device call replaced by a stand-in (no GPU): the timed region, the
kernel table, the whole-head roofline and the extra figures are assembled into ONE JSON line with the keys the
contract names, the options they switch are restored, and a failure inside an extra figure is reported as
`unavailable` instead of costing the line.  Also the reference arm's line on a tiny sample."""
import json
import types

import numpy as np
import pytest
import torch

import bench
from agrl.pytorch_b200 import _lib, metrics


class FakeEvent(object):
    clock = [0.0]

    def __init__(self, enable_timing=True):
        self.t = None

    def record(self, stream=None):
        FakeEvent.clock[0] += 1.0
        self.t = FakeEvent.clock[0]

    def elapsed_time(self, other):
        return 10.0 * (other.t - self.t)


class FakeProfile(object):
    def __init__(self, stream):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def totals(self):
        return {'pool': (13, 29.0), 'gemm_graph_layer': (26, 23.0), 'graph': (26, 11.0), 'attn': (13, 1.0),
                'gemm_distance': (1, 0.7), 'rank_mars': (1, 0.3)}


class FakeModel(object):
    def __init__(self, fail_when=None):
        self.head_split = _lib.SPLIT_BF16X2
        self.head_lowrank = True
        self.calls = []
        self.fail_when = fail_when

    def head(self, x1, x2, adj, S, out=None):
        state = (self.head_split, int(self.head_lowrank), 0)
        if self.fail_when is not None and self.fail_when(state):
            raise RuntimeError('injected failure')
        self.calls.append(state + (adj.shape[0],))
        out.zero_()
        return out


@pytest.fixture
def fake_device(monkeypatch):
    cpu = torch.device('cpu')
    real_device = torch.device
    monkeypatch.setattr(bench.torch, 'device', lambda *a, **k: cpu if a and a[0] == 'cuda' else real_device(*a, **k))
    monkeypatch.setattr(torch.cuda, 'set_device', lambda d: None)
    monkeypatch.setattr(torch.cuda, 'current_stream', lambda d=None: types.SimpleNamespace(cuda_stream=0))
    monkeypatch.setattr(torch.cuda, 'Event', FakeEvent)
    monkeypatch.setattr(torch.cuda, 'synchronize', lambda d=None: None)
    monkeypatch.setattr(torch.cuda, 'empty_cache', lambda: None)
    monkeypatch.setattr(_lib, 'require_device', lambda: None)
    monkeypatch.setattr(_lib, 'launch_count', lambda: 0)
    monkeypatch.setattr(_lib, 'profile', FakeProfile)
    monkeypatch.setattr(bench, 'make_pool', lambda n, dev, seed, pinned=False: (
        torch.zeros(n * bench.S, 1), torch.zeros(n * bench.S, 1), torch.zeros(n, 1)))
    monkeypatch.setattr(bench, 'C', 4)
    monkeypatch.setattr(metrics, 'compute_distance_matrix', lambda a, b, m='euclidean': torch.zeros(a.shape[0], b.shape[0]))
    monkeypatch.setattr(metrics, 'evaluate_rank', lambda *a, **k: (np.ones(50), np.float64(0.5)))

    class Sampler(object):
        def __init__(self, i):
            pass

        def start(self):
            pass

        def stop(self):
            return dict(sm_mhz=1700.0, sm_max_mhz=1965.0, reasons=['sw_power_cap'], samples=3, power_w=990.0)
    monkeypatch.setattr(bench, 'ClockSampler', Sampler)
    yield


def run(monkeypatch, capsys, model, argv=()):
    monkeypatch.setattr(bench, 'make_model', lambda dev, w: model)
    monkeypatch.setattr(bench.sys, 'argv', ['bench.py', '--steps', '2', '--no-e2e', '--no-cpu-baseline', '--no-eager', '--no-configs',
                                            '--no-parity', '--no-curve', '--no-energy'] + list(argv))
    bench.main()
    lines = [l for l in capsys.readouterr().out.splitlines() if l.strip()]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_b200_arm_line_and_extra_figures(fake_device, monkeypatch, capsys):
    model = FakeModel()
    line = run(monkeypatch, capsys, model)
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'roofline', 'kernel_table', 'gpu_launches', 'clocks', 'fast_mode'):
        assert key in line, key
    assert line['steps'] == 2 and line['warmup'] == 3 and line['n_gpus'] == 1 and line['clocks']['power_w'] == 990.0
    # the line's roofline is the WHOLE head against HBM (SURVEY 8d): J x 16 806 144 B / head time; FakeEvent makes a head pass 10 ms
    roof = line['roofline']
    assert roof['bound'] == 'hbm' and roof['unit'] == 'GB/s' and 'whole graph head' in roof['scope']
    J = bench.NQ + bench.NG
    assert abs(roof['achieved'] - J * bench.BYTES_PER_TRACKLET / 10e-3 / 1e9) < 1e-6 * roof['achieved']
    assert abs(roof['frac'] - roof['achieved'] / roof['peak']) < 1e-12
    assert roof['dominant_kernel']['kernel'] == 'pool' and roof['dominant_kernel']['bound'] == 'hbm'
    tab = line['kernel_table']
    assert tab['gemm_graph_layer']['bound'] == 'tensor' and tab['pool']['launches'] == 13 and tab['attn']['bound'] == 'hbm'
    assert abs(sum(r['share'] for r in tab.values()) - 1.0) < 1e-3
    assert 'head_ms' in line['fast_mode'] and 'head_hbm_frac' in line['fast_mode']
    # what the head was called with: default, fp16 plane -- and the last pass is in the default configuration again
    states = set(c[0] for c in model.calls)
    assert states == {_lib.SPLIT_BF16X2, _lib.SPLIT_FP16X1}
    assert model.calls[-1][0] == _lib.SPLIT_BF16X2 and model.head_split == _lib.SPLIT_BF16X2


def test_a_failing_extra_figure_does_not_cost_the_line(fake_device, monkeypatch, capsys):
    model = FakeModel(fail_when=lambda st: st[0] == _lib.SPLIT_FP16X1)            # the fp16 plane mode raises
    line = run(monkeypatch, capsys, model)
    assert 'injected failure' in line['fast_mode']['unavailable']
    assert line['value'] > 0 and line['roofline']['frac'] > 0
    assert model.head_split == _lib.SPLIT_BF16X2


class CallCountingModel(FakeModel):
    """Feature row i of the c-th head call (from 0) holds 1000 * c + i: a dumped row names the call that wrote it."""

    def head(self, x1, x2, adj, S, out=None):
        super().head(x1, x2, adj, S, out=out)
        c = len(self.calls) - 1
        out.copy_((1000 * c + torch.arange(out.shape[0], dtype=out.dtype))[:, None].expand_as(out))
        return out


def test_dump_outputs_writes_the_last_timed_step(fake_device, monkeypatch, capsys, tmp_path):
    evals = []

    def evaluate_rank(*a, **k):                                     # the n-th evaluation (from 1) returns cmc = mAP = n
        evals.append(None)
        return np.full(50, float(len(evals))), np.float64(len(evals))
    monkeypatch.setattr(metrics, 'evaluate_rank', evaluate_rank)
    line = run(monkeypatch, capsys, CallCountingModel(), ['--dump-outputs', str(tmp_path)])
    warmup, steps, pool, J = line['warmup'], line['steps'], line['config']['pool_tracklets'], bench.NQ + bench.NG
    assert (warmup, steps) == (3, 2) and len(evals) > warmup + steps            # evaluations also ran after the timed steps
    assert sorted(p.name for p in tmp_path.iterdir()) == ['cmc.npy', 'features.npy', 'mAP.npy']
    d = {k: np.load(str(tmp_path / (k + '.npy'))) for k in ('features', 'cmc', 'mAP')}
    assert d['features'].dtype == np.float32 and d['cmc'].dtype == np.float64 and d['mAP'].dtype == np.float64
    assert d['cmc'].shape == (50,) and d['mAP'].shape == ()
    assert np.all(d['cmc'] == warmup + steps) and float(d['mAP']) == warmup + steps     # the last timed evaluation
    # the fixed seeded row sample, each row as the last timed head pass wrote it
    rows = np.sort(np.random.RandomState(0).choice(J, bench.DUMP_FEATURE_ROWS, replace=False))
    calls_per_pass = -(-J // pool)
    want = 1000 * ((warmup + steps - 1) * calls_per_pass + rows // pool) + rows % pool
    f = d['features']
    assert f.shape == (bench.DUMP_FEATURE_ROWS, 2 * bench.C) and np.all(f == f[:, :1])
    assert np.array_equal(f[:, 0], want.astype(np.float32))
    assert sum(a.nbytes for a in d.values()) <= 64 << 20


@pytest.mark.parametrize('argv', [['--steps', '0'], ['--impl', 'reference', '--dump-outputs', 'x'],
                                  ['--workload', 'sweep', '--dump-outputs', 'x']])
def test_rejected_arguments(monkeypatch, argv):
    monkeypatch.setattr(bench.sys, 'argv', ['bench.py'] + argv)
    with pytest.raises(SystemExit):
        bench.main()


def test_reference_arm_line_reports_what_it_executed(monkeypatch, capsys):
    """--impl reference: same metric / unit / workload string as the B200 arm, the executed step time as ms_per_step, the
    extrapolation flagged (tiny sample here so that the CPU suite stays fast)."""
    monkeypatch.setattr(bench, 'NQ', 40); monkeypatch.setattr(bench, 'NG', 300)
    monkeypatch.setattr(bench, 'make_labels', lambda r, w: bench_labels())
    monkeypatch.setattr(bench.sys, 'argv', ['bench.py', '--impl', 'reference', '--steps', '2', '--warmup', '1', '--cpu-head-sample', '2'])
    bench.main()
    lines = [l for l in capsys.readouterr().out.splitlines() if l.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line['impl'] == 'reference' and line['metric'] == bench.METRIC and line['unit'] == 'tracklets/s'
    assert line['config']['workload'] == bench.WORKLOAD % 'euclidean'
    assert line['extrapolated'] is True and line['cpu_baseline']['steps_executed'] == 2 and line['cpu_baseline']['kind'] == 'port'
    assert abs(line['ms_per_step'] - line['cpu_baseline']['executed_step_ms']) < 1e-9
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['cpu_baseline']['cores'] >= 1
    assert line['value'] == line['cpu_baseline']['value'] == line['e2e']['value']


def bench_labels():
    from agrl.pytorch_b200 import synthetic as synth
    return synth.eval_labels((40, 300, 12, 3), seed=6)
