"""Host-side checks of the measurement tooling (no GPU): the algorithmic work bench.py divides by, the ncu launch-list
condenser behind roofline.traffic, and the bench line's config for both BASELINE image sizes."""
import importlib
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))


@pytest.fixture()
def bench():
    sys.path.insert(0, ROOT)
    mod = importlib.import_module('bench')
    old = (mod.IMAGE_SIZE, mod.BATCH_PER_GPU)
    yield mod
    mod.IMAGE_SIZE, mod.BATCH_PER_GPU = old


def test_algorithmic_flops_match_survey(bench):
    """SURVEY 8(d): 29.936 GFLOP/img at 416^2 and 63.947 at 608^2 (output_filter 125); per-layer table entries."""
    total, per = bench.conv_flops_per_image(416, 125)
    assert len(per) == 22
    assert abs(total / 1e9 - 29.936) < 2e-3
    assert abs(per[0] / 1e9 - 0.299) < 1e-3 and abs(per[18] / 1e9 - 3.190) < 1e-3 and abs(per[21] / 1e9 - 0.043) < 1e-3
    total608, _ = bench.conv_flops_per_image(608, 125)
    assert abs(total608 / 1e9 - 63.947) < 5e-3


def test_bench_config_follows_image_size(bench):
    cfg = bench.make_config(2)
    assert cfg['precision'] == 'bf16' and bench.make_config(1, 'bf16x3')['precision'] == 'bf16x3'
    assert cfg['image_size'] == 416 and cfg['global_batch'] == 128 and 'configs[1]' in cfg['workload']
    bench.IMAGE_SIZE, bench.BATCH_PER_GPU = 608, 32
    cfg = bench.make_config(1)
    assert cfg['image_size'] == 608 and cfg['global_batch'] == 32 and '608x608' in cfg['workload'] and 'configs[3]' in cfg['workload']


def test_dump_outputs_dtypes_and_size_cap(bench, tmp_path, monkeypatch):
    """--dump-outputs: float arrays as float32, integer ones as float64; past the cap the same seeded rows of every array."""
    import numpy as np
    import torch
    eng = type('Eng', (), {})()
    eng.net_out = torch.randn(6, 2, 2, 25)
    eng.boxes, eng.scores = torch.rand(6, 20, 4), torch.rand(6, 20, 20)
    eng.keep_idx = torch.randint(0, 20, (6, 20, 4), dtype=torch.int32)
    eng.keep_count = torch.randint(-1, 6, (6, 20), dtype=torch.int32)
    out = bench.engine_outputs(eng)
    kc = eng.keep_count.numpy()
    for j in range(4):
        assert np.array_equal(out['keep_idx'][..., j] == -1, kc <= j)
    bench.dump_outputs(str(tmp_path / 'all'), out)
    got = {k: np.load(str(tmp_path / 'all' / (k + '.npy'))) for k in out}
    assert got['net'].dtype == np.float32 and got['keep_idx'].dtype == np.float64
    assert np.array_equal(got['net'], eng.net_out.numpy()) and np.array_equal(got['keep_count'], kc)
    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', 10000)     # 18720 bytes in all
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), out)
    files = sorted(os.listdir(str(tmp_path / 'a')))
    assert files == sorted(k + '.npy' for k in list(out) + ['sampled_rows']) and files == sorted(os.listdir(str(tmp_path / 'b')))
    rows = np.load(str(tmp_path / 'a' / 'sampled_rows.npy')).astype(int)
    assert 0 < len(rows) < 6 and sum(os.path.getsize(str(tmp_path / 'a' / f)) - 128 for f in files) <= 10000
    for f in files:
        assert np.array_equal(np.load(str(tmp_path / 'a' / f)), np.load(str(tmp_path / 'b' / f)))
    assert np.array_equal(np.load(str(tmp_path / 'a' / 'scores.npy')), eng.scores.numpy()[rows])


def test_launch_list_condenser(tmp_path):
    """tools/ncu_launch_list.py: one step = flush memset .. next flush memset; conv DRAM bytes and share of the step."""
    hdr = '"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Device","CC","Section Name","Metric Name","Metric Unit","Metric Value"'
    rows = [hdr]

    def launch(i, name, ns, rd, wr):
        for metric, unit, val in (('dram__bytes_read.sum', 'byte', rd), ('dram__bytes_write.sum', 'byte', wr),
                                  ('gpu__time_duration.sum', 'ns', ns)):
            rows.append('"%d","1","python","h","%s","1","7","(1, 1, 1)","(1, 1, 1)","0","10.0","s","%s","%s","%s"'
                        % (i, name, metric, unit, val))
    flush = 'void at::native::vectorized_elementwise_kernel<4, at::native::FillFunctor<unsigned char>, std::array<char *, 1>>(int, T2, T3)'
    launch(0, 'void y2::conv_tc_kernel<256, 0, 2, 0, 0>(CUtensorMap_st, CUtensorMap_st, CUtensorMap_st, y2::ConvArgs)', 5000, 1, 1)
    launch(1, flush, 70000, 0, 10)
    launch(2, 'y2::conv1_u8_pool_kernel(CUtensorMap_st, y2::C1Args)', 100000, 1000, 2000)
    launch(3, 'void y2::conv_streamk2_kernel<1>(CUtensorMap_st, CUtensorMap_st, y2::SkArgs)', 300000, 3000, 4000)
    launch(4, 'void y2::detect_fused_kernel<20>(const float *, const float *, int)', 100000, 5, 5)
    launch(5, flush, 70000, 0, 10)
    src = tmp_path / 'l.csv'
    src.write_text('==PROF== noise line\n' + '\n'.join(rows) + '\n')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'ncu_launch_list.py'), str(src), str(tmp_path / 'x')],
                         capture_output=True, text=True, check=True).stdout
    d = json.loads(out)
    assert d['conv_launches_per_step'] == 2 and d['launches_per_step'] == 3
    assert d['conv_dram_bytes_per_step'] == 1000 + 2000 + 3000 + 4000
    assert abs(d['conv_share_of_step_under_ncu'] - 0.8) < 1e-9
    assert d['precision'] == 'bf16'
    step = (tmp_path / 'x_launches_bench_step_bf16.csv').read_text().splitlines()
    assert step[0].startswith('id,kernel') and len(step) == 1 + 5
    assert '"conv_streamk2_kernel<1>"' in step[3]
