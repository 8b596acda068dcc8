#!/usr/bin/env python
"""Summaries of ncu outputs for profiles/ (run in the dev container, no GPU needed).

  python scripts/summarize_ncu.py launches gpurun_out/launches.csv          > profiles/rNN_launches.md
  python scripts/summarize_ncu.py report   gpurun_out/prof.ncu-rep [regex]  > profiles/rNN_<kernel>.md
"""
import csv
import io
import re
import subprocess
import sys
from collections import OrderedDict

KEYS = ['gpu__time_duration.sum', 'dram__bytes_read.sum', 'dram__bytes_write.sum', 'dram__throughput.avg.pct_of_peak_sustained_elapsed',
        'gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed', 'sm__throughput.avg.pct_of_peak_sustained_elapsed',
        'sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active', 'sm__pipe_tensor_subpipe_hmma_cycles_active.avg.pct_of_peak_sustained_active',
        'sm__inst_executed_pipe_tensor.sum', 'sm__warps_active.avg.pct_of_peak_sustained_active', 'launch__registers_per_thread',
        'launch__shared_mem_per_block_dynamic', 'launch__grid_size', 'launch__block_size', 'lts__t_sector_hit_rate.pct',
        'l1tex__data_pipe_lsu_wavefronts_mem_shared.sum', 'smsp__cycles_active.avg', 'sm__cycles_elapsed.max',
        'sm__cycles_active.avg', 'l1tex__t_sector_hit_rate.pct', 'smsp__inst_executed.sum', 'dram__cycles_active.avg.pct_of_peak_sustained_elapsed']


def short(name):
    name = re.sub(r'\(.*', '', name)
    return name.replace('void ', '')


def launches(path):
    rows = []
    with open(path) as f:
        lines = [l for l in f if l.startswith('"')]
    for r in csv.DictReader(io.StringIO(''.join(lines))):
        if r.get('Metric Name') == 'gpu__time_duration.sum':
            v = float(r['Metric Value'].replace(',', ''))
            unit = r.get('Metric Unit', 'ns')
            v *= {'ns': 1e-3, 'us': 1.0, 'usecond': 1.0, 'ms': 1e3, 'msecond': 1e3, 'nsecond': 1e-3}.get(unit, 1e-3)
            rows.append((short(r['Kernel Name']), r['Grid Size'], r['Block Size'], v))
    agg = OrderedDict()
    for k, g, b, v in rows:
        a = agg.setdefault(k, [0, 0.0, g, b])
        a[0] += 1
        a[1] += v
    tot = sum(a[1] for a in agg.values())
    print('| kernel | launches | total us | mean us | share | grid | block |')
    print('|---|---|---|---|---|---|---|')
    for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        print('| `%s` | %d | %.1f | %.2f | %.1f%% | %s | %s |' % (k, a[0], a[1], a[1] / a[0], 100 * a[1] / tot, a[2], a[3]))
    print('\n%d launches, %.1f us total (ncu per-launch times are cold-cache and serialised: compare shares).' % (len(rows), tot))


def report(path, pattern=None):
    out = subprocess.run(['ncu', '-i', path, '--page', 'raw', '--csv'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                         text=True).stdout
    rd = list(csv.reader(io.StringIO(out)))
    hdr, units = rd[0], rd[1]
    for row in rd[2:]:
        d = dict(zip(hdr, row))
        if pattern and not re.search(pattern, d.get('Kernel Name', '')):
            continue
        print('### `%s`  grid %s block %s\n' % (short(d['Kernel Name']), d.get('Grid Size'), d.get('Block Size')))
        print('| metric | value | unit |')
        print('|---|---|---|')
        u = dict(zip(hdr, units))
        for k in KEYS:
            if k in d:
                print('| %s | %s | %s |' % (k, d[k], u.get(k, '')))
        print()


def traffic(path, samples_per_launch):
    """DRAM bytes per sample of each forward kernel class (ncu --set full capture of one chunk) as JSON."""
    import json
    out = subprocess.run(['ncu', '-i', path, '--page', 'raw', '--csv'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                         text=True).stdout
    rd = list(csv.reader(io.StringIO(out)))
    hdr, units = rd[0], rd[1]
    u = dict(zip(hdr, units))
    scale = {'byte': 1., 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
    res, nfc = {}, 0
    for row in rd[2:]:
        d = dict(zip(hdr, row))
        name = d['Kernel Name']
        cls = None
        m = re.search(r'Cfg<\(int\)(\d+), \(int\)\d+, \(int\)(\d+), \(int\)(\d+)', name) or \
            re.search(r'Cfg<(\d+), \d+, (\d+), (\d+)', name)
        if ('conv_tc_kernel' in name or 'conv_wt_kernel' in name) and m:
            cls = {('25', '3'): 'conv1', ('25', '16'): 'conv1', ('25', '24'): 'conv2', ('13', '32'): 'conv3', ('13', '48'): 'conv4'}.get((m.group(1), m.group(2)))
        elif 'fc_tc_kernel' in name or 'fc_tc_pair_kernel' in name:
            nfc += 1
            cls = 'fc%d' % nfc if nfc <= 2 else None
        elif 'gather_split_kernel' in name:
            cls = 'gather'
        elif 'pool_split_kernel' in name:
            cls = 'max1' if 'max1' not in res else 'max2'
        elif 'head_kernel' in name:
            cls = 'fc3'
        if cls is None or cls in res:
            continue
        rb = float(d['dram__bytes_read.sum']) * scale[u['dram__bytes_read.sum']]
        wb = float(d['dram__bytes_write.sum']) * scale[u['dram__bytes_write.sum']]
        res[cls] = {'dram_bytes_per_sample': (rb + wb) / samples_per_launch, 'dram_read_per_launch': rb,
                    'dram_write_per_launch': wb, 'samples_per_launch': samples_per_launch,
                    'duration_us': float(d['gpu__time_duration.sum']) * {'ns': 1e-3, 'us': 1., 'ms': 1e3, 's': 1e6}.get(
                        u['gpu__time_duration.sum'], 1.),
                    'tensor_pipe_pct': float(d.get('sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active', 'nan') or 'nan')}
    print(json.dumps(res, indent=1))


if __name__ == '__main__':
    if sys.argv[1] == 'launches':
        launches(sys.argv[2])
    elif sys.argv[1] == 'traffic':
        traffic(sys.argv[2], int(sys.argv[3]))
    else:
        report(sys.argv[2], sys.argv[3] if len(sys.argv) > 3 else None)
