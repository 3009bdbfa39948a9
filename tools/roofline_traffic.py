"""profiles/roofline_traffic_rNN.json from a per-launch ncu CSV (tools/gpu/r2_round_end.sh `layers*.csv`): average DRAM bytes and
duration per launch of the tcgen05 conv kernels (k_conv_umma + k_l1_chain + k_l2_chain), the `roofline.traffic` source of bench.py.
    python tools/roofline_traffic.py gpurun_out/layers.csv 5000 > profiles/roofline_traffic_r02.json"""
import csv, json, sys
path, stamps = sys.argv[1], int(sys.argv[2])
rows = [r for r in csv.reader(open(path)) if len(r) > 10 and r[0].isdigit()]
per = {}
for r in rows:
    per.setdefault(r[0], dict(name=r[4]))[r[12]] = float(r[14].replace(',', ''))
sel = [v for v in per.values() if any(k in v['name'] for k in ('k_conv_umma', 'k_l1_chain', 'k_l2_chain'))]
n = len(sel)
print(json.dumps(dict(kernel='k_conv_umma + k_l1_chain + k_l2_chain', launches=n, stamps_per_launch=stamps,
                      avg_traffic_bytes_per_launch=sum(v['dram__bytes_read.sum'] + v['dram__bytes_write.sum'] for v in sel) / n,
                      avg_us_per_launch=sum(v['gpu__time_duration.sum'] for v in sel) / n / 1e3,
                      source='ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum over %d consecutive tcgen05 conv launches, '
                             'bench.py --stamps %d (%s)' % (n, stamps, path)), indent=1))
