"""Turn $OUT/prof_<cfg>.ncu-rep + launches_<cfg>.csv (written by scripts/gpu_profile.sh; OUT defaults to profile_out)
into the committed summaries under profiles/ (dev tool).
usage: python scripts/ncu_summarize.py <cfg> <tag>"""
import csv, json, os, subprocess, sys, collections
cfg, tag = sys.argv[1], sys.argv[2]
out_dir = os.environ.get('OUT', 'profile_out')
rep = os.path.join(out_dir, f'prof_{cfg}.ncu-rep')
raw = subprocess.run(['ncu', '-i', rep, '--page', 'raw', '--csv'], capture_output=True, text=True).stdout
rows = list(csv.reader(raw.splitlines()))
hdr, units, vals = rows[0], rows[1], rows[2:]
keep = ['Kernel Name', 'launch__grid_size', 'launch__block_size', 'launch__registers_per_thread', 'gpu__time_duration.sum',
        'dram__bytes_read.sum', 'dram__bytes_write.sum', 'gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed',
        'sm__throughput.avg.pct_of_peak_sustained_elapsed', 'sm__warps_active.avg.pct_of_peak_sustained_active',
        'smsp__inst_executed.sum', 'sm__cycles_elapsed.max', 'smsp__cycles_active.avg',
        'smsp__issue_active.avg.pct_of_peak_sustained_active', 'smsp__thread_inst_executed_per_inst_executed.ratio',
        'l1tex__t_sector_hit_rate.pct', 'lts__t_sector_hit_rate.pct', 'launch__waves_per_multiprocessor',
        'l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum', 'smsp__inst_executed_op_shared_st.sum']
out = [f'ncu --set full --clock-control none --import-source on -k regex:qs_step_kernel, workload {cfg}, tag {tag}',
       '(cold-cache, serialised replays: compare shares and counts, not absolute times)']
d = {}
for i, h in enumerate(hdr):
    if h in keep:
        out.append(f'{h} [{units[i]}] = {[v[i] for v in vals]}')
        d[h] = (units[i], vals[0][i])
os.makedirs('profiles', exist_ok=True)
open(f'profiles/{tag}_ncu_full_{cfg}.txt', 'w').write('\n'.join(out) + '\n')
def tobytes(u, v):
    v = float(v.replace(',', ''))
    return v * {'byte': 1, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}[u]
traffic = tobytes(*d['dram__bytes_read.sum']) + tobytes(*d['dram__bytes_write.sum'])
tj = 'profiles/r02_traffic.json'
t = json.load(open(tj)) if os.path.exists(tj) else {}
t[cfg] = {'dram_bytes_per_launch': traffic, 'source': f'profiles/{tag}_ncu_full_{cfg}.txt (ncu --set full, cache control all: cold caches)'}
json.dump(t, open(tj, 'w'), indent=1, sort_keys=True)
# launch list
lr = [r for r in csv.reader(open(os.path.join(out_dir, f'launches_{cfg}.csv'))) if len(r) > 5]
ki, vi = lr[0].index('Kernel Name'), lr[0].index('Metric Value')
per = collections.defaultdict(list)
for r in lr[1:]:
    try: per[r[ki]].append(float(r[vi].replace(',', '')))
    except ValueError: pass
tot = sum(sum(v) for v in per.values())
with open(f'profiles/{tag}_launches_{cfg}.txt', 'w') as f:
    f.write(f'ncu --metrics gpu__time_duration.sum --clock-control none -s 30 -c 200 python bench.py --config {cfg} --steps 150 --warmup 8 --no-graph\n')
    f.write('kernel, launches, mean ns, share of GPU time in the captured window\n')
    for k, v in sorted(per.items(), key=lambda kv: -sum(kv[1])):
        f.write(f'{k}, {len(v)}, {sum(v)/len(v):.0f}, {100*sum(v)/tot:.1f}%\n')
src = subprocess.run(['ncu', '-i', rep, '--page', 'source', '--csv', '--print-source', 'sass,cuda'], capture_output=True, text=True).stdout
open('/tmp/src_cur.csv', 'w').write(src)
hs = subprocess.run([sys.executable, 'scripts/ncu_hotspots.py', '/tmp/src_cur.csv', '30'], capture_output=True, text=True).stdout
open(f'profiles/{tag}_hotspots_{cfg}.txt', 'w').write(hs)
print(open(f'profiles/{tag}_ncu_full_{cfg}.txt').read()); print(open(f'profiles/{tag}_launches_{cfg}.txt').read()); print(hs[-900:])
