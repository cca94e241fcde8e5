#!/bin/bash
# Turn the raw outputs of profiles/make_rNN.sh (gpurun_out/) into the committed summaries.  usage: refresh.sh r02
set -e
R=${1:-r02}
python profiles/ncu_summary.py gpurun_out/${R}_step_kernel.ncu-rep > profiles/${R}_step_kernel_ncu_summary.txt
python profiles/ncu_summary.py gpurun_out/${R}_step_kernel_fused.ncu-rep > profiles/${R}_step_kernel_fused_ncu_summary.txt
python - "$R" <<'PY'
import json, csv, subprocess, sys
R = sys.argv[1]
def traffic(rep, out, steps, what, note):
    txt = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(txt.splitlines())); hdr = rows[0]; units = rows[1]
    def val(r, k):
        i = hdr.index(k)
        return float(r[i]) * {'Mbyte': 1e6, 'Kbyte': 1e3, 'byte': 1, 'Gbyte': 1e9}.get(units[i], 1)
    launches = [dict(us=float(r[hdr.index('gpu__time_duration.sum')]), dram_read=val(r, 'dram__bytes_read.sum'),
                     dram_write=val(r, 'dram__bytes_write.sum'), inst=float(r[hdr.index('smsp__inst_executed.sum')])) for r in rows[2:]]
    mean = sum(l['dram_read'] + l['dram_write'] for l in launches) / len(launches)
    json.dump(dict(source=f"ncu --set full --clock-control none, profiles/make_{R}.sh, report {rep} ({what})", envs_per_launch=65536,
                   device_slots=100, steps_per_launch=steps, dram_bytes_per_launch=mean, launches=launches, note=note), open(out, 'w'), indent=1)
traffic(f"gpurun_out/{R}_step_kernel.ncu-rep", f"profiles/{R}_step_kernel_traffic.json", 1, "first launch = defender turn, second = attacker turn",
        "dram write bytes of one captured launch are small because the 31.2 MB bulk store stays in the 126 MB L2 until evicted; "
        "algorithmic bytes per launch = 67.4 MB, record traffic = 2 x 31.2 MB")
traffic(f"gpurun_out/{R}_step_kernel_fused.ncu-rep", f"profiles/{R}_step_kernel_fused_traffic.json", 4, "two launches of 4 fused plain steps each",
        "4 steps per launch: the 31.2 MB record span is read once and written once per launch (writes of one captured launch mostly stay in "
        "L2), plus 4 x 2 MB of action rows; algorithmic bytes per launch = 4 x 67.4 MB")
PY
for k in 1 2; do ncu -i gpurun_out/${R}_step_kernel.ncu-rep --page source --csv --print-source cuda,sass --kernel-id :::$k 2>/dev/null > gpurun_out/src_${R}_$k.csv; done
python profiles/ncu_lines.py gpurun_out/src_${R}_1.csv 25 > profiles/${R}_step_kernel_defender_lines.txt 2>/dev/null || true
python profiles/ncu_lines.py gpurun_out/src_${R}_2.csv 25 > profiles/${R}_step_kernel_attacker_lines.txt 2>/dev/null || true
tail -1 gpurun_out/${R}_bench.json > profiles/${R}_bench_line.json
cp gpurun_out/${R}_launches.csv profiles/${R}_launches.csv
[ -f gpurun_out/${R}_exclude_sweep.txt ] && cp gpurun_out/${R}_exclude_sweep.txt profiles/${R}_exclude_sweep.txt
# SASS evidence: bulk (TMA) copies + mbarrier waits in the step kernel, instruction count of the plain instantiation
SASS=$(cuobjdump -sass -fun '_Z15cyg_step_kernelILi4ELb0ELb0ELb0EEv10StepParams' cygym_b200/libcygym_b200.so 2>/dev/null || true)
{ echo "# cuobjdump -sass of cyg_step_kernel<4, no ROLL, no LOG> in cygym_b200/libcygym_b200.so (sm_100a)";
  echo "# SASS instructions: $(grep -cE '^\s+/\*[0-9a-f]{4,}\*/' <<< "$SASS")";
  echo "# bulk-copy / mbarrier / cluster instructions:"; grep -nE 'UBLKCP|UBLKPF|SYNCS|UTMA|FENCE|ELECT' <<< "$SASS" | sed 's/  */ /g' | head -40;
  echo "# opcode histogram (top 25):"; grep -oE '^\s+/\*[0-9a-f]{4,}\*/\s+(@!?U?P[0-9T] )?[A-Z0-9_.]+' <<< "$SASS" | awk '{print $NF}' | cut -d. -f1 | sort | uniq -c | sort -rn | head -25; } > profiles/${R}_step_kernel_sass.txt
ls -la profiles/${R}_*
