# Final evidence of round 2 in one run: GPU test suite, the plain bench (default run + reference arm), per-stage
# timings, the odometry loop, then the ncu passes (launch list of the same bench command, --set full of every hot
# kernel).  usage: bash tools/collect_final_r2.sh <tag>.  (The round-2 run also ran the original project's own test
# binaries, profiles/r2_reference_test_*; their sources are not part of this repository and nothing builds them now.)
T=${1:-r2f}
python -m pytest tests -q -m gpu > gpurun_out/${T}_gpu_tests.txt 2>&1; echo "gpu tests rc=$?"; tail -n 3 gpurun_out/${T}_gpu_tests.txt
python tools/run_odometry.py 45 > gpurun_out/${T}_odometry.txt 2>&1; tail -n 5 gpurun_out/${T}_odometry.txt
python tools/cfg4_diag.py 2,5,20,40 > gpurun_out/${T}_cfg4_diag.txt 2>&1; grep iterations gpurun_out/${T}_cfg4_diag.txt | cut -c1-120
bash tools/collect_profiles_r2.sh $T > gpurun_out/${T}_collect.log 2>&1
ncu --metrics gpu__time_duration.sum --clock-control none -k regex:"icp_keep|icp_fast|icp_coop|linearize" -c 200 --csv --log-file gpurun_out/${T}_cfg4_launches.csv python tools/cfg4_diag.py 12 > /dev/null 2>&1
python - <<PY
import csv
rows = [r for r in csv.reader(open("gpurun_out/${T}_cfg4_launches.csv")) if len(r) > 10 and r[0].isdigit()]
with open("gpurun_out/${T}_cfg4_launches.txt", "w") as f:
    f.write("config 4 (1.64 M x 1.54 M, GICP), second 12-iteration align: ncu --metrics gpu__time_duration.sum --clock-control none (cold-cache, serialised launches)\n")
    for r in rows[-47:]:
        f.write(f"{r[4][:60]:60s} {int(float(r[-1])) / 1e3:9.1f} us\n")
PY
bash tools/collect_ncu_full_r2.sh $T > gpurun_out/${T}_collect_full.log 2>&1
python - <<PY
import json
d = json.loads(open("gpurun_out/${T}_bench.json").read().strip().splitlines()[-1])
print("bench value", d["value"], "e2e", d["e2e"]["value"], "ms/iter", d["ms_per_iter"], "frac", d["roofline"]["frac"], "cpu", d.get("cpu_baseline", {}).get("value"))
print({k: (v.get("mqueries_per_s") or v.get("pairs_per_s") or v.get("GICP", {}).get("ms_per_iter")) for k, v in d.get("extras", {}).items() if isinstance(v, dict)})
PY
