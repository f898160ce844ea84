#!/bin/bash
# End-of-round evidence of HEAD (compiled-in defaults): tools/gpu_check.sh (smoke, -m gpu suite, full bench line), tools/gpu_profile.sh
# (launch lists of a KITTI and a dense step, ncu --set full of a 128-frame step with per-line tables), and the launch list of ONE
# one-frame call in reference order (the drop-in class's call pattern). Everything lands in gpurun_out/.
cd "${GRAFT_REPO_ROOT:-$(dirname "$0")/..}" || exit 1
mkdir -p gpurun_out
bash tools/gpu_check.sh 2>&1 | tee gpurun_out/check.log
[ -n "$SKIP_DENSE_FULL" ] && sed -i 's/^timeout 420 ncu --set full --clock-control none --import-source on -k regex:k_ -s \$SKIPD.*$/echo skip-dense-full/' tools/gpu_profile.sh
bash tools/gpu_profile.sh 2>&1 | tee gpurun_out/profile.log | tail -40
cat > /tmp/one_frame.py <<'PY'
import os, sys
REPO = os.getcwd()   # the repository root (cd above)
sys.path[:0] = [os.path.join(REPO, "patchwork-plusplus_b200"), os.path.join(REPO, "tests")]
import pwpp_b200
from conftest import load_kitti
a = load_kitti(0)
eng = pwpp_b200.Engine(device=0, num_streams=1); eng.set_output_order(1)
for _ in range(6):
    eng.estimate_host([a])
eng.close()
PY
PWPP_GRAPH=0 timeout 200 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:k_ --csv --log-file gpurun_out/r02_launches_one_frame.csv python /tmp/one_frame.py > /dev/null 2>&1
python - <<'PY'
import csv
rows = [r for r in csv.reader(open("gpurun_out/r02_launches_one_frame.csv")) if len(r) > 5 and r[0].isdigit()]
names = [r[4].split("(")[0] for r in rows]
starts = [i for i, n in enumerate(names) if n == names[0]]
last = rows[starts[-1]:]
print("one-frame call, reference order:", len(last), "launches,", round(sum(float(r[-1]) for r in last) / 1e3, 1), "us in total (serialised)")
for r in last:
    print("   ", r[4].split("(")[0][:50], r[7], r[8], round(float(r[-1]) / 1e3, 1), "us")
PY
