# A/B of library builds inside ONE box (box-to-box variance is ~3 %): usage  r2_ab.sh <name>...
# Each <name> is a library directory 3dscan_b200/lib_var_<name>; build one from another commit by running
#   SCAN3D_LIBDIR=$PWD/3dscan_b200/lib_var_<name> python 3dscan_b200/build.py
# in a checkout of that commit, and copy lib_var_<name> into this tree if that checkout is elsewhere.
D=gpurun_out/ab; rm -rf $D; mkdir -p $D
# AB_ARGS overrides the short single-context run, e.g. AB_ARGS="" for the driver-style default (1.4 s under the power cap)
B="python bench.py --no-e2e --no-cpu-baseline --no-rowshard ${AB_ARGS---steps 20 --batch 16 --contexts 1 --cta-limit 0}"
for i in 1 2 3; do
timeout 200 $B > $D/cur_$i.json 2>/dev/null
for v in "$@"; do
SCAN3D_LIBDIR=$PWD/3dscan_b200/lib_var_$v timeout 200 $B > $D/${v}_$i.json 2>/dev/null
done
done
python - <<'PY'
import glob, json
for f in sorted(glob.glob("gpurun_out/ab/*.json")):
    try:
        d = json.load(open(f))
        print(f"{f:45s} {d['roofline']['avg_launch_us']:8.1f} us/scan  frac {d['roofline']['frac']:.3f}  sm {d['clocks']['sm_mhz']} {d['clocks']['reasons']}")
    except Exception as e:
        print(f, "unreadable:", e)
PY
