# A/B of library builds on the remap kernel inside one box: usage r2_remap_ab.sh <name>...
# Each <name> is a library directory 3dscan_b200/lib_var_<name>; build one from another commit by running
#   SCAN3D_LIBDIR=$PWD/3dscan_b200/lib_var_<name> python 3dscan_b200/build.py
# in a checkout of that commit, and copy lib_var_<name> into this tree if that checkout is elsewhere.
D=gpurun_out/remap_ab; rm -rf $D; mkdir -p $D
for i in 1 2; do
timeout 200 python tools/bench_aux.py 2>/dev/null | grep "56-frame" > $D/cur_$i.json
for v in "$@"; do
SCAN3D_LIBDIR=$PWD/3dscan_b200/lib_var_$v timeout 200 python tools/bench_aux.py 2>/dev/null | grep "56-frame" > $D/${v}_$i.json
done
done
for f in $D/*.json; do echo "$f $(cut -c1-120 $f)"; done
