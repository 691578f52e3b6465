# Round evidence run (one gpurun call): full GPU test suite, smoke, bench (both arms + the stage-alone / 512-source
# configs), the ncu launch list of ONE pipeline pass restricted to the engine's kernels, and ncu --set full captures of
# every kernel class of that pass (exported to CSV on the box; the .ncu-rep files are dropped to stay under the 64 MiB
# return limit).   usage: bash scripts/gpu_evidence.sh <tag> [quick|ncu]     (outputs land in gpurun_out/<tag>_*)
TAG=${1:-r02}
O=gpurun_out
K='regex:conv_multi|conv_gemm|conv_pair|stem_conv|s2d_pack|pool_kernel|pool3x3s|layernorm|attention_mma|chanstats|gate_hidden|gate_out|bbox_kernel|resize_u8|head_kernel'
set -x
if [ "$2" != "ncu" ]; then
python -m pytest tests -m gpu -q -x --tb=short -p no:cacheprovider -rP > $O/${TAG}_gputests.log 2>&1; echo "pytest rc=$?"; tail -5 $O/${TAG}_gputests.log
python -c "import __graft_entry__ as g; g.smoke()" > $O/${TAG}_smoke.log 2>&1; echo "smoke rc=$?"; tail -2 $O/${TAG}_smoke.log
python bench.py --steps 20 --warmup 3 --breakdown $O/${TAG}_per_op.json > $O/${TAG}_bench.log 2>&1; echo "bench rc=$?"; tail -c 3800 $O/${TAG}_bench.log
fi
if [ "$2" != "quick" ] && [ "$2" != "ncu" ]; then
python bench.py --steps 20 --warmup 3 --no-cpu-baseline --no-yardstick --source-size 512 > $O/${TAG}_bench_src512.log 2>&1; tail -c 900 $O/${TAG}_bench_src512.log
python bench.py --workload unet --batch 64 --steps 20 > $O/${TAG}_bench_unet64.log 2>&1; tail -c 900 $O/${TAG}_bench_unet64.log
python bench.py --workload googlenet --steps 20 > $O/${TAG}_bench_googlenet256.log 2>&1; tail -c 700 $O/${TAG}_bench_googlenet256.log
python bench.py --impl reference --steps 2 --warmup 1 > $O/${TAG}_bench_ref.log 2>&1; tail -c 1200 $O/${TAG}_bench_ref.log
fi
# ---- ncu: one pass of the engine's kernels (the warm-up passes are skipped by counting ONLY matching kernels)
CMD="python scripts/one_pass.py --batch 128 --passes 3"
$CMD > $O/${TAG}_plain.log 2>&1 || { cat $O/${TAG}_plain.log; exit 1; }
L=$(grep LAUNCHES_PER_PASS $O/${TAG}_plain.log | awk '{print $2}'); echo "launches per pass: $L"
ncu --metrics gpu__time_duration.sum --clock-control none -k "$K" --launch-skip $((2 * L)) --launch-count $L --csv \
    --log-file $O/${TAG}_launches.csv $CMD > $O/${TAG}_ncu1.log 2>&1
echo "ncu launches rc=$?"
if grep -q elementwise_kernel $O/${TAG}_launches.csv; then echo "ERROR: torch kernels in the launch list"; fi
N=$(grep -c '^"' $O/${TAG}_launches.csv); echo "rows in the launch list (header + launches): $N"
if [ "$N" != "$((L + 1))" ]; then echo "ERROR: the kernel filter does not match every engine launch ($((N - 1)) of $L)"; fi
$CMD > $O/${TAG}_plain.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k "$K" --launch-skip $((2 * L)) --launch-count $L -o $O/${TAG}_full $CMD > $O/${TAG}_ncu2.log 2>&1
echo "ncu full rc=$?"
ncu -i $O/${TAG}_full.ncu-rep --page raw --csv > $O/${TAG}_full.raw.csv 2>/dev/null
ls -la $O/${TAG}_full.ncu-rep
rm -f $O/${TAG}_full.ncu-rep
ls -la $O | tail -14
