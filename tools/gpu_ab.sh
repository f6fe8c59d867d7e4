# A/B timing of other builds of the library (variants/<name>/libKMCUDA.so, e.g. built at another commit);
# optional: "ncu" = one ncu --set full capture of the product kernel, "tests" = the GPU test suite
mkdir -p gpurun_out
export PATH=/usr/local/cuda/bin:$PATH
LIBS="product=kmcuda_b200/libKMCUDA.so"
for d in variants/*/; do n=$(basename $d); [ -f $d/libKMCUDA.so ] && LIBS="$LIBS $n=$d/libKMCUDA.so"; done
timeout 1200 python tests/ab_kernel.py $LIBS > gpurun_out/r2_ab.txt 2>&1
cut -c1-330 gpurun_out/r2_ab.txt
for a in "$@"; do
if [ "$a" = "ncu" ]; then
timeout 900 ncu --set full --clock-control none --import-source on -k regex:tc_assign_kernel -s 3 -c 1 -f -o gpurun_out/r02_tc_assign_v7 \
    python bench.py --steps 2 --warmup 3 --skip-extras > gpurun_out/r02_ncu_full.log 2>&1; echo "ncu full rc=$?"; tail -2 gpurun_out/r02_ncu_full.log
fi
if [ "$a" = "tests" ]; then
timeout 1500 python -m pytest tests -m gpu -q --tb=short -p no:cacheprovider -x > gpurun_out/r2_pytest.txt 2>&1; echo "pytest rc=$?"; tail -n 5 gpurun_out/r2_pytest.txt
fi
done
