# the member-sum pass of the product build and of every variants/*/libKMCUDA.so at 8M and 1M rows
mkdir -p gpurun_out
export PATH=/usr/local/cuda/bin:$PATH
for n in 8000000 1000000; do
for lib in kmcuda_b200/libKMCUDA.so variants/*/libKMCUDA.so; do
KMCUDA_B200_LIB=$PWD/$lib timeout 120 python tools/sums_probe.py $n 2>&1 | grep SUMS | tee -a gpurun_out/r02_sums.txt
done; done
timeout 600 python -m pytest tests -m gpu -q --tb=short -p no:cacheprovider -k "member_sums or update" 2>&1 | tail -3
