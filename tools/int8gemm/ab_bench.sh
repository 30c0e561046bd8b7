# A/B of the INT8 path against the FP64 DMMA kernels (VBMF_B200_GEMM=dmma): GPU suite, smoke, alternated bench lines,
# output comparison of c3 / c4 after 23 iterations.  Usage: bash tools/int8gemm/ab_bench.sh [OUTDIR]
O=${1:-int8_ab_out}
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/card2.txt 2>&1
python -c "import __graft_entry__ as g; g.build(); g.smoke(); print('SMOKE OK')" > $O/smoke.txt 2>&1
timeout 900 python -m pytest -m gpu -q -p no:cacheprovider tests > $O/pytest_gpu.txt 2>&1; echo "rc=$?" >> $O/pytest_gpu.txt
B="python bench.py --gpus 1 --steps 20 --warmup 3"
for w in c3 c3shard8 c4 c4full; do
  for r in 1 2; do
    timeout 600 $B --workload $w > $O/b_${w}_int8_$r.json 2>$O/b_${w}_int8_$r.err
    [ $w = c3 ] || [ $r = 1 ] && VBMF_B200_GEMM=dmma timeout 600 $B --workload $w > $O/b_${w}_dmma_$r.json 2>$O/b_${w}_dmma_$r.err
  done
done
timeout 600 $B --workload c3 > $O/b_c3_int8_3.json 2>$O/b_c3_int8_3.err
VBMF_B200_GEMM=dmma timeout 600 $B --workload c3 > $O/b_c3_dmma_3.json 2>$O/b_c3_dmma_3.err
for w in c3 c4; do
  timeout 600 $B --workload $w --dump-outputs /tmp/d_${w}_int8 > /dev/null 2>&1
  VBMF_B200_GEMM=dmma timeout 600 $B --workload $w --dump-outputs /tmp/d_${w}_dmma > /dev/null 2>&1
  python tools/int8gemm/compare_dumps.py /tmp/d_${w}_int8 /tmp/d_${w}_dmma > $O/dumpdiff_$w.json 2>&1
done
timeout 900 $B --workload c5 > $O/b_c5_int8_1.json 2>$O/b_c5_int8_1.err
rm -rf /tmp/d_c3_* /tmp/d_c4_*
tail -n 3 $O/pytest_gpu.txt $O/smoke.txt
