# Evidence captures at the current kernel sources (run on the GPU box through gpurun, ONE call):
#   launch list of the default bench command, and one `ncu --set full` capture per workload, exported to raw CSV on
#   the box (the .ncu-rep files together exceed gpurun's 64 MiB return limit; only the products one comes back).
# Read here with tools/ncu_summarise.py -> profiles/r02_ncu_<workload>.json (stamped with the kernel-source hash).
set -x
O=gpurun_out
T=/tmp/ncu_reps
mkdir -p $T
B="python bench.py --steps 2 --warmup 3 --no-also --no-cpu-baseline --sustain-seconds 0.02"
$B > $O/r02_plain_reddit.log 2>&1 && ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $O/r02_launches_reddit_k256.csv $B > $O/r02_ncu_launches.log 2>&1
cap() {  # name, kernel regex, skip, count, bench args...
  name=$1; rx=$2; skip=$3; cnt=$4; shift 4
  python bench.py --steps 2 --warmup 3 --no-also --no-cpu-baseline --sustain-seconds 0.02 "$@" > $O/r02_plain_$name.log 2>&1 && \
  ncu --set full --clock-control none -k regex:$rx -s $skip -c $cnt -f -o $T/r02_prof_$name python bench.py --steps 2 --warmup 3 --no-also --no-cpu-baseline --sustain-seconds 0.02 "$@" > $O/r02_ncu_$name.log 2>&1
  ncu -i $T/r02_prof_$name.ncu-rep --page raw --csv > $O/r02_raw_$name.csv 2>> $O/r02_ncu_$name.log
}
cap reddit_k256 spmm_kernel 20 5
cap products_k256 spmm_kernel 4 1 --workload products_k256
cap arxiv_k256 spmm_kernel 4 1 --workload arxiv_k256
cap arxiv_k32 spmm_kernel 4 1 --workload arxiv_k32
cp $T/r02_prof_products_k256.ncu-rep $O/
ls -la $O | tail -20
