# tick-budget sweep: request cap (whole net-kernel rounds) x level budget of the tree kernel
set -x
mkdir -p gpurun_out
{
timeout -k 10 200 python tools/tick_timing.py 2048 800 1024
for L in 16 24 32; do AZ_REQ_CAP=1184 AZ_LEVELS_PER_TICK=$L timeout -k 10 200 python tools/tick_timing.py 2048 800 1536; done
AZ_REQ_CAP=1184 timeout -k 10 200 python tools/tick_timing.py 2048 800 1536
} > gpurun_out/sweep_tick.log 2>&1
grep -v "^+" gpurun_out/sweep_tick.log
