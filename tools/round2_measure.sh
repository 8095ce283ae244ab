# Round-2 measurement pass on the GPU box (outputs under gpurun_out/, prefix r2m).
# ncu reports are exported to raw CSV on the box: gpurun copies back at most 64 MiB.
T=r2m
python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/${T}_smoke.log 2>&1; echo smoke rc=$? >> gpurun_out/${T}_smoke.log
python bench.py > gpurun_out/${T}_bench.json 2> gpurun_out/${T}_bench.err
python bench.py --impl reference --steps 5 --warmup 1 > gpurun_out/${T}_ref.json 2> gpurun_out/${T}_ref.err
python bench.py --steps 2 --warmup 3 --no-extra --no-cpu --no-samplers > gpurun_out/${T}_short.json 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none -c 500 --csv --log-file gpurun_out/${T}_launches.csv python bench.py --steps 2 --warmup 3 --no-extra --no-cpu --no-samplers > gpurun_out/${T}_ncu_launch.log 2>&1
python tools/profile_kernels.py all down > gpurun_out/${T}_prof_plain.log 2>&1 && \
timeout 600 ncu --set full --clock-control none -k regex:'prune_small_kernel|down_walk_kernel|prune_dmma_kernel' -c 5 -f -o /tmp/${T}_c2c3 python tools/profile_kernels.py all > gpurun_out/${T}_ncu_full.log 2>&1
ncu -i /tmp/${T}_c2c3.ncu-rep --page raw --csv > gpurun_out/${T}_c2c3_raw.csv 2>/dev/null
timeout 300 ncu --set full --clock-control none -k regex:down_dmma_kernel --launch-skip 6 -c 1 -f -o /tmp/${T}_c3down python tools/profile_kernels.py c3 down > gpurun_out/${T}_ncu_down.log 2>&1
ncu -i /tmp/${T}_c3down.ncu-rep --page raw --csv > gpurun_out/${T}_c3down_raw.csv 2>/dev/null
timeout 300 ncu --set full --clock-control none -k regex:'down_leaf_scatter|expm_kernel' -c 2 -f -o /tmp/${T}_c3leaf python tools/c3_down_one.py > gpurun_out/${T}_ncu_leaf.log 2>&1
ncu -i /tmp/${T}_c3leaf.ncu-rep --page raw --csv > gpurun_out/${T}_c3leaf_raw.csv 2>/dev/null
timeout 300 ncu --set full --clock-control none -k regex:raoteh_kernel --launch-skip 2 -c 1 -f -o /tmp/${T}_c4 python tools/c4_one.py > gpurun_out/${T}_ncu_c4.log 2>&1
ncu -i /tmp/${T}_c4.ncu-rep --page raw --csv > gpurun_out/${T}_c4_raw.csv 2>/dev/null
tail -n 2 gpurun_out/${T}_smoke.log gpurun_out/${T}_ncu_full.log gpurun_out/${T}_ncu_down.log; ls -la gpurun_out | tail -15
