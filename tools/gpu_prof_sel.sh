#!/bin/bash
# ncu full captures of the two seeded selection kernels at 4 M reads (after a plain run of the same command)
T=${1:-r2r}
mkdir -p gpurun_out
python tools/profile_step.py --method rmi --bounds --reads 4000000 --steps 1 > gpurun_out/${T}_plain.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:"k_select_seeded" -c 1 -o gpurun_out/${T}_rmi_sel python tools/profile_step.py --method rmi --bounds --reads 4000000 --steps 1 > gpurun_out/${T}_ncu1.log 2>&1; echo "ncu rmi exit=$?"
python tools/profile_step.py --method lut --reads 4000000 --steps 1 > gpurun_out/${T}_plain2.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:"k_select_seeded" -c 1 -o gpurun_out/${T}_lut_sel python tools/profile_step.py --method lut --reads 4000000 --steps 1 > gpurun_out/${T}_ncu2.log 2>&1; echo "ncu lut exit=$?"
