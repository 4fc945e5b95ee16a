#!/bin/bash
O=gpurun_out/s11; mkdir -p $O
python tools/phase_run.py 1 > $O/phases.log 2>&1
RB_WIDE_CTAS=1 python tools/phase_run.py 1 >> $O/phases.log 2>&1
cat $O/phases.log
