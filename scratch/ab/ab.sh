#!/bin/bash
# A/B of two builds of the library on the same GPU (measurement script): build the two versions with
# `python -m curious_b200.build`, copy curious_b200/libcurious_b200.so to scratch/ab/lib_head.so / scratch/ab/lib_new.so
# (git-ignored), then run ./scratch/ab/ab.sh from the repository root on the GPU machine (env B = batch rows)
for rep in 1 2 3; do
  for v in head new; do
    cp scratch/ab/lib_$v.so curious_b200/libcurious_b200.so
    echo -n "$v: "; B=${B:-256} timeout 120 python scratch/ddpg_bench.py 2>&1 | tail -1
  done
done
cp scratch/ab/lib_new.so curious_b200/libcurious_b200.so
