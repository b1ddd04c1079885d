#!/bin/bash
# builds tools/pbs_bench (extra nvcc flags as arguments) and prints the register/spill summary per kernel
cd "$(dirname "$0")"
OUT=${OUT:-pbs_bench}
nvcc -O3 -std=c++17 -lineinfo -gencode arch=compute_100a,code=sm_100a -I../tfhe-aes-2_b200/csrc -Xptxas -v "$@" -o $OUT pbs_bench.cu 2> build_bench.log || { tail -30 build_bench.log; exit 1; }
grep -E "Compiling entry.*pbs_[a-z_]*kernel|registers|spill" build_bench.log | grep -A2 "kernelILi512" | grep -v "^--" | paste - - - | sed -E 's/.*tac[0-9]+(pbs_[a-z_]*kernel)ILi512ELi4ELi3E([LiE0-9]+)EEvPKm.* ([0-9]+) bytes stack frame, ([0-9]+) bytes spill stores, ([0-9]+) bytes spill loads.*Used ([0-9]+) registers.*/\1<\2> stack=\3 spill_st=\4 spill_ld=\5 regs=\6/; s/Li([0-9]+)E/\1,/g; s/,>/>/'
