#!/bin/bash
# registers / spills / stack of the k_run instantiations the benchmarks launch (ptxas -v); no GPU needed.  The last pattern:
# every instantiation for more than 64 trains (NW = 2: learn / greedy / full at 8, 16 and 32 lanes).  Then every k_eval
# instantiation (the greedy kernel of evaluation contexts: one-word maps at 1-32 lanes, TH and ONE, and NW = 2 at 8, 16, 32).
cd "$(dirname "$0")/.."
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -shared -Xptxas -v -I include \
  -o /tmp/sfl_ptxas.so network-distributed-q-learning_b200/csrc/sfl_api.cu 2>&1 | \
  awk '/Compiling entry function/ {name=$0} /Used [0-9]+ registers/ {print name; print prev; print $0} {prev=$0}' | \
  grep -A2 -E "k_runILi32ELi0ELb0ELb0ELb0ELb0ELi1E|k_runILi32ELi0ELb0ELb0ELb0ELb1ELi1E|k_runILi16ELi0ELb1ELb0ELb1ELb0ELi1E|k_runILi16ELi0ELb0ELb0ELb1ELb1ELi1E|k_runILi32ELi0ELb0ELb1ELb0ELb0ELi1E|k_runILi32ELi2ELb0ELb0ELb0ELb0ELi1E|k_runILi(8|16|32)ELi[012]ELb0ELb0ELb0ELb0ELi2E|k_evalILi" | \
  sed -e 's/ptxas info    : //' -e "s/Compiling entry function '_ZN.*k_run/k_run/" -e "s/Compiling entry function '_Z6k_eval/k_eval/" -e "s/' for 'sm_100a'//"
