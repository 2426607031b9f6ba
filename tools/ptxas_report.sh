#!/bin/bash
# registers / spills of every trace_kernel variant: tools/ptxas_report.sh
cd "$(dirname "$0")/../optable_b200/csrc"
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xptxas -v -c -o /tmp/optb_$$.o optb.cu 2>&1 \
 | grep -E "error|Compiling entry|registers|spill" | paste - - - | sed -E 's/ptxas info\s+: //g' | grep -E "error|trace_kernel" \
 | sed -E 's/.*trace_kernelILb([01])ELb([01])ELi([012])ELb([01])ELb([01])E.*sm_100a.\s+/\1\2\3\4\5 /' | sed -E 's/bytes //g; s/cumulative stack size, //; s/used 1 barriers, //' | cut -c1-200
rm -f /tmp/optb_$$.o
