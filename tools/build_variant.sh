#!/bin/bash
# A/B builds of one kernel source with extra -D flags:
#   tools/build_variant.sh NAME SRC.cu -DFOO=1 ...   ->  disenlink_b200/_variants/lib_NAME.so
# (load with DL_LIB_PATH=disenlink_b200/_variants/lib_NAME.so; the other objects come from the regular build)
set -e
cd "$(dirname "$0")/.."
name=$1
python -m disenlink_b200.build --variant "$@"
grep -A2 "flILi8ELi16\|Li8, *Li16\|ILi8ELi16" disenlink_b200/_variants/${name}.ptxas.log | grep -E "spill|Used" | head -4
