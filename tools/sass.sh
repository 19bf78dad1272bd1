#!/bin/bash
# usage: tools/sass.sh <obj-basename> <demangled-substring>   -> SASS of the first matching kernel (no encodings)
obj=$(dirname "$0")/../neighbour_feature_pooling_b200/build/$1.o
cuobjdump -sass $obj | awk -v pat="$2" '
/Function :/ { on = 0; cmd = "echo " $3 " | c++filt"; cmd | getline dm; close(cmd); if (index(dm, pat)) on = 1 }
on && !/^\s*\/\* 0x/ { sub(/\/\* 0x[0-9a-f]* \*\//, ""); print }'
