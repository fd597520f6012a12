#!/bin/bash
# same-box A/B of solve-kernel builds: scripts/ab_lm.sh <target>:<lib1>,<lib2>,... ...  ("default" = in-tree libacm.so)
for rep in 1 2; do for grp in "$@"; do
  export TARGET=${grp%%:*}; specs=${grp#*:}
  for lib in ${specs//,/ }; do
    if [ "$lib" = default ]; then unset ACM_LIB_PATH; else export ACM_LIB_PATH=$PWD/build/ab/libacm_$lib.so; fi
    echo -n "rep$rep $lib: "; python scripts/lm_ab.py | tail -1
  done
done; done
