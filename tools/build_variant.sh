#!/bin/bash
# Builds an A/B variant of libsso_b200.so: recompiles the listed curve translation units and the field probe (the test-only
# kernels of sso_test_field_op, tests/test_field_conformance.py) with extra -D flags and links them with the base build's other
# objects.   tools/build_variant.sh NAME "FLAGS" [curve ...]   (default curve: bls12_377)
# Result: snark-setup-operator_b200/variants/libsso_b200_NAME.so (select with SSO_B200_LIB=... ; see tools/gpu_kernel_ab.py)
set -e
NAME=$1; FLAGS=$2; shift 2 || true
CURVES=${@:-bls12_377}
ROOT=$(cd "$(dirname "$0")/.." && pwd)
CSRC=$ROOT/snark-setup-operator_b200/csrc
BASE=$ROOT/snark-setup-operator_b200/build
OUT=$ROOT/snark-setup-operator_b200/variants
mkdir -p $OUT/$NAME
OBJS="$BASE/abi.o"
for c in bls12_377 bw6_761 mnt4_753 mnt6_753; do
  if [[ " $CURVES " == *" $c "* ]]; then
    nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xptxas -v $FLAGS \
      -c $CSRC/curve_$c.cu -o $OUT/$NAME/curve_$c.o 2> $OUT/$NAME/curve_$c.ptxas.log || { tail -30 $OUT/$NAME/curve_$c.ptxas.log; exit 1; }
    OBJS="$OBJS $OUT/$NAME/curve_$c.o"
  else
    OBJS="$OBJS $BASE/curve_$c.o"
  fi
done
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xptxas -v $FLAGS \
  -c $CSRC/field_probe.cu -o $OUT/$NAME/field_probe.o 2> $OUT/$NAME/field_probe.ptxas.log || { tail -30 $OUT/$NAME/field_probe.ptxas.log; exit 1; }
OBJS="$OBJS $OUT/$NAME/field_probe.o"
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $OUT/libsso_b200_$NAME.so $OBJS
echo built $OUT/libsso_b200_$NAME.so
