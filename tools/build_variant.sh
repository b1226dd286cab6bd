# usage: bash tools/build_variant.sh NAME   -> variants/lib_NAME.so, built from the sources as they are in the tree
# (e.g. a parent commit's, for an A/B run that selects the library with GNX_B200_LIB)
N=$1
mkdir -p variants
cd geonomics_b200/csrc && nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -shared gnx_api.cu -o ../../variants/lib_$N.so 2>&1 | grep -v "warning #177\|^$\|cur = c->cur\|\^\|Remark"
