#!/bin/bash
# developer A/B builds of libvgl_b200 with extra -D flags: scripts/dev_build_variant.sh <name> <flags...> -> dev/lib_<name>.so
set -e
name=$1; shift
cd "$(dirname "$0")/.."
mkdir -p dev/obj_$name
for f in vectorgraphlibrary_b200/csrc/*.cu; do
  o=dev/obj_$name/$(basename ${f%.cu}).o
  if [ "$(basename $f)" = "pagerank.cu" ] || [ "$(basename $f)" = "pagerank_bins.cu" ] || [ "$(basename $f)" = "sssp.cu" ] || [ ! -f $o ]; then
    nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo --expt-relaxed-constexpr --extended-lambda -Xcompiler -fPIC,-O2,-fopenmp -I include -I vectorgraphlibrary_b200/csrc "$@" -c $f -o $o &
  fi
done
wait
nvcc -shared -o dev/lib_$name.so dev/obj_$name/*.o -Xcompiler -fopenmp -lcudart_static -ldl -lrt -lpthread
echo dev/lib_$name.so
