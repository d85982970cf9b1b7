#!/bin/bash
# Tuning builds of the K5 kernel: tools/variants/lib_k5_<NSTAGE>_<NWU>_<INBOXES>.so (every other object from the in-tree build).
set -e
cd "$(dirname "$0")/.."
mkdir -p tools/variants
# one object per source present: a stale object of a deleted source would define its symbols a second time
objs=""
for src in adapter4rec_b200/csrc/*.cu; do
  name=$(basename "$src" .cu)
  [ "$name" = adapter_rows_sm100 ] || objs="$objs adapter4rec_b200/build/$name.o"
done
for v in "$@"; do
  IFS=_ read ns nwu inb <<< "$v"
  nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 --extended-lambda -Xcompiler -fPIC -Xcompiler -fvisibility=hidden \
    -DA4R_K5_NSTAGE=$ns -DA4R_K5_NWU=$nwu -DA4R_K5_INBOXES=$inb -c adapter4rec_b200/csrc/adapter_rows_sm100.cu -o /tmp/k5_$v.o
  nvcc -shared -o tools/variants/lib_k5_$v.so $objs /tmp/k5_$v.o -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC -lcudart_static -ldl -lrt -lpthread
  echo built $v
done
