# trace build of the library (per-role timelines, B2D_TRACE / B2D_TRACE_DUMP) -> tools/ubench/build/libb2det_trace.so
set -e
cd "$(dirname "$0")/../aerial_image_recognition_b200/csrc"
mkdir -p ../../tools/ubench/build/tr
for f in engine conv_tc pool preprocess postprocess dedup tta; do
  /usr/local/cuda/bin/nvcc -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -gencode arch=compute_100a,code=sm_100a -DB2D_ENABLE_TRACE -c $f.cu -o ../../tools/ubench/build/tr/$f.o &
done
wait
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o ../../tools/ubench/build/libb2det_trace.so ../../tools/ubench/build/tr/*.o -lcudart_static -ldl -lrt -lpthread
