# usage: bash tools/build_variant.sh <name> <nvcc -D flags...>   -> flowhigh_b200/lib/libflowhigh_b200_<name>.so
# (select it with FLOWHIGH_B200_LIB=<path>; A/B of compile-time options inside one gpurun call)
name=$1; shift
cd "$(dirname "$0")/../flowhigh_b200" || exit 1
mkdir -p lib/obj_$name
for f in dsp backbone vocoder_f32 vocoder_tc tc_conv attention_tc5; do
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -fvisibility=hidden "$@" \
    -c csrc/$f.cu -o lib/obj_$name/$f.o &
done
wait
nvcc -shared -o lib/libflowhigh_b200_$name.so lib/obj_$name/*.o -gencode arch=compute_100a,code=sm_100a && echo lib/libflowhigh_b200_$name.so
