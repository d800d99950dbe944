# Builds libecho_b200 with -DECHO_BOUNDS_CHECK (every scene-derived index and stack pointer checked, echo_scene.cuh ECHO_CHECK) into
# variants/lib_bounds.so. Run the GPU suite against it with:  ECHO_B200_LIBRARY=$PWD/variants/lib_bounds.so python -m pytest tests -m gpu
# PreparedScene.close() raises when a check failed. (compute-sanitizer is not available on the GPU pool.)
set -e
cd "$(dirname "$0")/../echorenderer_b200/csrc"
out=/tmp/echo_bounds_build
rm -rf $out && mkdir -p $out
for f in api trace instanced build sweep lightbuild packbuild render debug peaks; do
  nvcc -std=c++17 -O3 -gencode arch=compute_100a,code=sm_100a -lineinfo -fmad=false -Xcompiler -fPIC -DECHO_BOUNDS_CHECK -c $f.cu -o $out/$f.o &
done
wait
nvcc -shared -o ../../variants/lib_bounds.so $out/*.o -gencode arch=compute_100a,code=sm_100a
ls -la ../../variants/lib_bounds.so
