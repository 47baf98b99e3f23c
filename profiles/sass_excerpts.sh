#!/bin/bash
# cuobjdump -sass evidence per hot kernel (what ptxas emitted for sm_100a), from the in-tree objects of android_svo_b200/build.sh:
#   profiles/r2_sass/<kernel>.txt = resource line from the ptxas log, opcode histogram, the SASS listing (offset + instruction)
# bash profiles/sass_excerpts.sh     (no GPU needed)
cd "$(dirname "$0")/.."
OUT=profiles/r2_sass
mkdir -p $OUT
dump() {  # object, function-name regex, output name
  local obj=$1 re=$2 name=$3
  cuobjdump -sass android_svo_b200/lib/$obj.o | awk -v re="$re" '/Function : /{f = ($0 ~ re)} f' > /tmp/sass_$name.txt
  {
    echo "# $name  (android_svo_b200/csrc/$obj.cu, sm_100a, nvcc 12.9, -O3 -fmad=false -lineinfo)"
    grep -A3 "Compiling entry function.*$re" android_svo_b200/lib/$obj.ptxas.log | grep -E "Used|spill" | sed 's/ptxas info    : /# /' | head -4
    echo "# opcode histogram (static instruction count)"
    grep -E "^\s+/\*[0-9a-f]{4,6}\*/" /tmp/sass_$name.txt | awk '{op=$2; if (op ~ /^@/) op=$3; sub(/;$/, "", op); print op}' | sort | uniq -c | sort -rn | head -40 | sed 's/^/#   /'
    echo "# SASS"
    grep -E "Function :|^\s+/\*[0-9a-f]{4,6}\*/" /tmp/sass_$name.txt | sed -E 's#\s+/\* 0x[0-9a-f]+ \*/##'
  } > $OUT/$name.txt
  echo "$name: $(grep -cE '^\s+/\*[0-9a-f]{4,6}\*/' /tmp/sass_$name.txt) instructions"
}
dump pyramid 'pyramid_fused_kernelILb0ELi4' pyramid_fused_kernel
dump fast 'fast_kernel' fast_kernel
dump sparse_align 'sparse_align_kernelILi128ELi1' sparse_align_kernel_128_1
dump matcher 'match_prepare_kernel' match_prepare_kernel
dump matcher 'seeds_geom_kernelINS_14SeedSrcCompact' seeds_geom_kernel_compact
dump matcher 'epi_search_kernel' epi_search_kernel
dump matcher 'lk_refine_kernel' lk_refine_kernel
dump matcher 'seeds_finish_kernelINS_14SeedSrcCompact' seeds_finish_kernel_compact
