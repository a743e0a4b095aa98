#!/bin/bash
# Full SASS listings of the kernels that dominate the large-problem path (profiles/<round>_sass_<kernel>.txt), hex encodings
# stripped.  No GPU needed: cuobjdump reads the sm_100a cubin inside libba_gpu.so.
#   scripts/dump_sass.sh                    round r02, the default kernel list
#   scripts/dump_sass.sh r06 k_sp_schur     one round's kernels; a name matches the kernel of exactly that name
cd "$(dirname "$0")/.." || exit 1
SO=3dsmc-bundle-adjustment_b200/libba_gpu.so
ROUND=${1:-r02}
shift
KERNELS=${*:-k_sp_schur k_spchol_tree k_spchol_factor k_spchol_update k_spchol_solve kf_pt_blocks kf_cam_blocks kf_schur_pass1 kf_linearize k_linearize}
for k in $KERNELS; do
  if [ "$ROUND" = r02 ]; then pat="$k"; else pat="Function : _Z[0-9]+${k}[^_]"; fi
  cuobjdump -sass $SO | awk -v k="$pat" '/Function :/{p=($0 ~ k)} p' |
    sed -E 's#[[:space:]]*/\* 0x[0-9a-f]+ \*/[[:space:]]*$##; /^[[:space:]]*\/\* 0x[0-9a-f]+ \*\/[[:space:]]*$/d' > profiles/${ROUND}_sass_$k.txt
done
if [ "$ROUND" = r02 ]; then
  awk '/Function :/{n++} n<=1' profiles/r02_sass_k_linearize.txt > profiles/.t && mv profiles/.t profiles/r02_sass_k_linearize.txt
fi
wc -l profiles/${ROUND}_sass_*.txt
