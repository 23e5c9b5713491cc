#!/bin/bash
# SASS summary of the shipped library -> profiles/<tag>_sass_summary.txt      usage: tools/sass_summary.sh r2
tag=${1:-rXX}
lib=pertrenderer_b200/libpertshade.so
out=profiles/${tag}_sass_summary.txt
tmp=$(mktemp)
cuobjdump -sass $lib > $tmp
{
echo "# SASS summary of $lib (python -m pertrenderer_b200.build --force)"
echo "# cuobjdump -sass libpertshade.so | grep -c <mnemonic>"
for m in UBLKCP UTMALDG SYNCS LDGSTS IMAD.WIDE.U32 MUFU ATOMS LDG.E.128 STG.E.128 HMMA UTCHMMA; do printf "%-16s %s\n" $m $(grep -c "$m" $tmp); done
echo
echo "# functions (kernels and out-of-line device functions): $(grep -c 'Function :' $tmp)"
echo "# LDGSTS: cp.async copy of the saved winners rows in the main pass of backward (a bulk copy + mbarrier was measured in its place: +1 %, r2_notes.md)"
echo "# UBLKCP / SYNCS (TMA 1-D bulk copy + mbarrier): 0.  A bulk-copy scan of the forward was measured and rejected"
echo "#   (DESIGN.md section 3, r2_notes.md)"
echo "# no tensor-core mnemonics: the path has no dense contraction (north_star)"
echo "# instructions per production kernel (config 2, K = 50; the SM's instruction cache holds 2048):"
awk '/Function :/{if(name)print n, name; name=$3; n=0} /^ +\/\*[0-9a-f]{4}\*\//{n++} END{print n,name}' $tmp | grep "PhiloxNoiseTILi10EEES2_Li2ELb0ELb1ELi0ELb0ELb0E\|fwd_fallback_kernelINS_12PhiloxNoiseTILi10EEELi4ELi\(16\|96\)ELb0E\|shade_bwd_kernelINS_12PhiloxNoiseTILi10EEELi2ELb0ELb0ELb1ELb1E\|shade_bwd_fallback_kernelINS_12PhiloxNoiseTILi10EEELi4ELb0E" | while read n name; do echo "#   $n  $(echo $name | c++filt | cut -c1-150)"; done
} > $out
rm -f $tmp
cat $out
