# A/B with repeats on ONE box (box-to-box spread of the step time is ~1 %, so variants are compared inside one call):
# early part of the grouped dW+Adam launch off (0) / on (92 SMs, the default).  Other knobs measured the same way this
# round: DRVAE_B200_STEPK, build variants through DRVAE_B200_LIB (tools/r02_rowlb.sh, tools/r02_dwa_ab.sh), and
# schedule variants since removed (DESIGN.md §4, profiles/r02_experiments.md).
for rep in 1 2 3; do
for g in 0 92; do
  DRVAE_B200_DWA_EARLY_SMS=$g python bench.py --steps 30 --warmup 5 --no-cpu-baseline --no-extras 2>/dev/null | python -c "
import json,sys
for l in sys.stdin:
    if l.startswith('{'):
        d=json.loads(l); print('early $g: ms/step %.4f e2e %.4g' % (d['ms_per_step'], d['e2e']['value']))"
done
done
