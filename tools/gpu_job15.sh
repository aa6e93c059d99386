echo "=== glamr_3dpw (camera from persons) iteration"
GLAMR_LBS_PATH=tcblend CFG=glamr_3dpw GLAMR_B200_SO=glamr_b200/libglamr_b200_exp.so timeout 300 python tools/iter_skip_exp.py 2>&1 | tail -1 | sed "s/^/tcblend  /"
echo "=== c5 sequence breakdown"
CFG=glamr_3dpw GAPS=1 timeout 300 python tools/e2e_breakdown.py 0 300 1 2>&1 | head -24 | cut -c1-250
