set -x
timeout 300 python tools/diag_target.py 2>&1 | tail -80
(cd deepmimic_b200/csrc && make profile >/dev/null 2>&1)
DM_LIB=$PWD/deepmimic_b200/libdeepmimic_b200_prof.so timeout 300 python tools/section_profile.py 2>&1 | tail -40
timeout 900 python -m pytest tests/test_qd_envelope_gpu.py tests/test_parity2_gpu.py -m gpu -q --tb=short -s 2>&1 | tail -60
DM_LIB=$PWD/deepmimic_b200/libdeepmimic_b200_precise.so timeout 600 python -m pytest tests/test_qd_envelope_gpu.py -m gpu -q --tb=short -s 2>&1 | tail -30
