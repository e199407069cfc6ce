#!/bin/bash
# Memory-safety pass over the device-array copies (pa_field_upload_device / pa_field_download_device, k_array4_copy), the
# companion of asan_check.sh: the emulated library with pointer attributes (build_emu_ptr.py) built with AddressSanitizer,
# then dense, strided and ghosted sources and destinations on every box shape of a set of golden fixtures, and every error
# path.  "Device" arrays are heap blocks with red zones, so a row or component index outside an array is a hard error here.
#   usage: tests/emu/asan_check_device_io.sh
set -e
ROOT=$(cd "$(dirname "$0")/../.." && pwd)
LIB=$(cd "$ROOT/tests/emu" && python -c "import build_emu_ptr; print(build_emu_ptr.build(asan=True))")
OUT=$(dirname "$LIB")
cat > "$OUT/run.py" <<PY
import importlib.util, os, sys
sys.path.insert(0, "$ROOT"); sys.path.insert(0, "$ROOT/tests"); sys.path.insert(0, "$ROOT/tests/emu")
from peleanalysis_b200 import capi as pc
spec = importlib.util.spec_from_file_location("capi_emulated", pc.__file__); emu = importlib.util.module_from_spec(spec); spec.loader.exec_module(emu)
emu.LIB_PATH = "$LIB"; os.environ["PA_NORMAL_MATH"] = "fast"; emu.init(0)
import test_emu_device_io as E, test_gpu_device_io as DIO
from helpers import load_golden
DB = E.EmuBackend(emu)
n = 0
for name in ("c3_three_levels", "mixed_boxes", "thin", "np2", "ratio4", "filter_c3_subset"):
    pf, z = load_golden(name)
    per = tuple(int(v) for v in z["is_per"]) if "is_per" in z.files else (0, 0, 0)
    for ng in (1, 2):
        DIO.check_upload_download(emu, DB, pf, per, ng=ng); n += 1
DIO.check_errors(emu, DB); n += 1
print("asan check (device arrays): %d runs, no error" % n)
PY
ASAN_OPTIONS=detect_leaks=0:detect_stack_use_after_return=0 LD_PRELOAD=$(gcc -print-file-name=libasan.so) python "$OUT/run.py"
