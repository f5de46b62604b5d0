#!/bin/bash
# Robustness check of the host-side scene parser (rrtb_host.cpp: grammar of scene.h:212-452) -- CPU only: build it with
# AddressSanitizer + UndefinedBehaviorSanitizer behind a tiny driver and feed it mutated copies of the reference's scenes
# (truncated, shuffled, tokens replaced by keywords / nan / inf / huge numbers, random bytes inserted).  The parser may
# reject a file, it may not crash, overflow or leak.   usage: tools/fuzz_parser.sh [n_files] [scenes_dir]
N=${1:-600}; SC=${2:-$(dirname "$0")/../oracle/_ref/scenes}
[ -d "$SC" ] || SC="$(dirname "$0")/../tests/golden/scenes"
ROOT="$(cd "$(dirname "$0")/.." && pwd)"; W=$(mktemp -d /tmp/rrtb_fuzz.XXXXXX); mkdir -p $W/in
cat > $W/drv.cpp <<EOF
#include <stdint.h>
#include "$ROOT/include/rrtb.h"
extern "C" { // the device-side entry points rrtb_host.cpp refers to (rrtb_scene_upload); never called here
int rrtb_scene_stage_moving_triangles(rrtb_ctx *, const rrtb_mtriangle *, int32_t) { return 0; }
int rrtb_scene_stage_background(rrtb_ctx *, const float *) { return 0; }
int rrtb_scene_set(rrtb_ctx *, const rrtb_camera *, const rrtb_material *, int32_t, const rrtb_sphere *, int32_t, const rrtb_msphere *, int32_t,
                   const rrtb_triangle *, int32_t, int32_t) { return 0; }
}
int main(int argc, char **argv) {
    for (int i = 1; i < argc; ++i) {
        rrtb_scene *s = nullptr; int code = 0; char err[512];
        if (rrtb_scene_parse_file(argv[i], 320, 200, &s, &code, err, 512) == 0 && s) { int32_t c[6]; float bg[3]; rrtb_scene_counts(s, c); rrtb_scene_background(s, bg); rrtb_scene_free(s); }
    }
    return 0;
}
EOF
g++ -std=c++17 -O1 -g -fsanitize=address,undefined -fno-omit-frame-pointer $W/drv.cpp $ROOT/rrt_b200/csrc/rrtb_host.cpp -o $W/drv -lz || exit 1
python3 - "$SC" "$W/in" "$N" <<'PY'
import glob, os, random, sys
sc, out, n = sys.argv[1], sys.argv[2], int(sys.argv[3])
random.seed(7)
base = [open(p).read() for p in sorted(glob.glob(os.path.join(sc, "*.txt")))]
toks = ["camera", "material", "sphere", "moving_sphere", "obj", "obj_inst", "triangle", "mobj", "kobj", "lambertian", "metal", "dielectric",
        "translate", "rotate", "scale", "diffuse_light", "background", "#", "nan", "inf", "-inf", "1e39", "-1e-50", "0", "m0", "m999", "", "9999999999999999999999", "/", "o0"]
for k in range(n):
    lines = random.choice(base).split("\n")
    how = random.randint(0, 5)
    if how == 0:
        lines = lines[:random.randint(0, len(lines))]
    elif how == 1:
        for _ in range(random.randint(1, 6)):
            i = random.randrange(len(lines)); w = lines[i].split(" "); w[random.randrange(len(w))] = random.choice(toks); lines[i] = " ".join(w)
    elif how == 2:
        for _ in range(random.randint(1, 6)):
            lines.insert(random.randrange(len(lines) + 1), " ".join(random.choice(toks) for _ in range(random.randint(1, 12))))
    elif how == 3:
        random.shuffle(lines)
    elif how == 4:
        s = "\n".join(lines); i = random.randrange(max(len(s), 1))
        lines = (s[:i] + "".join(chr(random.randrange(1, 127)) for _ in range(random.randint(1, 40))) + s[i:]).split("\n")
    else:
        lines = [l for l in lines if random.random() > 0.2]
    open(os.path.join(out, "f%04d.txt" % k), "w").write("\n".join(lines))
PY
cd $W/in && ../drv f*.txt > ../out.log 2>&1; rc=$?
bad=$(grep -c "runtime error\|ERROR: AddressSanitizer\|ERROR: LeakSanitizer" ../out.log)
echo "parser fuzz: $N files, driver exit $rc, sanitizer findings $bad  ($W/out.log)"
[ $rc -eq 0 ] && [ "$bad" -eq 0 ]
