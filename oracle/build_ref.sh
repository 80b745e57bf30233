#!/bin/bash
# TEST INFRASTRUCTURE ONLY.
# Builds the UNMODIFIED reference (intel/yask) hot path out-of-tree into oracle/_ref/
# from the sources where they lie under /root/reference, plus oracle/ref_driver.cpp
# against each resulting kernel library.  Nothing is copied from /root/reference and
# nothing is written there (YASK_OUTPUT_DIR keeps all outputs under oracle/_ref/yask,
# see /root/reference/src/common/common.mk:38-55).
#
# NOTE (see DESIGN.md "Oracle"): the reference's hot path is *generated* code (its
# stencil compiler + perl loop generators run at build time), so it cannot be built by
# "gcc on a few source files".  We therefore drive the reference's own makefiles, in
# this container only; the GPU box uses the prebuilt oracle/_ref/ files (git-ignored,
# but shipped by gpurun) and never needs /root/reference.
#
# usage: [REF_ALL=1] oracle/build_ref.sh [arch]     (arch: avx512 (default) | avx2 | intel64)
#   default: the references bench.py's CPU arms and the live-reference tests need: iso3dfd (default + strict),
#            awp_elastic fp32 and ssg fp64 (default flags), ~4 min;
#   REF_ALL=1: every solution the golden fixtures were generated from (~90 kernel builds, over an hour);
#   REF_RADII=1: only iso3dfd at radius 1 and 2 (fixtures of the temporal tile), ~3 min.
#
# Outputs: oracle/_ref/yask/        the reference's own output tree (build products and intermediates);
#          oracle/_ref/ship/        what the tests and bench.py run, kept apart from that tree so that it can be
#                                   copied on its own to a machine without the reference:
#            bin/, lib/             the reference harnesses and drivers of the benchmarked stencils;
#            refc/                  the reference's stencil COMPILER, which the product's build-time CUDA emitter
#                                   (yask_b200/emitter) drives as its front-end -- a build tool, not part of the oracle;
#            tests/                 the reference's own C++ API tests (src/kernel/tests), compiled unmodified against
#                                   this project's C++ API header and libraries (yask_b200/lib, built first), and its
#                                   Python API tests, byte-compiled.
set -e
REF=${YASK_REFERENCE:-/root/reference}
HERE=$(cd "$(dirname "$0")" && pwd)
OUT=$HERE/_ref/yask
ARCH=${1:-avx512}
J=${JOBS:-8}

if [ ! -d "$REF/src/kernel" ]; then
    echo "build_ref.sh: $REF not present (GPU box?) -- using prebuilt oracle/_ref as is"
    exit 0
fi
mkdir -p "$OUT"
LOG=$HERE/_ref/build.log
: > "$LOG"

SHIP=$HERE/_ref/ship
REFC=$SHIP/refc
if [ ! -x "$REFC/bin/yask_compiler.exe" ]; then
    echo "[build_ref] yask compiler -> oracle/_ref/ship/refc"
    mkdir -p "$REFC"
    # the library first, with a SONAME: the executable then records it by name, not by this tree's path, so the staged
    # compiler runs wherever ship/ is copied (the emitter puts refc/lib on LD_LIBRARY_PATH)
    make -C "$REF/src/compiler" YASK_OUTPUT_DIR="$REFC" mpi=0 arch=$ARCH -j$J EXTRA_YC_CXXFLAGS=-Wl,-soname,libyask_compiler.so \
        "$REFC/lib/libyask_compiler.so" >> "$LOG" 2>&1
    make -C "$REF/src/compiler" YASK_OUTPUT_DIR="$REFC" mpi=0 arch=$ARCH -j$J compiler >> "$LOG" 2>&1
    rm -rf "$REFC/build"
fi
# the reference's kernel makefile looks for the compiler in its own output tree
mkdir -p "$OUT/bin" "$OUT/lib"
ln -sf "$REFC/bin/yask_compiler.exe" "$OUT/bin/yask_compiler.exe"
ln -sf "$REFC/lib/libyask_compiler.so" "$OUT/lib/libyask_compiler.so"

# stencil  suffix  real_bytes  extra-make-args
build_kernel() {
    local st=$1 suf=$2 rb=$3; shift 3
    local tag="$st$suf.$ARCH"
    if [ ! -f "$OUT/lib/libyask_kernel.$tag.so" ] || [ ! -x "$OUT/bin/yask_kernel.$tag.exe" ]; then
        echo "[build_ref] kernel $tag"
        make -C "$REF/src/kernel" YASK_OUTPUT_DIR="$OUT" stencil=$st YK_STENCIL_SUFFIX=$suf arch=$ARCH \
            mpi=0 numa=0 real_bytes=$rb -j$J "$@" default >> "$LOG" 2>&1
    fi
    if [ ! -x "$OUT/bin/ref_driver.$tag" ] || [ "$HERE/ref_driver.cpp" -nt "$OUT/bin/ref_driver.$tag" ]; then
        g++ -std=c++17 -O2 -fopenmp -I"$REF/include" "$HERE/ref_driver.cpp" \
            -L"$OUT/lib" -Wl,-rpath,'$ORIGIN/../lib' -lyask_kernel.$tag -lrt -o "$OUT/bin/ref_driver.$tag"
    fi
}

# Default flags (GCC -O3 => -ffp-contract=fast: FMAs formed by the host compiler) and
# "-strict" (-ffp-contract=off: pure IEEE mul/add in DSL order), SURVEY.md section 7 hard part 1.
build_kernel iso3dfd ""        4
build_kernel iso3dfd "-strict" 4 EXTRA_YK_CXXFLAGS=-ffp-contract=off
if [ "$ARCH" = "avx512" ]; then
    build_kernel awp_elastic ""        4
    build_kernel ssg "-fp64"        8
fi
if [ "${REF_ALL:-0}" = "1" ] || [ "${REF_RADII:-0}" = "1" ]; then
    # iso3dfd at the radii of the temporal tile (the reference fixes the radius at build time): fixtures for tests/test_temporal_*
    for r in 1 2 4; do        # 4: the usual 8th-order stencil, served by the one-step kernel of that radius
        build_kernel iso3dfd "-r$r"        4 radius=$r
        build_kernel iso3dfd "-r$r-strict" 4 radius=$r EXTRA_YK_CXXFLAGS=-ffp-contract=off
    done
fi
if [ "${REF_ALL:-0}" = "1" ]; then
    build_kernel awp_elastic "-strict" 4 EXTRA_YK_CXXFLAGS=-ffp-contract=off
    build_kernel ssg "-fp64-strict" 8 EXTRA_YK_CXXFLAGS=-ffp-contract=off
    build_kernel iso3dfd "-fp64"        8
    build_kernel iso3dfd "-fp64-strict" 8 EXTRA_YK_CXXFLAGS=-ffp-contract=off
    # further solutions the CUDA emitter covers (SURVEY.md section 8f-1); "3axis" is the heat3d-style shape
    for st in awp iso3dfd_sponge 3axis 3axis_with_diags 3plane cube tti awp_elastic_abc awp_abc test_1d test_2d test_3d test_boundary_3d test_stream_3d fsg fsg_abc ssg2 ssg_merged fsg2; do
        build_kernel $st ""        4
        build_kernel $st "-strict" 4 EXTRA_YK_CXXFLAGS=-ffp-contract=off
    done
    # second batch: remaining example/test solutions (filters, merged/abc FSG variants, 1-D/2-D tests, stages,
    # scratch vars, step conditions, math functions)
    for st in box_filter gaussian_filter fsg2_abc fsg_merged fsg_merged_abc test_boundary_1d test_boundary_2d test_partial_3d \
              test_stages_1d test_stages_2d test_stages_3d test_stream_1d test_stream_2d test_reverse_2d \
              test_scratch_1d test_scratch_2d test_scratch_3d test_scratch_boundary_1d test_scratch_stages_1d \
              test_step_cond_1d test_func_1d test_misc_2d wave2d swe2d; do
        build_kernel $st ""        4
        build_kernel $st "-strict" 4 EXTRA_YK_CXXFLAGS=-ffp-contract=off
    done
fi
# Strip debug info (the reference builds with -g) and drop the (large) intermediate build tree.
strip --strip-debug "$OUT"/lib/libyask_kernel.*.so "$OUT"/bin/yask_kernel.*.exe "$OUT"/bin/ref_driver.* "$REFC"/bin/* "$REFC"/lib/* 2>/dev/null || true
if [ "${KEEP_BUILD:-0}" != "1" ]; then rm -rf "$OUT/build"; fi
# what the GPU box runs: the reference harnesses of the three benchmarked stencils and the iso3dfd API drivers
mkdir -p "$SHIP/bin" "$SHIP/lib"
for tag in iso3dfd.$ARCH iso3dfd-strict.$ARCH awp_elastic.$ARCH ssg-fp64.$ARCH; do
    [ -f "$OUT/lib/libyask_kernel.$tag.so" ] || continue
    cp -u "$OUT/lib/libyask_kernel.$tag.so" "$SHIP/lib/"
    cp -u "$OUT/bin/yask_kernel.$tag.exe" "$OUT/bin/ref_driver.$tag" "$SHIP/bin/" 2>/dev/null || true
done
# the reference's own API tests against this project's libraries, on the solutions those libraries are built for
# (yask_b200/csrc/Makefile YK_STENCILS); the Python ones run with the pybind11 modules under yask_b200/lib/python
YB=$(cd "$HERE/.." && pwd)/yask_b200
TESTS=$REF/src/kernel/tests
if [ -f "$YB/lib/libyask_b200.so" ]; then
    mkdir -p "$SHIP/tests"
    api_test() {    # source  stencil  output
        local out=$SHIP/tests/$3
        if [ ! -x "$out" ] || [ "$TESTS/$1.cpp" -nt "$out" ] || [ "$YB/include/yask_kernel_api.hpp" -nt "$out" ]; then
            g++ -std=c++17 -O1 -I"$YB/include" "$TESTS/$1.cpp" -L"$YB/lib" -lyask_kernel.$2.b200 -lyask_b200 \
                -Wl,-rpath,'$ORIGIN/../../../../yask_b200/lib' -o "$out"
        fi
    }
    for st in iso3dfd awp_elastic ssg test_3d; do
        api_test yask_kernel_api_test $st ref_kernel_api_test.$st
    done
    api_test yask_kernel_api_exception_test iso3dfd ref_kernel_api_exception_test.iso3dfd
    for t in yask_kernel_api_test yask_kernel_api_exception_test; do
        ${PYTHON:-python} -c "import py_compile, sys; py_compile.compile(sys.argv[1], cfile=sys.argv[2], doraise=True)" \
            "$TESTS/$t.py" "$SHIP/tests/ref_$t.pyc"
    done
else
    echo "[build_ref] yask_b200/lib not built: the reference's API tests are not compiled"
fi
echo "[build_ref] done: $(ls "$OUT/bin" | grep -c ref_driver) reference driver(s) under $OUT/bin"
