#!/bin/sh
# Builds oracle/_ref/libslam_ref.so: the reference's own hot-path sources (headers under
# slam_viz/include/slam_viz/core + src/core/file_utils.cpp), compiled UNMODIFIED where they lie under
# $REFERENCE_ROOT (a checkout of the original project) against oracle/eigen_standin (Eigen is not in this image) with the
# reference's release flags (-O3 -DNDEBUG, slam_viz/CMakeLists.txt:13).  Nothing is copied into the repository;
# the output directory is git-ignored.  Exits 0 without building when REFERENCE_ROOT names no such checkout.
set -e
cd "$(dirname "$0")"
REF="$REFERENCE_ROOT/slam_viz"
if [ -z "$REFERENCE_ROOT" ] || [ ! -f "$REF/include/slam_viz/core/icp.hpp" ]; then
    echo "REFERENCE_ROOT does not name the original project's checkout: oracle/_ref not built"
    exit 0
fi
mkdir -p _ref
g++ -std=c++17 -O3 -DNDEBUG -ffp-contract=off -fPIC -shared \
    -I eigen_standin -I "$REF/include" \
    -o _ref/libslam_ref.so ref_harness.cpp "$REF/src/core/file_utils.cpp"
echo "built oracle/_ref/libslam_ref.so from $REF"
