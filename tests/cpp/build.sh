#!/bin/sh
# Builds the C++17 host-API tests against the in-tree libraries (no GPU needed to compile).
set -e
cd "$(dirname "$0")"
ROOT=../..
HOST=$ROOT/lidar-slam-from-scratch_b200/host
g++ -std=c++17 -O2 -Wall -Wno-unused-function -I$ROOT/include -I$HOST \
    host_api_test.cpp -o host_api_test \
    -L$ROOT/lidar-slam-from-scratch_b200 -lslam_b200 -L$ROOT/oracle -loracle -L$ROOT/synth -lsynth \
    -Wl,-rpath,'$ORIGIN/../../lidar-slam-from-scratch_b200' -Wl,-rpath,'$ORIGIN/../../oracle' -Wl,-rpath,'$ORIGIN/../../synth'
# the same test through the headers' Eigen branch (`__has_include(<Eigen/Dense>)`): Eigen itself is not in this image, the
# Eigen-API stand-in of the oracle (oracle/eigen_standin) takes its place, so PointCloud::Matrix etc. are Eigen-style types
g++ -std=c++17 -O2 -Wall -Wno-unused-function -I$ROOT/oracle/eigen_standin -I$ROOT/include \
    -I$HOST host_api_test.cpp -o host_api_test_eigenapi \
    -L$ROOT/lidar-slam-from-scratch_b200 -lslam_b200 -L$ROOT/oracle -loracle -L$ROOT/synth -lsynth \
    -Wl,-rpath,'$ORIGIN/../../lidar-slam-from-scratch_b200' -Wl,-rpath,'$ORIGIN/../../oracle' -Wl,-rpath,'$ORIGIN/../../synth'
echo "built tests/cpp/host_api_test and tests/cpp/host_api_test_eigenapi"
# the multi-GPU exchanges from a C++ host program (NCCL communicator owned by the caller)
g++ -std=c++17 -O2 -Wall -I$ROOT/include -I/usr/local/cuda/include gather_test.cpp -o gather_test \
    -L$ROOT/lidar-slam-from-scratch_b200 -lslam_b200 -lnccl -L/usr/local/cuda/lib64 -lcudart \
    -Wl,-rpath,'$ORIGIN/../../lidar-slam-from-scratch_b200'
echo "built tests/cpp/gather_test"

# The node's include order and call sites against the mirror, compile-only, in both branches of dense.hpp.
# REFERENCE_ROOT: the original project's checkout, where there is one (its include directory goes last)
REF=${REFERENCE_ROOT:+$REFERENCE_ROOT/slam_viz}
REF_INC=${REF:+-I$REF/include}
mkdir -p obj
g++ -std=c++17 -O1 -Wall -c -I$HOST -I$ROOT/include $REF_INC call_sites_test.cpp -o obj/call_sites_noeigen.o
g++ -std=c++17 -O1 -Wall -c -I$ROOT/oracle/eigen_standin -I$HOST -I$ROOT/include $REF_INC call_sites_test.cpp \
    -o obj/call_sites_eigenapi.o
echo "compiled tests/cpp/call_sites_test.cpp (no-Eigen and Eigen-API branches)"

# INTEGRATION.md section 1, literally: the reference's UNMODIFIED slam_node.cpp and file_utils.cpp compiled with the
# mirror directory in front of the reference's include directory (ROS 2 = tests/cpp/ros_stubs, Eigen = the oracle's
# stand-in, PoseGraph = a GTSAM-free test double), linked against libslam_b200.so.  Needs the reference's sources:
# where they are absent the binary is not built and the tests that run it skip.
if [ -n "$REF" ] && [ -f "$REF/src/ros/slam_node.cpp" ]; then
    INC="-Iros_stubs -I$ROOT/oracle/eigen_standin -I$HOST -I$ROOT/include $REF_INC"
    g++ -std=c++17 -O2 -c $INC "$REF/src/ros/slam_node.cpp" -o obj/slam_node.o
    g++ -std=c++17 -O2 -c $INC "$REF/src/core/file_utils.cpp" -o obj/file_utils.o
    g++ -std=c++17 -O2 -Wall -c $INC pose_graph_double.cpp -o obj/pose_graph_double.o
    g++ obj/slam_node.o obj/file_utils.o obj/pose_graph_double.o -o slam_node_dropin \
        -L$ROOT/lidar-slam-from-scratch_b200 -lslam_b200 -Wl,-rpath,'$ORIGIN/../../lidar-slam-from-scratch_b200'
    echo "built tests/cpp/slam_node_dropin from $REF (unmodified slam_node.cpp + file_utils.cpp over the mirror headers)"
else
    echo "REFERENCE_ROOT does not name the original project's checkout: tests/cpp/slam_node_dropin not built"
fi
