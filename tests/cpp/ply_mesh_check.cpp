// ply_mesh_check.cpp -- CPU-only check of the mesh form of kfusion::writePly (include/kfusion/io/ply.hpp)
#include <kfusion/io/ply.hpp>
#include <cstdio>
#include <limits>
int main(int argc, char **argv)
{
    if (argc < 2) return 2;
    const int n = 5, m = 3;
    cv::Mat vertices(1, n, CV_32FC4), normals(1, n, CV_32FC4), triangles(m, 1, CV_32SC3);
    for (int i = 0; i < n; ++i) {
        float *p = vertices.ptr<float>() + 4 * i, *q = normals.ptr<float>() + 4 * i;
        p[0] = 0.25f * i; p[1] = 1.f - i; p[2] = 0.5f + i; p[3] = 0.f;
        q[0] = 1.f; q[1] = 0.f; q[2] = 0.f; q[3] = 0.f;
    }
    normals.ptr<float>()[4 * 2] = std::numeric_limits<float>::quiet_NaN();   // normal 2 is written as 0 0 0
    const int tri[m][3] = {{0, 1, 2}, {2, 1, 3}, {3, 4, 2}};
    for (int t = 0; t < m; ++t)
        for (int k = 0; k < 3; ++k) triangles.ptr<int>()[3 * t + k] = tri[t][k];
    const long a = kfusion::writePly(std::string(argv[1]) + "/mesh.ply", vertices, normals, triangles);
    const long b = kfusion::writePly(std::string(argv[1]) + "/mesh_no_normals.ply", vertices, cv::Mat(), triangles);
    std::printf("%ld %ld\n", a, b);
    return 0;
}
