// kfusion/io/ply.hpp -- export of the extracted canonical cloud (SURVEY.md 8f(4); the reference lists "Export the reconstructions to
// .ply or .obj files" under its next steps, Report.md, and has no such code).  Header-only, host-only: it takes what
// cuda::TsdfVolume::get_cloud_host() / get_normal_host() return (1 x N CV_32FC4 rows of kfusion::Point / Normal,
// tsdf_volume.cpp:313-325) and writes a binary little-endian PLY with float x y z [nx ny nz]; points with a NaN coordinate are skipped
// (normals that are NaN -- extractNormals marks points within two voxels of the border that way, tsdf_volume.cu:744-751 -- are
// written as 0 0 0).  Returns the number of vertices written, -1 if the file cannot be opened.
#pragma once
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include <opencv2/core/core.hpp>

namespace kfusion
{
    inline long writePly(const std::string& path, const cv::Mat& cloud, const cv::Mat& normals = cv::Mat())
    {
        const int n = cloud.cols * cloud.rows;
        const bool with_normals = !normals.empty() && normals.cols * normals.rows == n;
        const float *p = cloud.ptr<float>(), *q = with_normals ? normals.ptr<float>() : 0;
        std::vector<float> out;
        out.reserve((size_t)n * (with_normals ? 6 : 3));
        long count = 0;
        for (int i = 0; i < n; ++i) {
            const float *v = p + 4 * (size_t)i;
            if (std::isnan(v[0]) || std::isnan(v[1]) || std::isnan(v[2])) continue;
            out.push_back(v[0]); out.push_back(v[1]); out.push_back(v[2]);
            if (with_normals) {
                const float *m = q + 4 * (size_t)i;
                const bool bad = std::isnan(m[0]) || std::isnan(m[1]) || std::isnan(m[2]);
                out.push_back(bad ? 0.f : m[0]); out.push_back(bad ? 0.f : m[1]); out.push_back(bad ? 0.f : m[2]);
            }
            ++count;
        }
        std::FILE *f = std::fopen(path.c_str(), "wb");
        if (!f) return -1;
        std::fprintf(f, "ply\nformat binary_little_endian 1.0\ncomment dynamicfusion canonical cloud\nelement vertex %ld\n"
                        "property float x\nproperty float y\nproperty float z\n", count);
        if (with_normals) std::fprintf(f, "property float nx\nproperty float ny\nproperty float nz\n");
        std::fprintf(f, "end_header\n");
        if (!out.empty()) std::fwrite(&out[0], sizeof(float), out.size(), f);
        std::fclose(f);
        return count;
    }

    // Mesh form (not in the reference): what cuda::TsdfVolume::fetchMesh / KinFu::getMesh return -- vertices and normals 1 x N CV_32FC4,
    // triangles M x 1 CV_32SC3 (or any 4-byte-element Mat holding 3*M indices) -- as a binary little-endian PLY with float x y z [nx ny nz]
    // per vertex and `element face M` / `property list uchar int vertex_indices`.  Every vertex is written as given (mesh vertices are
    // finite, and dropping one would shift the indices); NaN normals are written as 0 0 0.  Returns the number of vertices written, -1 if
    // the file cannot be opened.
    inline long writePly(const std::string& path, const cv::Mat& vertices, const cv::Mat& normals, const cv::Mat& triangles)
    {
        const int n = vertices.cols * vertices.rows;
        const bool with_normals = !normals.empty() && normals.cols * normals.rows == n;
        const long m = triangles.empty() ? 0 : (long)((size_t)triangles.rows * triangles.cols * triangles.elemSize() / 12);
        const float *p = n ? vertices.ptr<float>() : 0, *q = with_normals ? normals.ptr<float>() : 0;
        std::vector<float> out;
        out.reserve((size_t)n * (with_normals ? 6 : 3));
        for (int i = 0; i < n; ++i) {
            const float *v = p + 4 * (size_t)i;
            out.push_back(v[0]); out.push_back(v[1]); out.push_back(v[2]);
            if (with_normals) {
                const float *w = q + 4 * (size_t)i;
                const bool bad = std::isnan(w[0]) || std::isnan(w[1]) || std::isnan(w[2]);
                out.push_back(bad ? 0.f : w[0]); out.push_back(bad ? 0.f : w[1]); out.push_back(bad ? 0.f : w[2]);
            }
        }
        std::vector<unsigned char> faces((size_t)m * 13);
        const unsigned char *t = m ? triangles.ptr<unsigned char>() : 0;
        for (long i = 0; i < m; ++i) {
            faces[13 * (size_t)i] = 3;
            std::memcpy(&faces[13 * (size_t)i + 1], t + 12 * (size_t)i, 12);
        }
        std::FILE *f = std::fopen(path.c_str(), "wb");
        if (!f) return -1;
        std::fprintf(f, "ply\nformat binary_little_endian 1.0\ncomment dynamicfusion mesh\nelement vertex %d\n"
                        "property float x\nproperty float y\nproperty float z\n", n);
        if (with_normals) std::fprintf(f, "property float nx\nproperty float ny\nproperty float nz\n");
        std::fprintf(f, "element face %ld\nproperty list uchar int vertex_indices\nend_header\n", m);
        if (!out.empty()) std::fwrite(&out[0], sizeof(float), out.size(), f);
        if (!faces.empty()) std::fwrite(&faces[0], 1, faces.size(), f);
        std::fclose(f);
        return n;
    }
}
