// The three BGR instantiations of resize_u8c3_kernel on the same 256 packed frames -> 416x416: packed (uniform stride),
// pitched (LAYOUT, with the packed layout as its record) and ragged (one descriptor per frame, all of one size, which the
// library's own calls never send there: a one-size call takes the uniform kernel).  CUDA events, 15 rounds of 20 launches,
// the three alternating in rotated order; medians in ms, and whether the outputs are equal.
//
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 --expt-relaxed-constexpr \
//        -I yolo-compression-and-deployment-in-fpga_b200/csrc -o /tmp/resize_pitched_bgr tools/micro/resize_pitched_bgr.cu
#include "resize.cu"
#include <cstdio>
#include <vector>
#include <algorithm>
using namespace yb;
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e)); return 1; } } while (0)
int main() {
    const int B = 256, dh = 416, dw = 416; int sm = 148;
    for (auto g : std::vector<std::pair<int,int>>{{480,640},{1080,1920}}) {
        int sh = g.first, sw = g.second; size_t fb = (size_t)sh * sw * 3, bytes = fb * B;
        std::vector<uint8_t> h(bytes); uint32_t s = 1; for (auto &v : h) { s = s * 1664525u + 1013904223u; v = s >> 24; }
        uint8_t *src, *dst[3]; CK(cudaMalloc(&src, bytes)); CK(cudaMemcpy(src, h.data(), bytes, cudaMemcpyHostToDevice));
        for (auto &d : dst) CK(cudaMalloc(&d, (size_t)B * dh * dw * 3));
        std::vector<int4> yt(dh); std::vector<int2> xt(dw); resize_geometry_tables(sh, sw, dh, dw, yt.data(), xt.data());
        int4 *ytab; int2 *xtab; CK(cudaMalloc(&ytab, dh * 16)); CK(cudaMalloc(&xtab, dw * 8));
        CK(cudaMemcpy(ytab, yt.data(), dh * 16, cudaMemcpyHostToDevice)); CK(cudaMemcpy(xtab, xt.data(), dw * 8, cudaMemcpyHostToDevice));
        ResizeLayout L{}; L.stride = fb; L.pitch[0] = 3 * sw; ResizeLayout *ld; CK(cudaMalloc(&ld, sizeof L)); CK(cudaMemcpy(ld, &L, sizeof L, cudaMemcpyHostToDevice));
        std::vector<ResizeFrame> fr(B); for (int i = 0; i < B; ++i) fr[i] = {(unsigned long long)i * fb, 3 * sw, 0};
        ResizeFrame *fd; CK(cudaMalloc(&fd, B * sizeof(ResizeFrame))); CK(cudaMemcpy(fd, fr.data(), B * sizeof(ResizeFrame), cudaMemcpyHostToDevice));
        auto run = [&](int k) {
            if (k == 0) return resize_launch<false>(src, bytes, nullptr, B, sh, sw, dst[0], dh, dw, xtab, ytab, sm, 0);
            if (k == 1) return resize_launch<false, RS_BGR, true>(src, bytes, (const ResizeFrame *)ld, B, sh, sw, dst[1], dh, dw, xtab, ytab, sm, 0);
            return resize_launch<true>(src, bytes, fd, B, 0, 0, dst[2], dh, dw, xtab, ytab, sm, 0);
        };
        const char *names[3] = {"packed", "layout", "ragged"};
        std::vector<float> t[3]; cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
        for (int r = 0; r < 15; ++r) for (int j = 0; j < 3; ++j) { int k = (j + r) % 3;
            run(k); run(k); cudaEventRecord(e0); for (int i = 0; i < 20; ++i) run(k); cudaEventRecord(e1); cudaEventSynchronize(e1);
            float ms; cudaEventElapsedTime(&ms, e0, e1); t[k].push_back(ms / 20); }
        CK(cudaDeviceSynchronize());
        std::vector<uint8_t> o0((size_t)B*dh*dw*3), o1(o0.size()), o2(o0.size());
        CK(cudaMemcpy(o0.data(), dst[0], o0.size(), cudaMemcpyDeviceToHost)); CK(cudaMemcpy(o1.data(), dst[1], o0.size(), cudaMemcpyDeviceToHost)); CK(cudaMemcpy(o2.data(), dst[2], o0.size(), cudaMemcpyDeviceToHost));
        printf("256 x %dx%d -> 416x416: outputs equal %d %d, ms", sh, sw, (int)(o0 == o1), (int)(o0 == o2));
        for (int k = 0; k < 3; ++k) { std::sort(t[k].begin(), t[k].end()); printf(" %s=%.4f", names[k], t[k][7]); } printf("\n");
        cudaFree(src); for (auto d : dst) cudaFree(d); cudaFree(ytab); cudaFree(xtab); cudaFree(ld); cudaFree(fd);
    }
    return 0;
}
