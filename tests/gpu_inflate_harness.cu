// Conformance harness of the device inflate kernel (tests/test_gpu_inflate_conformance.py builds it with the library's
// nvcc flags).  It includes the kernel source, as tools/inflate_bench.cu does, and runs one batch per input file exactly
// as the engine would: the test lays the batch out (compressed offsets at any byte phase, raw offsets at any phase or
// packed back to back, any order and repetition), this program only uploads it and runs it.
//   usage: gpu_inflate_harness in.bin out.bin [in.bin out.bin ...]
// in.bin:  u32 n_blocks, comp_bytes, raw_bytes, 0; InflateBlock[n_blocks]; u32 crc[n_blocks]; comp_bytes bytes
// out.bin: u32 status without SpecOut, status with SpecOut, 1 if both runs left the same raw buffer; raw_bytes bytes (the
//          run with SpecOut); per block u32 cnt, end and, unless cnt is kSpecNone, cnt record offsets
// The compressed buffer has the engine's 4096 bytes of slack behind it; the raw buffer is filled with 0xA5 before every
// run, so that the test can check that nothing outside the blocks' outputs was written.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../bamsignals_b200/csrc/inflate.cu"

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e_)); return 2; } } while (0)

static int run_one(const char* in_path, const char* out_path) {
    FILE* f = fopen(in_path, "rb");
    if (!f) { perror(in_path); return 1; }
    uint32_t hdr[4];
    if (fread(hdr, 4, 4, f) != 4) { fclose(f); return 1; }
    const uint32_t n = hdr[0], comp_bytes = hdr[1], raw_bytes = hdr[2];
    std::vector<bsg::InflateBlock> blocks(n);
    std::vector<uint32_t> crcs(n);
    std::vector<uint8_t> comp(comp_bytes);
    const bool ok = fread(blocks.data(), sizeof(bsg::InflateBlock), n, f) == n && fread(crcs.data(), 4, n, f) == n &&
                    fread(comp.data(), 1, comp_bytes, f) == comp_bytes;
    fclose(f);
    if (!ok) { fprintf(stderr, "%s: short read\n", in_path); return 1; }
    uint8_t *d_comp, *d_raw;
    bsg::InflateBlock* d_blocks;
    uint32_t *d_crc, *d_spec;
    bsg::DeviceScalars* d_sc;
    CK(cudaMalloc(&d_comp, size_t(comp_bytes) + 4096));
    CK(cudaMemset(d_comp, 0, size_t(comp_bytes) + 4096));
    CK(cudaMalloc(&d_raw, size_t(raw_bytes) + 8));
    CK(cudaMalloc(&d_blocks, size_t(n) * sizeof(bsg::InflateBlock) + 16));
    CK(cudaMalloc(&d_crc, size_t(n) * 4 + 16));
    CK(cudaMalloc(&d_spec, bsg::inflate_spec_words(int(n)) * 4));
    CK(cudaMalloc(&d_sc, sizeof(bsg::DeviceScalars)));
    CK(cudaMemcpy(d_comp, comp.data(), comp_bytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_blocks, blocks.data(), size_t(n) * sizeof(bsg::InflateBlock), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_crc, crcs.data(), size_t(n) * 4, cudaMemcpyHostToDevice));
    uint32_t status[2];
    std::vector<uint8_t> raw[2];
    for (int with_spec = 0; with_spec < 2; ++with_spec) {
        CK(cudaMemset(d_raw, 0xA5, raw_bytes));
        CK(cudaMemset(d_sc, 0, sizeof(bsg::DeviceScalars)));
        bsg::launch_inflate(d_blocks, int(n), d_comp, d_raw, with_spec ? d_spec : nullptr, d_sc, 0);
        CK(cudaGetLastError());
        bsg::launch_crc32(d_blocks, d_crc, int(n), d_raw, d_sc, 0);
        CK(cudaGetLastError());
        CK(cudaDeviceSynchronize());
        bsg::DeviceScalars sc;
        CK(cudaMemcpy(&sc, d_sc, sizeof(sc), cudaMemcpyDeviceToHost));
        status[with_spec] = sc.status;
        raw[with_spec].resize(raw_bytes);
        CK(cudaMemcpy(raw[with_spec].data(), d_raw, raw_bytes, cudaMemcpyDeviceToHost));
    }
    std::vector<uint32_t> spec(bsg::inflate_spec_words(int(n)));
    CK(cudaMemcpy(spec.data(), d_spec, spec.size() * 4, cudaMemcpyDeviceToHost));
    FILE* o = fopen(out_path, "wb");
    if (!o) { perror(out_path); return 1; }
    const uint32_t same = raw[0] == raw[1] ? 1u : 0u;
    fwrite(status, 4, 2, o);
    fwrite(&same, 4, 1, o);
    fwrite(raw[1].data(), 1, raw_bytes, o);
    for (uint32_t b = 0; b < n; ++b) {
        const uint32_t cnt = spec[b], end = spec[n + b];
        fwrite(&cnt, 4, 1, o);
        fwrite(&end, 4, 1, o);
        if (cnt != bsg::kSpecNone) fwrite(spec.data() + 2 * size_t(n) + size_t(b) * bsg::kSpecStride, 4, cnt, o);
    }
    fclose(o);
    cudaFree(d_comp); cudaFree(d_raw); cudaFree(d_blocks); cudaFree(d_crc); cudaFree(d_spec); cudaFree(d_sc);
    return 0;
}

int main(int argc, char** argv) {
    if (argc < 3 || (argc - 1) % 2) { fprintf(stderr, "usage: %s in.bin out.bin [in.bin out.bin ...]\n", argv[0]); return 1; }
    for (int i = 1; i + 1 < argc; i += 2) {
        const int rc = run_one(argv[i], argv[i + 1]);
        if (rc) return rc;
    }
    return 0;
}
