// Per-stream mode of the decode-core harness: the same inflate_block (tests/host_inflate_harness.cpp, compiled in here with
// its main() renamed) over a corpus of raw DEFLATE streams (tests/deflate_forge.py write_corpus: <u32 in_len><u32 isize>
// <u32 crc><bytes> per case).  Every stream is decoded from a private buffer with the device buffer's 4096 bytes of
// slack, starting at every byte phase 0-7 of the 64-bit bit-reader units; one line per case and phase:
//   case <i> phase <p> rc <rc> crc <crc32 of the ISIZE output bytes>
//   usage: host_inflate_cases corpus.bin
#define main host_inflate_harness_main
#include "host_inflate_harness.cpp"
#undef main

int main(int argc, char** argv) {
    if (argc < 2) return 2;
    FILE* f = fopen(argv[1], "rb");
    if (!f) return 2;
    std::vector<uint8_t> d;
    uint8_t tmp[65536];
    size_t k;
    while ((k = fread(tmp, 1, sizeof tmp, f)) > 0) d.insert(d.end(), tmp, tmp + k);
    fclose(f);
    int idx = 0;
    for (size_t off = 0; off + 12 <= d.size(); ++idx) {
        uint32_t in_len, isize, crc;
        memcpy(&in_len, d.data() + off, 4);
        memcpy(&isize, d.data() + off + 4, 4);
        memcpy(&crc, d.data() + off + 8, 4);
        if (off + 12 + in_len > d.size()) return 2;
        for (uint32_t phase = 0; phase < 8; ++phase) {
            std::vector<uint64_t> buf((size_t(phase) + in_len + 4096 + 7) / 8, 0);
            uint8_t* b8 = reinterpret_cast<uint8_t*>(buf.data());
            memcpy(b8 + phase, d.data() + off + 12, in_len);
            std::vector<uint8_t> out(size_t(isize) + 64, 0);
            const int rc = inflate_block(b8, phase, in_len, out.data(), isize);
            printf("case %d phase %u rc %d crc %u\n", idx, phase, rc, uint32_t(crc32(crc32(0, nullptr, 0), out.data(), isize)));
        }
        off += 12 + in_len;
    }
    return 0;
}
