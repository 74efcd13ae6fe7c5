// Host build of the BGZF block decoder (rala_b200/csrc/bgzf.cuh), the code lane 0 of k_bgzf_inflate runs, for the CPU
// suite (tests/test_bgzf_reader.py).  stdin: records of (u32 in_len, u32 isize, u32 crc, in_len bytes of raw DEFLATE);
// stdout per record: u32 status (a bgzf::BgzfError), then the isize output bytes when the status is 0.  Input and output
// sit at the very ends of their own heap buffers so that an out-of-bounds access lands outside them (run under
// valgrind or an ASan build to see it; the plain build checks the results).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../rala_b200/csrc/bgzf.cuh"

int main() {
    uint32_t table[256];
    for (uint32_t i = 0; i < 256; ++i) table[i] = bgzf::crc_table_entry(i);
    bgzf::Tables* t = new bgzf::Tables;
    uint32_t hdr[3];
    while (fread(hdr, 4, 3, stdin) == 3) {
        const uint32_t in_len = hdr[0], isize = hdr[1], crc = hdr[2];
        uint8_t* in = (uint8_t*) malloc(in_len ? in_len : 1);
        if (in_len && fread(in, 1, in_len, stdin) != in_len) return 2;
        uint8_t* out = (uint8_t*) malloc(isize ? isize : 1);
        uint32_t rc = bgzf::inflate(in, in_len, out, isize, *t);
        if (rc == bgzf::kOk && bgzf::crc_update(0, out, isize, table) != crc) rc = bgzf::kCrc;
        fwrite(&rc, 4, 1, stdout);
        if (rc == bgzf::kOk) fwrite(out, 1, isize, stdout);
        free(in);
        free(out);
    }
    delete t;
    return 0;
}
