// v2p::VcfText::load_bgzf (include/v2p_host.hpp) end to end: a bgzip'd VCF -> inflated text, line table and columns 1-9
// on the host -> FORMAT/BCSQ mask matrix on the device.  The file is written here with stored DEFLATE blocks (no zlib).
// `vcf_bgzf_host_test --no-gpu` only checks that the mirror compiles and links; without the flag it needs a GPU.
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "v2p_host.hpp"

#define CHECK(c)                                                        \
    do {                                                                \
        if (!(c)) {                                                     \
            std::printf("FAIL %s:%d: %s\n", __FILE__, __LINE__, #c);   \
            return 1;                                                   \
        }                                                               \
    } while (0)

static uint32_t crc32(const std::string& s) {
    uint32_t c = 0xFFFFFFFFu;
    for (unsigned char b : s) {
        c ^= b;
        for (int k = 0; k < 8; ++k) c = (c >> 1) ^ ((c & 1u) ? 0xEDB88320u : 0u);
    }
    return ~c;
}

static void put16(std::string& o, uint32_t v) { o += (char)(v & 255), o += (char)(v >> 8 & 255); }
static void put32(std::string& o, uint32_t v) { put16(o, v & 0xffff), put16(o, v >> 16); }

// one BGZF block holding `raw` as a single final stored DEFLATE block
static std::string block(const std::string& raw) {
    std::string o = std::string("\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0", 16);
    put16(o, (uint32_t)(18 + 5 + raw.size() + 8 - 1));
    o += '\x01';
    put16(o, (uint32_t)raw.size()), put16(o, ~(uint32_t)raw.size() & 0xffff);
    o += raw;
    put32(o, crc32(raw)), put32(o, (uint32_t)raw.size());
    return o;
}

int main(int argc, char** argv) {
    if (argc > 1 && std::strcmp(argv[1], "--no-gpu") == 0) {
        std::printf("OK (host only)\n");
        return 0;
    }
    const std::string hdr = "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tNA1\tNA2\tNA3";
    const std::string text = "##fileformat=VCFv4.2\r\n" + hdr + "\r\n" +
                             "1\t100\t.\tC\tT\t.\t.\tBCSQ=a,b\tGT:BCSQ\t0|1:2\t1|1:3,1\t0|0:0\n" +
                             "1\t101\t.\tC\tT\t.\t.\tBCSQ=c\tGT:AD:BCSQ\t1|0:4,4:1\t5\t0\n";
    // blocks cut inside the #CHROM line and inside a cell, then the EOF block
    const size_t cut1 = 40, cut2 = text.find("3,1") + 1;
    const std::string eof("\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0\x1b\0\x03\0\0\0\0\0\0\0\0\0", 28);
    const std::string gz = block(text.substr(0, cut1)) + block(text.substr(cut1, cut2 - cut1)) + block(text.substr(cut2)) + eof;
    v2p::VcfText vcf(0);
    const v2p_vcf_lines& ix = vcf.load_bgzf(gz);
    const v2p_vcf_bgzf& bz = vcf.bgzf();
    CHECK(ix.n_samples == 3 && ix.n_lines == 2 && bz.n_blocks == 4 && bz.text_bytes == text.size() && ix.h2d_bytes == gz.size());
    CHECK(std::string(reinterpret_cast<const char*>(bz.head), ix.header_end) == text.substr(0, ix.header_end));
    CHECK((vcf.sample_names() == std::vector<std::string>{"NA1", "NA2", "NA3"}));
    CHECK(vcf.fixed(1) == "1\t101\t.\tC\tT\t.\t.\tBCSQ=c\tGT:AD:BCSQ\t");
    std::string back(text.size(), '\0');
    CHECK(v2p_device_read(&back[0], bz.text, back.size()) == V2P_OK && back == text);
    const v2p_vcf_masks m = vcf.parse_masks({1, 0});
    CHECK((v2p::VcfText::read(m) == std::vector<uint32_t>{1, 0, 5, 0, 0, 0, 2, 0, 3, 1, 0, 0}));
    std::string bad = gz;
    bad[bad.size() - 28 - 8] ^= 1;  // the last data block's CRC
    bool threw = false;
    try {
        vcf.load_bgzf(bad);
    } catch (const v2p::EngineError& e) {
        const std::string want = "BGZF block 2 at byte " + std::to_string(gz.size() - 28 - (text.size() - cut2) - 5 - 18 - 8) + ": CRC-32";
        threw = e.status == V2P_ERR_BGZF && std::string(e.what()).find(want) != std::string::npos;
    }
    CHECK(threw);
    threw = false;
    try {
        vcf.load_bgzf(text);
    } catch (const v2p::EngineError& e) {
        threw = e.status == V2P_ERR_BGZF && std::string(e.what()).find("not BGZF: recompress with bgzip") != std::string::npos;
    }
    CHECK(threw);
    CHECK(vcf.load_bgzf(gz).n_lines == 2 && vcf.parse_masks({0}).words_per_cell == 2);  // usable after the errors
    CHECK(vcf.load(text).n_lines == 2 && vcf.bgzf().n_blocks == 0);
    std::printf("OK\n");
    return 0;
}
