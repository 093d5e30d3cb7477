// v2p::VcfText (include/v2p_host.hpp) end to end: VCF text -> line table -> FORMAT/BCSQ mask matrix on the device.
// `vcf_host_test --no-gpu` only checks that the mirror compiles and links; without the flag it needs a GPU.
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

int main(int argc, char** argv) {
    if (argc > 1 && std::strcmp(argv[1], "--no-gpu") == 0) {
        std::printf("OK (host only)\n");
        return 0;
    }
    const std::string hdr = "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tNA1\tNA2\tNA3";
    const std::string text = "##fileformat=VCFv4.2\r\n" + hdr + "\r\n" +
                             "1\t100\t.\tC\tT\t.\t.\tBCSQ=a,b\tGT:BCSQ\t0|1:2\t1|1:3,1\t0|0:0\r\n\r\n" +
                             "1\t101\t.\tC\tT\t.\t.\tBCSQ=c\tGT:AD:BCSQ\t1|0:4,4:1\t5\t0\n" +
                             "1\t102\t.\tC\tT\t.\t.\tBCSQ=d\tGT:BCSQ\t1\t2\tx";  // malformed third cell, no final newline
    v2p::VcfText vcf(0);
    const v2p_vcf_lines& ix = vcf.load(text);
    CHECK(ix.n_samples == 3 && ix.n_lines == 3);
    CHECK(text.substr(ix.header_begin, ix.header_end - ix.header_begin) == hdr);
    CHECK((vcf.sample_names() == std::vector<std::string>{"NA1", "NA2", "NA3"}));
    CHECK(text.substr(ix.line_begin[1], ix.cells_begin[1] - ix.line_begin[1]) == "1\t101\t.\tC\tT\t.\t.\tBCSQ=c\tGT:AD:BCSQ\t");
    const v2p_vcf_masks m = vcf.parse_masks({1, 0});
    CHECK(m.n_records == 2 && m.n_samples == 3 && m.words_per_cell == 2);
    const std::vector<uint32_t> got = v2p::VcfText::read(m);
    CHECK((got == std::vector<uint32_t>{1, 0, 5, 0, 0, 0, 2, 0, 3, 1, 0, 0}));
    bool threw = false;
    try {
        vcf.parse_masks({2});
    } catch (const v2p::EngineError& e) {
        threw = e.status == V2P_ERR_VCF_PARSE && std::string(e.what()).find("line 6, sample column 3") != std::string::npos;
    }
    CHECK(threw);
    CHECK(vcf.parse_masks({0}).words_per_cell == 2);  // usable after the error
    std::printf("OK\n");
    return 0;
}
