// tests/emu/encode_sha256_emu.cc -- TEST INFRASTRUCTURE ONLY.
// Prints the SHA-256 of the frame the emulated encode path (K5 fragment compressor, K6 plan + place) makes for every case
// of test_encode_emu.cc, with the fragment index and the chunk offset table each on and off, in every thread resume order
// of the emulator.  tests/test_encode_bytes.py compares them with digests recorded from an earlier build, so a change that
// is meant to rearrange the encoder's work, not its output, is checked byte for byte.
// The encode path (gpu_encode) is test_encode_emu.cc's own, so both programs run the kernels the same way; the inputs and
// the case list below are that program's, in the same order, from the same seed.
//   usage: encode_sha256_emu [modes]      one line per frame: "sha256 <mode> <case>[+index][+offsets] <hex digest>"
#define main test_encode_emu_main
#include "test_encode_emu.cc"
#undef main

// SHA-256 (FIPS 180-4) of a frame, as lowercase hex
static std::string sha256_hex(const std::vector<uint8_t> &msg)
{
    static const uint32_t K[64] = {
        0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5, 0xd807aa98, 0x12835b01, 0x243185be,
        0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc, 0x2de92c6f, 0x4a7484aa,
        0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147, 0x06ca6351, 0x14292967, 0x27b70a85,
        0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85, 0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3,
        0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116, 0x1e376c08, 0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f,
        0x682e6ff3, 0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208, 0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};
    uint32_t h[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
    std::vector<uint8_t> m = msg;
    const uint64_t bits = 8ull * msg.size();
    m.push_back(0x80);
    while (m.size() % 64 != 56) m.push_back(0);
    for (int i = 7; i >= 0; i--) m.push_back((uint8_t)(bits >> (8 * i)));
    auto rotr = [](uint32_t x, int n) { return (x >> n) | (x << (32 - n)); };
    for (size_t at = 0; at < m.size(); at += 64) {
        uint32_t w[64];
        for (int i = 0; i < 16; i++) w[i] = (uint32_t)m[at + 4 * i] << 24 | (uint32_t)m[at + 4 * i + 1] << 16 | (uint32_t)m[at + 4 * i + 2] << 8 | m[at + 4 * i + 3];
        for (int i = 16; i < 64; i++) {
            const uint32_t s0 = rotr(w[i - 15], 7) ^ rotr(w[i - 15], 18) ^ (w[i - 15] >> 3), s1 = rotr(w[i - 2], 17) ^ rotr(w[i - 2], 19) ^ (w[i - 2] >> 10);
            w[i] = w[i - 16] + s0 + w[i - 7] + s1;
        }
        uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
        for (int i = 0; i < 64; i++) {
            const uint32_t t1 = hh + (rotr(e, 6) ^ rotr(e, 11) ^ rotr(e, 25)) + ((e & f) ^ (~e & g)) + K[i] + w[i];
            const uint32_t t2 = (rotr(a, 2) ^ rotr(a, 13) ^ rotr(a, 22)) + ((a & b) ^ (a & c) ^ (b & c));
            hh = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
        }
        h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += hh;
    }
    char hex[65];
    for (int i = 0; i < 8; i++) snprintf(hex + 8 * i, 9, "%08x", h[i]);
    return std::string(hex, 64);
}

int main(int argc, char **argv)
{
    const int modes = argc > 1 ? atoi(argv[1]) : 3;
    std::mt19937 rng(777);
    // a 256x128 picture with gradients + noise + bars, block-compressed by the oracle
    const int W = 256, H = 128;
    std::vector<uint8_t> img(W * H * 4);
    for (int y = 0; y < H; y++)
        for (int x = 0; x < W; x++) {
            uint8_t *p = &img[4 * (y * W + x)];
            bool bar = y < 16 || y >= H - 16;
            for (int c = 0; c < 3; c++) p[c] = bar ? 16 : (uint8_t)(40 + (x * (c + 1)) % 160 + (y * 3) % 40 + (rng() % 4));
            p[3] = (uint8_t)(x);
        }
    auto blocks = [&](int kind) {
        std::vector<uint8_t> b((W / 4) * (H / 4) * (kind == 0 || kind == 3 ? 8 : 16));
        if (kind == 0) orc_bc1_encode_clusterfit(img.data(), W, H, b.data(), 1);
        else if (kind == 1) orc_bc3_encode_clusterfit(img.data(), W, H, b.data(), 1);
        else if (kind == 2) orc_ycocg_dxt5_encode_clusterfit(img.data(), W, H, b.data(), 1);
        else orc_bc4_encode_squish(img.data(), W, H, 3, b.data());
        return b;
    };
    std::vector<uint8_t> dxt1 = blocks(0), dxt5 = blocks(1), ycocg = blocks(2), rgtc = blocks(3);
    std::vector<uint8_t> noise(70000 - 70000 % 16), flat(16 * 5000);
    for (auto &b : noise) b = (uint8_t)rng();
    for (size_t i = 0; i < flat.size(); i++) flat[i] = (uint8_t)(0x30 + (i % 16));
    // bigger than one fragment, so chunk streams are concatenations of fragment streams
    std::vector<uint8_t> big;
    for (int r = 0; r < 5; r++) big.insert(big.end(), ycocg.begin(), ycocg.end());
    for (size_t i = 0; i < big.size(); i += 977) big[i] ^= (uint8_t)rng();

    struct Case { std::string name; std::vector<Tex> tex; };
    std::vector<Case> cases = {
        {"dxt1_1chunk", {{dxt1, 0x83F0, 1, 1}}},
        {"dxt1_3chunks", {{dxt1, 0x83F0, 1, 3}}},
        {"dxt5_4chunks", {{dxt5, 0x83F3, 1, 4}}},
        {"ycocg_8chunks", {{ycocg, 0x01, 1, 8}}},
        {"ycocg_limit_7_to_x", {{ycocg, 0x01, 1, 7}}},
        {"rgtc_2chunks", {{rgtc, 0x8DBB, 1, 2}}},
        {"hapm", {{ycocg, 0x01, 1, 4}, {rgtc, 0x8DBB, 1, 2}}},
        {"hapm_mixed_none", {{ycocg, 0x01, 0, 4}, {rgtc, 0x8DBB, 1, 2}}},
        {"none_single", {{dxt5, 0x83F3, 0, 5}}},
        {"none_pair", {{ycocg, 0x01, 0, 1}, {rgtc, 0x8DBB, 0, 1}}},
        {"noise_fallback_whole", {{noise, 0x83F3, 1, 2}}},
        {"flat_rle", {{flat, 0x01, 1, 2}}},
        {"big_multi_fragment", {{big, 0x01, 1, 2}}},
        {"big_1chunk", {{big, 0x8E8C, 1, 1}}},
        {"tiny_16", {{std::vector<uint8_t>(16, 0x55), 0x01, 1, 1}}},
        {"tiny_8", {{std::vector<uint8_t>(8, 0x11), 0x83F0, 1, 1}}},
        {"kat_a_64x55", {{std::vector<uint8_t>(64, 0x55), 0x83F0, 1, 1}}},
    };
    // per-chunk fallback: half compressible, half noise, two chunks
    {
        std::vector<uint8_t> mix(ycocg.begin(), ycocg.begin() + 16384);
        mix.insert(mix.end(), noise.begin(), noise.begin() + 16384);
        cases.push_back({"mixed_chunk_fallback", {{mix, 0x01, 1, 2}}});
    }
    // random shapes: sizes that are not multiples of the fragment or of the chunk count, 1..9 chunks, content
    // stitched from picture blocks, repeated blocks, flat runs and noise (exercises partial fragments, chunk-count
    // limiting, both fallbacks and the persistent grid's striding in combinations no hand-made case has)
    for (int r = 0; r < 8; r++) {
        const size_t blocks16 = 200 + rng() % 12000;
        std::vector<uint8_t> v;
        while (v.size() < blocks16 * 16) {
            const int what = rng() % 5;
            const size_t n = 16 * (1 + rng() % 700);
            if (what == 0) { size_t at = (rng() % (ycocg.size() / 16 - n / 16 - 1)) * 16; v.insert(v.end(), ycocg.begin() + at, ycocg.begin() + at + n); }
            else if (what == 1 && v.size() >= 4096) { size_t at = v.size() - 16 * (1 + rng() % 200); for (size_t i = 0; i < n; i++) v.push_back(v[at + i % 16]); }
            else if (what == 2) { uint8_t b16[16]; for (auto &b : b16) b = (uint8_t)rng(); for (size_t i = 0; i < n; i++) v.push_back(b16[i % 16]); }
            else if (what == 3) { for (size_t i = 0; i < n; i++) v.push_back((uint8_t)rng()); }
            else { for (size_t i = 0; i < n; i++) v.push_back((uint8_t)((i / 16) & 0xFF)); }
        }
        v.resize(blocks16 * 16);
        cases.push_back({"random_" + std::to_string(r), {{v, 0x01, 1, (unsigned)(1 + rng() % 9)}}});
    }
    static const char *const kVariant[4] = {"", "+index", "+offsets", "+index+offsets"};
    for (int mode = 0; mode < modes; mode++)
        for (auto &c : cases)
            for (uint32_t wi = 0; wi < 4; wi++)
                printf("sha256 %d %s%s %s\n", mode, c.name.c_str(), kVariant[wi], sha256_hex(gpu_encode(c.tex, mode, wi)).c_str());
    return 0;
}
