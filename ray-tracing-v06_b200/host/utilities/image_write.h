// image_write.h — the output stage after the renderer: PNG / PPM (8-bit) and PFM (float) writers, and the PFM reader
// that loads environment maps.
//
// The reference writes a JPG through stb_image_write (write_renderbuffer, main/src/FirstApp.cpp:108-122: uint8 =
// value * 255.999f, RGB, stbi_flip_vertically_on_write(true), quality 95).  The vendored stb header is MSVC-only
// (sprintf_s), and a lossy format is a poor carrier for parity checks, so the lossless PNG is the 8-bit format here:
// written from scratch (zlib container with stored - uncompressed - deflate blocks, CRC-32, Adler-32), no dependency.
// The bytes themselves come from the device (rtb_download_rgb8: quantised and row-flipped on the GPU).
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

namespace rtb_host {

inline uint32_t crc32_update(uint32_t crc, const uint8_t* p, size_t n) {
	static uint32_t table[256]; static bool ready = false;
	if (!ready) {
		for (uint32_t i = 0; i < 256; ++i) { uint32_t c = i; for (int k = 0; k < 8; ++k) c = (c & 1u) ? 0xEDB88320u ^ (c >> 1) : c >> 1; table[i] = c; }
		ready = true;
	}
	for (size_t i = 0; i < n; ++i) crc = table[(crc ^ p[i]) & 0xFFu] ^ (crc >> 8);
	return crc;
}

// rgb: width * height * 3 bytes, row 0 = TOP row of the picture.
inline bool write_png(const std::string& path, uint32_t width, uint32_t height, const uint8_t* rgb) {
	FILE* f = fopen(path.c_str(), "wb");
	if (!f) return false;
	auto be32 = [](uint8_t* p, uint32_t v) { p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v; };
	auto chunk = [&](const char* type, const std::vector<uint8_t>& data) {
		uint8_t hdr[8]; be32(hdr, (uint32_t)data.size()); hdr[4] = type[0]; hdr[5] = type[1]; hdr[6] = type[2]; hdr[7] = type[3];
		fwrite(hdr, 1, 8, f);
		if (!data.empty()) fwrite(data.data(), 1, data.size(), f);
		uint32_t crc = crc32_update(0xFFFFFFFFu, hdr + 4, 4);
		if (!data.empty()) crc = crc32_update(crc, data.data(), data.size());
		uint8_t tail[4]; be32(tail, crc ^ 0xFFFFFFFFu); fwrite(tail, 1, 4, f);
	};
	static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
	fwrite(sig, 1, 8, f);
	std::vector<uint8_t> ihdr(13); be32(&ihdr[0], width); be32(&ihdr[4], height); ihdr[8] = 8; ihdr[9] = 2; ihdr[10] = 0; ihdr[11] = 0; ihdr[12] = 0;   // 8-bit RGB
	chunk("IHDR", ihdr);
	// raw scanlines: filter byte 0 + width * 3 bytes each
	const size_t row = 1 + (size_t)width * 3, raw_size = row * height;
	std::vector<uint8_t> raw(raw_size);
	for (uint32_t y = 0; y < height; ++y) { raw[y * row] = 0; for (size_t k = 0; k < (size_t)width * 3; ++k) raw[y * row + 1 + k] = rgb[(size_t)y * width * 3 + k]; }
	// zlib stream: header, stored deflate blocks of at most 65535 bytes, Adler-32 of the raw data
	std::vector<uint8_t> z; z.reserve(raw_size + raw_size / 65535 * 5 + 16);
	z.push_back(0x78); z.push_back(0x01);
	size_t pos = 0;
	do {
		const size_t n = raw_size - pos < 65535 ? raw_size - pos : 65535;
		z.push_back(pos + n == raw_size ? 1 : 0);
		z.push_back((uint8_t)(n & 0xFF)); z.push_back((uint8_t)(n >> 8)); z.push_back((uint8_t)(~n & 0xFF)); z.push_back((uint8_t)((~n >> 8) & 0xFF));
		z.insert(z.end(), raw.begin() + pos, raw.begin() + pos + n);
		pos += n;
	} while (pos < raw_size);
	uint32_t a = 1, b = 0;
	for (size_t i = 0; i < raw_size; ++i) { a = (a + raw[i]) % 65521u; b = (b + a) % 65521u; }
	uint8_t ad[4]; be32(ad, (b << 16) | a); z.insert(z.end(), ad, ad + 4);
	chunk("IDAT", z);
	chunk("IEND", {});
	return fclose(f) == 0;
}

// rgb: row 0 = TOP row.
inline bool write_ppm(const std::string& path, uint32_t width, uint32_t height, const uint8_t* rgb) {
	FILE* f = fopen(path.c_str(), "wb");
	if (!f) return false;
	fprintf(f, "P6\n%u %u\n255\n", width, height);
	fwrite(rgb, 1, (size_t)width * height * 3, f);
	return fclose(f) == 0;
}

// rgba: the float render buffer (row 0 = BOTTOM row, as PFM stores it); alpha is dropped.
inline bool write_pfm(const std::string& path, uint32_t width, uint32_t height, const float* rgba) {
	FILE* f = fopen(path.c_str(), "wb");
	if (!f) return false;
	fprintf(f, "PF\n%u %u\n-1.0\n", width, height);
	for (size_t i = 0; i < (size_t)width * height; ++i) fwrite(rgba + 4 * i, sizeof(float), 3, f);
	return fclose(f) == 0;
}

// PFM reader (colour "PF" or greyscale "Pf", either byte order): rgb = height rows x width x RGB with row 0 = TOP (PFM
// stores rows bottom-up, so they are flipped; a greyscale map is spread to three channels).  false with `err` set on a file
// that is missing, truncated or not a PFM.
inline bool read_pfm(const std::string& path, std::vector<float>& rgb, int& width, int& height, std::string& err) {
	FILE* f = fopen(path.c_str(), "rb");
	if (!f) { err = "cannot open " + path; return false; }
	char kind[3] = {0, 0, 0};
	double scale = 0.0;
	width = height = 0;
	const bool ok_header = fscanf(f, "%2s %d %d %lf", kind, &width, &height, &scale) == 4 && fgetc(f) != EOF;   // (one whitespace byte ends the header)
	const int ch = kind[0] == 'P' && kind[1] == 'F' ? 3 : (kind[0] == 'P' && kind[1] == 'f' ? 1 : 0);
	if (!ok_header || ch == 0 || width <= 0 || height <= 0 || scale == 0.0 || (int64_t)width * height > (int64_t(1) << 28)) {
		fclose(f); err = path + " is not a PFM image"; return false;
	}
	std::vector<float> raw((size_t)width * height * ch);
	const size_t got = fread(raw.data(), sizeof(float), raw.size(), f);
	fclose(f);
	if (got != raw.size()) { err = path + ": truncated PFM data"; return false; }
	if (scale > 0.0) {   // big-endian file
		for (float& v : raw) { uint32_t u; memcpy(&u, &v, 4); u = __builtin_bswap32(u); memcpy(&v, &u, 4); }
	}
	rgb.resize((size_t)width * height * 3);
	for (int y = 0; y < height; ++y)
		for (int x = 0; x < width; ++x)
			for (int c = 0; c < 3; ++c)
				rgb[((size_t)y * width + x) * 3 + c] = raw[((size_t)(height - 1 - y) * width + x) * ch + (ch == 3 ? c : 0)];
	return true;
}

// Binary PPM (P6, maxval 255) -> width x height x RGB8, row 0 = the top row of the picture (the row order image textures use).
inline bool read_ppm(const std::string& path, std::vector<uint8_t>& rgb, int& width, int& height, std::string& err) {
	FILE* f = fopen(path.c_str(), "rb");
	if (!f) { err = "cannot open " + path; return false; }
	auto field = [f](int& v) {   // the next decimal field of the header, skipping whitespace and # comments
		int c = fgetc(f);
		for (;;) {
			while (c == ' ' || c == '\t' || c == '\r' || c == '\n') c = fgetc(f);
			if (c != '#') break;
			while (c != '\n' && c != EOF) c = fgetc(f);
		}
		if (c < '0' || c > '9') return false;
		v = 0;
		for (; c >= '0' && c <= '9'; c = fgetc(f)) { v = v * 10 + (c - '0'); if (v > (1 << 20)) return false; }
		return c == ' ' || c == '\t' || c == '\r' || c == '\n';   // (one whitespace byte ends the header)
	};
	int maxval = 0;
	width = height = 0;
	const bool ok = fgetc(f) == 'P' && fgetc(f) == '6' && field(width) && field(height) && field(maxval);
	if (!ok || width <= 0 || height <= 0 || maxval != 255 || (int64_t)width * height > (int64_t(1) << 26)) {
		fclose(f); err = path + " is not a binary PPM (P6) image with 8-bit samples"; return false;
	}
	rgb.resize((size_t)width * height * 3);
	const size_t got = fread(rgb.data(), 1, rgb.size(), f);
	fclose(f);
	if (got != rgb.size()) { err = path + ": truncated PPM data"; return false; }
	return true;
}

inline bool has_suffix(const std::string& s, const char* suf) { const std::string t(suf); return s.size() >= t.size() && s.compare(s.size() - t.size(), t.size(), t) == 0; }

}  // namespace rtb_host
