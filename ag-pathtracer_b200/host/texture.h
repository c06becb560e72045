// host/texture.h -- HDRTexture with the reference's surface (/root/reference/texture.h:41-84):
// a lat-long float RGB image loaded from a Radiance .hdr file.  Upstream decodes with
// stb_image's stbi_loadf; this is an independent reader of the same format (header, flat or
// new-style RLE scanlines, RGBE -> float as byte * 2^(e-136)), so both sides see the same floats.
// Lookups (HDRTexture::value, texture.h:59-67) happen on the device.
#pragma once

#include <cstdio>
#include <stdexcept>

#include "precomp.h"
#include "agpt.h"

class Texture {
public:
	virtual ~Texture() {}
};

class HDRTexture : public Texture {
public:
	HDRTexture(const std::string& filename) {
		FILE* f = fopen(filename.c_str(), "rb");
		if (!f) return;                       // like upstream, a missing file leaves an empty texture
		bool ok = ReadHeader(f) && ReadPixels(f);
		fclose(f);
		if (!ok) { width = height = 0; rgb.clear(); }
	}
	int Width() const { return width; }
	int Height() const { return height; }
	float3 GetPixel(int x, int y) const { const float* p = &rgb[3 * ((size_t)y * width + x)]; return float3(p[0], p[1], p[2]); }
	const std::vector<float>& Data() const { return rgb; }

private:
	bool ReadHeader(FILE* f) {
		char line[256];
		if (!fgets(line, sizeof(line), f)) return false;
		if (strncmp(line, "#?RADIANCE", 10) != 0 && strncmp(line, "#?RGBE", 6) != 0) return false;
		bool format = false;
		while (fgets(line, sizeof(line), f)) {
			if (line[0] == '\n' || line[0] == '\r') break;
			if (strncmp(line, "FORMAT=32-bit_rle_rgbe", 22) == 0) format = true;
		}
		if (!format) return false;
		if (!fgets(line, sizeof(line), f)) return false;
		return sscanf(line, "-Y %d +X %d", &height, &width) == 2 && width > 0 && height > 0;
	}
	static void Decode(const unsigned char* p, float* out) {
		if (p[3] == 0) { out[0] = out[1] = out[2] = 0.f; return; }
		float scale = (float)ldexp(1.0f, (int)p[3] - (128 + 8));
		out[0] = p[0] * scale; out[1] = p[1] * scale; out[2] = p[2] * scale;
	}
	bool ReadPixels(FILE* f) {
		rgb.assign((size_t)width * height * 3, 0.f);
		std::vector<unsigned char> scan((size_t)width * 4);
		for (int y = 0; y < height; y++) {
			unsigned char head[4];
			if (fread(head, 1, 4, f) != 4) return false;
			bool rle = width >= 8 && width < 32768 && head[0] == 2 && head[1] == 2 && !(head[2] & 0x80);
			if (!rle) {
				// flat: the four bytes are the first pixel
				memcpy(&scan[0], head, 4);
				size_t rest = (size_t)(y == 0 ? width : width) * 4 - 4;
				if (fread(&scan[4], 1, rest, f) != rest) return false;
			}
			else {
				if (((head[2] << 8) | head[3]) != width) return false;
				for (int c = 0; c < 4; c++) {
					int x = 0;
					while (x < width) {
						int count = fgetc(f);
						if (count == EOF) return false;
						if (count > 128) {
							int value = fgetc(f);
							count -= 128;
							if (value == EOF || x + count > width) return false;
							while (count--) scan[(size_t)(x++) * 4 + c] = (unsigned char)value;
						}
						else {
							if (count == 0 || x + count > width) return false;
							while (count--) { int v = fgetc(f); if (v == EOF) return false; scan[(size_t)(x++) * 4 + c] = (unsigned char)v; }
						}
					}
				}
			}
			for (int x = 0; x < width; x++) Decode(&scan[(size_t)x * 4], &rgb[3 * ((size_t)y * width + x)]);
		}
		return true;
	}

	int width = 0, height = 0;
	std::vector<float> rgb;
};

// EXTENSION (not a reference class: upstream has one colour per material): a linear RGB float image supplied by the
// caller, the base colour of a DisneyMaterial.  Lookups happen on the device (include/agpt.h agpt_upload_textures).
class ImageTexture : public Texture {
public:
	ImageTexture(int width, int height, std::vector<float> rgb) : width(width), height(height), rgb(std::move(rgb)) {
		if (width < 1 || height < 1 || this->rgb.size() != 3 * (size_t)width * height) throw std::runtime_error("ImageTexture: need width, height >= 1 and width * height * 3 floats");
	}
	int Width() const { return width; }
	int Height() const { return height; }
	agpt_texture Export() const { agpt_texture t; t.width = width; t.height = height; t.rgb = rgb.data(); return t; }
	static std::shared_ptr<ImageTexture> Make(int width, int height, std::vector<float> rgb) { return std::make_shared<ImageTexture>(width, height, std::move(rgb)); }

private:
	int width, height;
	std::vector<float> rgb;
};

