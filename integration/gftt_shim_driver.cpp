// gftt_shim_driver.cpp — runs GFTT_ORB_B200 the way Memory::createSignature drives a Feature2D (generateKeypoints with the depth mask,
// then generateDescriptors for the keypoints it returned) on one raw 8-bit gray image, and writes what came out.
// usage: gftt_shim_driver IMAGE.raw WIDTH HEIGHT MASK.raw|- MAX_FEATURES OUT.bin
// OUT.bin: int32 n, n x 6 float32 (x, y, size, angle, response, octave), n x 32 descriptor bytes.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>
#include <rtabmap/core/Features2d.h>

namespace rtabmap {
Feature2D * createGfttOrbB200(const ParametersMap & parameters);
}

static bool read_file(const char * path, std::vector<unsigned char> & out, size_t bytes)
{
	FILE * f = std::fopen(path, "rb");
	if (!f) return false;
	out.resize(bytes);
	const size_t got = std::fread(out.data(), 1, bytes, f);
	std::fclose(f);
	return got == bytes;
}

int main(int argc, char ** argv)
{
	if (argc != 7)
	{
		std::fprintf(stderr, "usage: %s IMAGE.raw WIDTH HEIGHT MASK.raw|- MAX_FEATURES OUT.bin\n", argv[0]);
		return 2;
	}
	const int w = std::atoi(argv[2]), h = std::atoi(argv[3]);
	std::vector<unsigned char> img, msk;
	if (w <= 0 || h <= 0 || !read_file(argv[1], img, static_cast<size_t>(w) * h)) return 2;
	const bool has_mask = std::string(argv[4]) != "-";
	if (has_mask && !read_file(argv[4], msk, static_cast<size_t>(w) * h)) return 2;
	rtabmap::ParametersMap p;
	p["Kp/MaxFeatures"] = argv[5];
	rtabmap::Feature2D * det = rtabmap::createGfttOrbB200(p);
	if (det->getType() != rtabmap::Feature2D::kFeatureGfttOrb) return 3;
	cv::Mat image(h, w, CV_8U, img.data());
	cv::Mat mask = has_mask ? cv::Mat(h, w, CV_8U, msk.data()) : cv::Mat();
	std::vector<cv::KeyPoint> kps = det->generateKeypoints(image, mask);
	cv::Mat desc = det->generateDescriptors(image, kps);
	FILE * f = std::fopen(argv[6], "wb");
	if (!f) return 2;
	const int n = static_cast<int>(kps.size());
	std::fwrite(&n, sizeof(int), 1, f);
	for (const cv::KeyPoint & k : kps)
	{
		const float row[6] = {k.pt.x, k.pt.y, k.size, k.angle, k.response, static_cast<float>(k.octave)};
		std::fwrite(row, sizeof(float), 6, f);
	}
	if (n) std::fwrite(desc.data, 1, static_cast<size_t>(n) * 32, f);
	std::fclose(f);
	delete det;
	std::printf("gftt shim driver ok: %d keypoints\n", n);
	return 0;
}
