// GFTT_ORB_B200 — rtabmap::Feature2D for Kp/DetectorStrategy=8 (GFTT/ORB, the reference's default) backed by liblcd_b200.so.
//
// Feature2D::create (corelib/src/Features2d.cpp:617) gets one more case: `case Feature2D::kFeatureGfttOrb: return gpu ? new GFTT_ORB_B200(p) :
// new GFTT_ORB(p);`.  The reference's GFTT_ORB detects with cv::GFTTDetector (GFTT::generateKeypointsImpl, Features2d.cpp:2148-2178) and
// describes with cv::ORB::compute (GFTT_ORB::generateDescriptorsImpl, :2351-2355); the engine does both in one pass
// (lcd_set_detector(LCD_DETECTOR_GFTT_ORB)), so, as in ORB_B200, the descriptors of the last detection are handed out when
// generateDescriptorsImpl is called for the same keypoints.  ORB::compute drops the corners within ORB/EdgeThreshold of the border:
// the keypoints returned here are already the ones that keep a descriptor.
#include <rtabmap/core/Features2d.h>
#include <rtabmap/utilite/ULogger.h>
#include "lcd_b200.h"

namespace rtabmap {

class GFTT_ORB_B200 : public Feature2D
{
public:
	explicit GFTT_ORB_B200(const ParametersMap & parameters = ParametersMap()) : Feature2D(parameters), e_(0), n_(0)
	{
		p_.n_features = 1000; p_.n_levels = 1; p_.scale_factor = 2.0f; p_.edge_threshold = 19; p_.fast_threshold = 20; p_.patch_size = 31;
		p_.min_depth = 0; p_.max_depth = 0; p_.depth_as_mask = 1; p_.fx = p_.fy = 1; p_.cx = p_.cy = 0;
		g_.quality_level = 0.001; g_.min_distance = 7; g_.block_size = 3; g_.use_harris = 0; g_.k = 0.04;
		lcd_config c;
		c.device = 0; c.desc_type = LCD_DESC_U8; c.desc_dim = 32; c.max_words = 1024; c.max_signatures = 1024; c.max_queries = 4096; c.max_batch = 1;
		e_ = lcd_create(&c);
		if (!e_) UERROR("B200 GFTT/ORB engine: %s", lcd_last_error(0));
		parseParameters(parameters);
	}
	~GFTT_ORB_B200() override { lcd_destroy(e_); }
	Feature2D::Type getType() const override { return kFeatureGfttOrb; }

	void parseParameters(const ParametersMap & parameters) override
	{
		Feature2D::parseParameters(parameters);
		Parameters::parse(parameters, "GFTT/QualityLevel", g_.quality_level);  // Parameters.h:313
		Parameters::parse(parameters, "GFTT/MinDistance", g_.min_distance);    // :314
		Parameters::parse(parameters, "GFTT/BlockSize", g_.block_size);        // :315
		bool harris = g_.use_harris != 0;
		Parameters::parse(parameters, "GFTT/UseHarrisDetector", harris);       // :316
		g_.use_harris = harris ? 1 : 0;
		Parameters::parse(parameters, "GFTT/K", g_.k);                         // :317
		Parameters::parse(parameters, "ORB/EdgeThreshold", p_.edge_threshold); // :322
		Parameters::parse(parameters, "ORB/PatchSize", p_.patch_size);        // :326
		p_.n_features = getMaxFeatures();
		if (e_ && lcd_set_detector(e_, LCD_DETECTOR_GFTT_ORB, &g_) != LCD_OK) UERROR("%s", lcd_last_error(e_));
	}

private:
	std::vector<cv::KeyPoint> generateKeypointsImpl(const cv::Mat & image, const cv::Rect & roi, const cv::Mat & mask) override
	{
		std::vector<cv::KeyPoint> out;
		if (!e_ || image.empty()) return out;
		if (roi.x != 0 || roi.y != 0 || roi.width != image.cols || roi.height != image.rows)
		{
			UERROR("GFTT_ORB_B200 works on whole images (Kp/RoiRatios and Kp/GridRows/Cols must stay at their defaults)");
			return out;
		}
		const int cap = p_.n_features;
		std::vector<lcd_keypoint> kp(cap);
		desc_ = cv::Mat(cap, 32, CV_8U);
		const int rc = lcd_orb_detect_describe(e_, 1, image.data, image.cols, image.rows, image.channels(), mask.empty() ? 0 : mask.data,
		                                       mask.empty() ? LCD_DEPTH_NONE : LCD_DEPTH_MASK_U8, &p_, cap, kp.data(), desc_.data, 0, &n_);
		if (rc != LCD_OK)
		{
			UERROR("%s", lcd_last_error(e_));
			n_ = 0;
			return out;
		}
		out.resize(n_);
		for (int i = 0; i < n_; ++i)
		{
			out[i].pt.x = kp[i].x; out[i].pt.y = kp[i].y; out[i].size = kp[i].size; out[i].angle = kp[i].angle;
			out[i].response = kp[i].response; out[i].octave = kp[i].octave;
		}
		return out;
	}

	cv::Mat generateDescriptorsImpl(const cv::Mat &, std::vector<cv::KeyPoint> & keypoints) const override
	{
		if ((int)keypoints.size() != n_) UWARN("GFTT_ORB_B200: descriptors requested for %d keypoints, the last detection found %d", (int)keypoints.size(), n_);
		return n_ ? desc_.rowRange(0, n_) : cv::Mat();
	}

	lcd_engine * e_;
	lcd_orb_params p_;
	lcd_gftt_params g_;
	cv::Mat desc_;
	int n_;
};

Feature2D * createGfttOrbB200(const ParametersMap & parameters) { return new GFTT_ORB_B200(parameters); }

} // namespace rtabmap
