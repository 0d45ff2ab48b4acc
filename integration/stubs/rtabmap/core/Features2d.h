// rtabmap::Feature2D — the interface ORB_B200 implements (corelib/include/rtabmap/core/Features2d.h:115-260).
#pragma once
#include <vector>
#include <opencv2/core.hpp>
#include <rtabmap/core/Parameters.h>
namespace rtabmap {
class Feature2D
{
public:
	enum Type { kFeatureUndef = -1, kFeatureSurf = 0, kFeatureSift = 1, kFeatureOrb = 2, kFeatureGfttOrb = 8 };             // :117-134
	virtual ~Feature2D() {}                                                                             // :222
	int getMaxFeatures() const { return maxFeatures_; }                                                 // :214
	float getMinDepth() const { return _minDepth; }                                                     // :216
	float getMaxDepth() const { return _maxDepth; }                                                     // :217
	// the public, non-virtual entry points Memory::createSignature calls (:224-229): reduced here to the forwarding they end in
	std::vector<cv::KeyPoint> generateKeypoints(const cv::Mat & image, const cv::Mat & mask = cv::Mat()) { cv::Rect roi; roi.width = image.cols; roi.height = image.rows; return generateKeypointsImpl(image, roi, mask); }
	cv::Mat generateDescriptors(const cv::Mat & image, std::vector<cv::KeyPoint> & keypoints) const { return generateDescriptorsImpl(image, keypoints); }
	virtual void parseParameters(const ParametersMap & p) { Parameters::parse(p, "Kp/MaxFeatures", maxFeatures_); Parameters::parse(p, "Kp/MinDepth", _minDepth); Parameters::parse(p, "Kp/MaxDepth", _maxDepth); } // :234
	virtual Feature2D::Type getType() const = 0;                                                        // :236
protected:
	Feature2D(const ParametersMap & = ParametersMap()) {}                                               // :239
private:
	virtual std::vector<cv::KeyPoint> generateKeypointsImpl(const cv::Mat & image, const cv::Rect & roi, const cv::Mat & mask = cv::Mat()) = 0; // :242
	virtual cv::Mat generateDescriptorsImpl(const cv::Mat & image, std::vector<cv::KeyPoint> & keypoints) const = 0;                            // :243
	int maxFeatures_ = 500;
	float _maxDepth = 0, _minDepth = 0;
};
} // namespace rtabmap
