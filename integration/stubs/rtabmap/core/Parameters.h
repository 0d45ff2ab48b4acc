// rtabmap::ParametersMap and the parse helpers the shims call (corelib/include/rtabmap/core/Parameters.h:61, :941-948).
#pragma once
#include <cstdlib>
#include <map>
#include <string>
namespace rtabmap {
typedef std::map<std::string, std::string> ParametersMap;
class Parameters
{
public:
	static bool parse(const ParametersMap & p, const std::string & key, int & v) { auto i = p.find(key); if (i == p.end()) return false; v = std::atoi(i->second.c_str()); return true; }
	static bool parse(const ParametersMap & p, const std::string & key, float & v) { auto i = p.find(key); if (i == p.end()) return false; v = static_cast<float>(std::atof(i->second.c_str())); return true; }
	static bool parse(const ParametersMap & p, const std::string & key, double & v) { auto i = p.find(key); if (i == p.end()) return false; v = std::atof(i->second.c_str()); return true; }
	static bool parse(const ParametersMap & p, const std::string & key, bool & v) { auto i = p.find(key); if (i == p.end()) return false; v = i->second == "true" || i->second == "1"; return true; }
};
} // namespace rtabmap
