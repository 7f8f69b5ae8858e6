// TEST INFRASTRUCTURE — stand-in for Thirdparty/DBoW2/DBoW2/BowVector.h (a std::map from word id to word value), used when the frame
// drop-in is compiled without the reference tree (tests/cpp/shim_frame).
#pragma once
#include <map>
namespace DBoW2 {
typedef unsigned int WordId;
typedef double WordValue;
class BowVector : public std::map<WordId, WordValue> {};
}  // namespace DBoW2
