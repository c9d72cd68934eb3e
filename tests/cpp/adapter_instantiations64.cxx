// Compile-and-run check of the drop-in header for the 64-bit integer pixel types (tests/test_int64_oracle.py): the
// filter instantiates for long, unsigned long, long long and unsigned long long (ITK's IdentifierType is unsigned long),
// each maps to the pixel code of its size and signedness, and the codes of the other types are the ones they had.
#include <type_traits>
#include <vector>

#include "itkImage.h"
#include "itkMesh.h"
#include "itkCuberilleImageToMeshFilter.h"

template <typename T>
constexpr int Code() { return itk::cuberille_detail::PixelCode<T>::value; }

template <typename T>
constexpr int Expected() { return sizeof( T ) == 8 ? ( std::is_signed<T>::value ? CUB_I64 : CUB_U64 )
                                                   : ( std::is_signed<T>::value ? CUB_I32 : CUB_U32 ); }

static_assert( Code<long>() == Expected<long>() && Code<unsigned long>() == Expected<unsigned long>(), "long" );
static_assert( Code<long long>() == CUB_I64 && Code<unsigned long long>() == CUB_U64, "long long" );
static_assert( Code<unsigned char>() == CUB_U8 && Code<signed char>() == CUB_I8, "8-bit" );
static_assert( Code<char>() == ( std::is_signed<char>::value ? CUB_I8 : CUB_U8 ), "char" );
static_assert( Code<unsigned short>() == CUB_U16 && Code<short>() == CUB_I16, "16-bit" );
static_assert( Code<unsigned int>() == CUB_U32 && Code<int>() == CUB_I32, "32-bit" );
static_assert( Code<float>() == CUB_F32 && Code<double>() == CUB_F64, "float" );

template <typename TPixel, typename TMeshPixel>
int Instantiate()
{
  typedef itk::CuberilleImageToMeshFilter<itk::Image<TPixel, 3>, itk::Mesh<TMeshPixel, 3> > FilterType;
  typename FilterType::Pointer f = FilterType::New();
  f->SetIsoSurfaceValue( static_cast<TPixel>( 1 ) );
  f->GenerateTriangleFacesOn();
  f->ProjectVerticesToIsoSurfaceOff();
  f->SavePixelAsCellDataOn();
  f->SetLabelValue( static_cast<TPixel>( 5 ) );
  std::vector<TPixel> labels;
  labels.push_back( static_cast<TPixel>( 3 ) );
  labels.push_back( static_cast<TPixel>( ( 1ull << 53 ) + 2 ) );
  f->InsideRangeOff();
  f->SetLabelValues( labels );
  return f->GetLabelValues() == labels ? 0 : 1;
}

int main()
{
  int bad = 0;
  bad += Instantiate<long, float>();
  bad += Instantiate<unsigned long, unsigned long>();
  bad += Instantiate<long long, double>();
  bad += Instantiate<unsigned long long, unsigned long long>();
  return bad;
}
