// range_test01.cxx — the inside-range setters of include/itkCuberilleImageToMeshFilter.h (SetInsideRange, SetLabelValue,
// InsideRangeOff and their getters), built against the minimal ITK stand-in (tests/itk_shim).  Two modes:
//   range_test01 Instantiate
//       no device needed: the setters and getters instantiate and behave for every pixel type of the reference's users
//   range_test01 RangeTest01 <in.mha> <lower> <upper> <expPoints> <expCells> [triangles]
//       the mesh of the voxels in [lower, upper] of an uncompressed 3-D MET_UCHAR MetaImage (SetLabelValue when
//       lower == upper), after checking that Update() refuses the range while the default projection is on; the
//       pass/fail rule of the reference's driver (Testing/CuberilleTest01.cxx:193-204).
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <iterator>
#include <map>
#include <sstream>
#include <string>
#include <vector>

#include "itkImage.h"
#include "itkMesh.h"
#include "itkCuberilleImageToMeshFilter.h"

template <typename TPixel, typename TMeshPixel>
int Instantiate()
{
  typedef itk::CuberilleImageToMeshFilter<itk::Image<TPixel, 3>, itk::Mesh<TMeshPixel, 3> > FilterType;
  typename FilterType::Pointer f = FilterType::New();
  if ( f->GetInsideRangeOn() ) { return 1; }
  f->SetInsideRange( static_cast<TPixel>( 1 ), static_cast<TPixel>( 2 ) );
  if ( !f->GetInsideRangeOn() || f->GetInsideRangeLower() != static_cast<TPixel>( 1 ) || f->GetInsideRangeUpper() != static_cast<TPixel>( 2 ) )
    {
    return 1;
    }
  f->SetLabelValue( static_cast<TPixel>( 3 ) );
  if ( f->GetInsideRangeLower() != static_cast<TPixel>( 3 ) || f->GetInsideRangeUpper() != static_cast<TPixel>( 3 ) ) { return 1; }
  f->InsideRangeOff();
  return f->GetInsideRangeOn() ? 1 : 0;
}

typedef unsigned char PixelType;
typedef itk::Image< PixelType, 3 > ImageType;
typedef itk::Mesh< PixelType, 3 > MeshType;
typedef itk::CuberilleImageToMeshFilter< ImageType, MeshType > CuberilleType;

static ImageType::Pointer ReadRawMetaImage( const char * filename )
{
  std::ifstream f( filename, std::ios::binary );
  if ( !f ) { throw itk::ExceptionObject( __FILE__, __LINE__, std::string( "cannot open " ) + filename ); }
  std::map<std::string, std::string> meta;
  std::string line;
  while ( std::getline( f, line ) )
    {
    const size_t eq = line.find( '=' );
    if ( eq == std::string::npos ) continue;
    std::string key = line.substr( 0, eq ), val = line.substr( eq + 1 );
    while ( !key.empty() && key[key.size() - 1] == ' ' ) key.erase( key.size() - 1 );
    while ( !val.empty() && val[0] == ' ' ) val.erase( 0, 1 );
    while ( !val.empty() && ( val[val.size() - 1] == '\r' || val[val.size() - 1] == ' ' ) ) val.erase( val.size() - 1 );
    meta[key] = val;
    if ( key == "ElementDataFile" ) break;
    }
  if ( meta["ElementDataFile"] != "LOCAL" || meta["ElementType"] != "MET_UCHAR" || meta["NDims"] != "3" || meta["CompressedData"] == "True" )
    { throw itk::ExceptionObject( __FILE__, __LINE__, "unsupported MetaImage (need 3-D uncompressed MET_UCHAR, LOCAL data)" ); }
  ImageType::SizeType size; ImageType::IndexType start; start.Fill( 0 );
  { std::istringstream ss( meta["DimSize"] ); ss >> size[0] >> size[1] >> size[2]; }
  std::vector<unsigned char> payload( ( std::istreambuf_iterator<char>( f ) ), std::istreambuf_iterator<char>() );
  const size_t n = size[0] * size[1] * size[2];
  if ( payload.size() < n ) { throw itk::ExceptionObject( __FILE__, __LINE__, "MetaImage payload too short" ); }
  ImageType::Pointer image = ImageType::New();
  ImageType::RegionType region; region.SetSize( size ); region.SetIndex( start );
  image->SetRegions( region );
  image->Allocate();
  std::copy( payload.begin(), payload.begin() + n, image->GetBufferPointer() );
  return image;
}

int RangeTest01( int argc, char * argv [] )
{
  if ( argc < 6 )
    {
    std::cout << "USAGE: RangeTest01 InputImage Lower Upper ExpectedNumberOfPoints ExpectedNumberOfCells [GenerateTriangleFaces]"
              << std::endl;
    return EXIT_FAILURE;
    }
  const PixelType lower = static_cast<PixelType>( std::atoi( argv[2] ) ), upper = static_cast<PixelType>( std::atoi( argv[3] ) );
  const unsigned long expectedPoints = std::strtoul( argv[4], 0, 10 ), expectedCells = std::strtoul( argv[5], 0, 10 );
  const bool triangles = argc > 6 ? std::atoi( argv[6] ) != 0 : true;
  try
    {
    CuberilleType::Pointer filter = CuberilleType::New();
    filter->SetInput( ReadRawMetaImage( argv[1] ) );
    if ( lower == upper ) { filter->SetLabelValue( lower ); }
    else { filter->SetInsideRange( lower, upper ); }
    filter->SetGenerateTriangleFaces( triangles );
    bool refused = false;
    try
      {
      filter->Update();
      }
    catch ( itk::ExceptionObject & err )
      {
      refused = std::string( err.what() ).find( "ProjectVerticesToIsoSurfaceOff" ) != std::string::npos;
      }
    if ( !refused )
      {
      std::cerr << "ERROR: an inside range with projection on was not refused" << std::endl;
      return EXIT_FAILURE;
      }
    filter->ProjectVerticesToIsoSurfaceOff();
    filter->Update();
    MeshType::Pointer mesh = filter->GetOutput();
    filter->Print( std::cout );
    std::cout << "Mesh has " << mesh->GetNumberOfPoints() << " vertices and " << mesh->GetNumberOfCells() << " cells" << std::endl;
    int status = EXIT_SUCCESS;
    if ( mesh->GetNumberOfPoints() != expectedPoints )
      {
      std::cerr << "ERROR: Expected mesh with " << expectedPoints << " points, but found " << mesh->GetNumberOfPoints() << std::endl;
      status = EXIT_FAILURE;
      }
    if ( mesh->GetNumberOfCells() != expectedCells )
      {
      std::cerr << "ERROR: Expected mesh with " << expectedCells << " cells, but found " << mesh->GetNumberOfCells() << std::endl;
      status = EXIT_FAILURE;
      }
    return status;
    }
  catch ( itk::ExceptionObject & err )
    {
    std::cerr << "ExceptionObject caught !" << std::endl << err << std::endl;
    return EXIT_FAILURE;
    }
}

int main( int argc, char * argv [] )
{
  if ( argc > 1 && std::string( argv[1] ) == "Instantiate" )
    {
    int bad = 0;
    bad += Instantiate<unsigned char, unsigned char>();
    bad += Instantiate<signed char, float>();
    bad += Instantiate<unsigned short, unsigned short>();
    bad += Instantiate<short, double>();
    bad += Instantiate<unsigned int, float>();
    bad += Instantiate<int, int>();
    bad += Instantiate<float, float>();
    bad += Instantiate<double, double>();
    return bad;
    }
  if ( argc > 1 && std::string( argv[1] ) == "RangeTest01" ) { return RangeTest01( argc - 1, argv + 1 ); }
  std::cout << "USAGE: " << argv[0] << " Instantiate | RangeTest01 <in.mha> <lower> <upper> <expPoints> <expCells> [triangles]"
            << std::endl;
  return EXIT_FAILURE;
}
