// labels64_test01.cxx — include/itkCuberilleImageToMeshFilter.h on 64-bit integer images, built against the minimal ITK
// stand-in (tests/itk_shim) by tests/test_gpu_int64.py.  Two modes, both on a raw x-fastest volume file:
//   labels64_test01 Labels <in.raw> <nx> <ny> <nz> <label> [label ...]
//       an itk::Image<unsigned long, 3> label map (ITK's IdentifierType): every label in one Update() with
//       SetLabelValues; each label's part of the mesh must equal the mesh of a SetLabelValue( k ) run of the same
//       filter class, points bit for bit and cells with the ids shifted
//   labels64_test01 Iso <in.raw> <nx> <ny> <nz> <iso> <out.bin>
//       an itk::Image<long long, 3> meshed at iso with the default triangles and projection; out.bin receives the
//       points (float32 x, y, z) and then the cells (uint64 ids, three per triangle)
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <string>
#include <vector>

#include "itkImage.h"
#include "itkMesh.h"
#include "itkCuberilleImageToMeshFilter.h"

template <typename TImage>
static typename TImage::Pointer ReadRaw( const char * filename, char * dims [] )
{
  typename TImage::SizeType size;
  typename TImage::IndexType start;
  start.Fill( 0 );
  for ( int a = 0; a < 3; a++ ) { size[a] = std::strtoull( dims[a], 0, 10 ); }
  typename TImage::Pointer image = TImage::New();
  typename TImage::RegionType region;
  region.SetSize( size );
  region.SetIndex( start );
  image->SetRegions( region );
  image->Allocate();
  const size_t n = size[0] * size[1] * size[2];
  std::ifstream f( filename, std::ios::binary );
  f.read( reinterpret_cast<char *>( image->GetBufferPointer() ), n * sizeof( typename TImage::PixelType ) );
  if ( !f ) { throw itk::ExceptionObject( __FILE__, __LINE__, std::string( "cannot read " ) + filename ); }
  return image;
}

// the points (x, y, z per point) and the cells (ids per cell) of a mesh
template <typename TMesh>
static void Flatten( TMesh * mesh, std::vector<float> & points, std::vector<uint64_t> & cells )
{
  points.clear();
  cells.clear();
  for ( unsigned long i = 0; i < mesh->GetNumberOfPoints(); i++ )
    {
    const typename TMesh::PointType & p = mesh->GetPoints()->GetElement( i );
    for ( int a = 0; a < 3; a++ ) { points.push_back( p[a] ); }
    }
  for ( unsigned long i = 0; i < mesh->GetNumberOfCells(); i++ )
    {
    typename TMesh::CellType * c = 0;
    mesh->GetCell( i, c );
    for ( typename TMesh::CellType::PointIdConstIterator it = c->PointIdsBegin(); it != c->PointIdsEnd(); ++it ) { cells.push_back( *it ); }
    }
}

static int Labels( int argc, char * argv [] )
{
  typedef itk::Image< unsigned long, 3 > ImageType;
  typedef itk::Mesh< unsigned long, 3 > MeshType;
  typedef itk::CuberilleImageToMeshFilter< ImageType, MeshType > CuberilleType;
  std::vector<unsigned long> labels;
  for ( int i = 5; i < argc; i++ ) { labels.push_back( std::strtoul( argv[i], 0, 10 ) ); }
  ImageType::Pointer image = ReadRaw<ImageType>( argv[1], argv + 2 );
  CuberilleType::Pointer filter = CuberilleType::New();
  filter->SetInput( image );
  filter->SetLabelValues( labels );
  filter->ProjectVerticesToIsoSurfaceOff();
  filter->Update();
  std::vector<float> points;
  std::vector<uint64_t> cells;
  Flatten( filter->GetOutput(), points, cells );
  const std::vector<uint64_t> & po = filter->GetLabelPointOffsets();
  const std::vector<uint64_t> & co = filter->GetLabelCellOffsets();
  std::cout << "Mesh of " << labels.size() << " labels has " << points.size() / 3 << " vertices and " << cells.size() / 3
            << " cells" << std::endl;
  if ( po.size() != labels.size() + 1 || co.size() != labels.size() + 1 || po.back() * 3 != points.size() || co.back() * 3 != cells.size() )
    {
    std::cerr << "ERROR: the label offsets do not add up to the mesh" << std::endl;
    return EXIT_FAILURE;
    }
  for ( size_t i = 0; i < labels.size(); i++ )
    {
    CuberilleType::Pointer one = CuberilleType::New();
    one->SetInput( image );
    one->SetLabelValue( labels[i] );
    one->ProjectVerticesToIsoSurfaceOff();
    one->Update();
    std::vector<float> p1;
    std::vector<uint64_t> c1;
    Flatten( one->GetOutput(), p1, c1 );
    bool same = p1.size() == 3 * ( po[i + 1] - po[i] ) && c1.size() == 3 * ( co[i + 1] - co[i] ) &&
                ( p1.empty() || std::memcmp( &p1[0], &points[3 * po[i]], p1.size() * sizeof( float ) ) == 0 );
    for ( size_t k = 0; same && k < c1.size(); k++ ) { same = cells[3 * co[i] + k] == c1[k] + po[i]; }
    if ( !same )
      {
      std::cerr << "ERROR: the part of label " << labels[i] << " differs from its SetLabelValue run" << std::endl;
      return EXIT_FAILURE;
      }
    }
  return EXIT_SUCCESS;
}

static int Iso( int argc, char * argv [] )
{
  typedef itk::Image< long long, 3 > ImageType;
  typedef itk::Mesh< float, 3 > MeshType;
  typedef itk::CuberilleImageToMeshFilter< ImageType, MeshType > CuberilleType;
  if ( argc < 7 ) { return EXIT_FAILURE; }
  ImageType::Pointer image = ReadRaw<ImageType>( argv[1], argv + 2 );
  CuberilleType::Pointer filter = CuberilleType::New();
  filter->SetInput( image );
  filter->SetIsoSurfaceValue( std::strtoll( argv[5], 0, 10 ) );
  filter->Update();
  std::vector<float> points;
  std::vector<uint64_t> cells;
  Flatten( filter->GetOutput(), points, cells );
  std::ofstream out( argv[6], std::ios::binary );
  out.write( reinterpret_cast<const char *>( points.data() ), points.size() * sizeof( float ) );
  out.write( reinterpret_cast<const char *>( cells.data() ), cells.size() * sizeof( uint64_t ) );
  std::cout << "Mesh has " << points.size() / 3 << " vertices and " << cells.size() / 3 << " cells" << std::endl;
  return out ? EXIT_SUCCESS : EXIT_FAILURE;
}

int main( int argc, char * argv [] )
{
  try
    {
    if ( argc > 6 && std::string( argv[1] ) == "Labels" ) { return Labels( argc - 1, argv + 1 ); }
    if ( argc > 7 && std::string( argv[1] ) == "Iso" ) { return Iso( argc - 1, argv + 1 ); }
    }
  catch ( itk::ExceptionObject & err )
    {
    std::cerr << "ExceptionObject caught !" << std::endl << err << std::endl;
    return EXIT_FAILURE;
    }
  std::cout << "USAGE: " << argv[0] << " Labels <in.raw> <nx> <ny> <nz> <label> [label ...] | Iso <in.raw> <nx> <ny> <nz> <iso> <out.bin>"
            << std::endl;
  return EXIT_FAILURE;
}
